"""The DP kernels across the whole scoring domain bsw_create accepts: match 1..127, mismatch 0..127, ambig -127..match,
gap opens 0..16000 - e with extends >= 1, end_bonus 0..16000, zdrop 1..32767, both z-drop modes.  The kernel a pair
runs on, the 16-bit arithmetic of the packed kernels and the band all depend on these values, so every test here draws
seeded schemes from that domain, adds fixed corner schemes, and builds pairs at the boundaries that depend on the scheme.

CPU: the emulated sweeps of the packed kernel (k16), the warp-per-pair register kernel (w16), the int32 ring kernel
(l32) and bsw_global's second kernel (g2) against the oracle, the packed sweeps with several shared-memory fill bytes.
GPU: bsw_extend through every route, bsw_extend_packed, bsw_extend32, bsw_extend_retry, bsw_global, bsw_global32 and
bsw_reg2aln against their oracles, bit for bit."""
from __future__ import annotations

import ctypes as C
import zlib

import numpy as np
import pytest

from conftest import results_matrix
from oracle.pyoracle import make_params

PAIR_FIELDS = ("score", "qle", "tle", "gtle", "gscore", "max_off")
FILLS = (0xA5, 0x80, 0x7F)          # shared memory before a pair: -23131, -32640 and 32639 in every halfword
W16_MAX_QLEN = 255                  # w16::MAX_QLEN
EXT16_TOP = 32767                   # bsw_extend's domain: h0 + len2 * match <= 32767


# ---------------------------------------------------------------------------------------------------------------------
# Schemes
# ---------------------------------------------------------------------------------------------------------------------
def _logint(rng, lo: int, hi: int) -> int:
    """An integer in [lo, hi], log-uniform in (v - lo + 1): small values as often as large ones."""
    v = lo - 1 + int(np.exp(rng.uniform(0.0, np.log(hi - lo + 2))))
    return min(max(v, lo), hi)


def _scheme(match, mismatch, ambig, o_del, e_del, o_ins, e_ins, zdrop, end_bonus, w):
    return dict(match=match, mismatch=mismatch, ambig=ambig, o_del=o_del, e_del=e_del, o_ins=o_ins, e_ins=e_ins,
                zdrop=zdrop, end_bonus=end_bonus, w=w)


# fixed corners of the domain (w is the band the tests call with)
CORNERS = {
    "match127": _scheme(127, 4, -1, 6, 1, 6, 1, 100, 5, 100),                  # next to nothing fits the packed kernels
    "match127_amb": _scheme(127, 127, 127, 16000 - 9, 9, 0, 1, 32767, 16000, 50),
    "mismatch0": _scheme(2, 0, -1, 3, 2, 5, 1, 40, 5, 30),
    "ambig_m127": _scheme(3, 5, -127, 8, 2, 6, 3, 60, 0, 100),
    "ambig0": _scheme(1, 4, 0, 6, 1, 6, 1, 100, 5, 100),
    "ambig_match": _scheme(5, 7, 5, 10, 3, 10, 3, 200, 20, 60),
    "samegap_diff_e": _scheme(2, 6, -2, 7, 1, 5, 3, 80, 5, 100),                 # oe_del == oe_ins, e_del != e_ins
    "samegap_diff_e2": _scheme(1, 4, -1, 2, 6, 5, 3, 100, 5, 40),
    "same_e_diff_o": _scheme(1, 4, -1, 5, 2, 9, 2, 100, 5, 100),                 # e_del == e_ins, oe_del != oe_ins
    "e_ins_4681": _scheme(1, 4, -1, 6, 1, 6, 4681, 100, 5, 100),               # the warp kernel's last e_ins
    "e_ins_4682": _scheme(1, 4, -1, 6, 1, 6, 4682, 100, 5, 100),               # refused by the warp kernel
    "open_max": _scheme(1, 4, -1, 16000 - 3, 3, 16000 - 1, 1, 100, 5, 100),   # gap opens of 16000 - e
    "end_bonus0": _scheme(1, 4, -1, 6, 1, 6, 1, 100, 0, 100),
    "end_bonus_max": _scheme(2, 3, -1, 4, 2, 4, 2, 50, 16000, 100),
    "zdrop1": _scheme(1, 4, -1, 6, 1, 6, 1, 1, 5, 100),
    "zdrop_max": _scheme(3, 2, 1, 5, 1, 5, 1, 32767, 10, 200),
    "match6": _scheme(6, 9, -3, 12, 2, 9, 5, 300, 30, 40),                     # (h0 + len2 * 6) * 7 reaches 32767 exactly
    "match63": _scheme(63, 20, -20, 30, 4, 30, 4, 2000, 100, 20),             # (h0 + len2 * 63) * 64 reaches 32768 exactly
}


def _fits(s: dict, path: str, max_len: int) -> bool:
    """The path's own documented domain for pairs of up to max_len bases (both sides)."""
    mx = max(s["match"], s["mismatch"], abs(s["ambig"]))
    if path == "extend32":                        # h0 + len2 * max score + end_bonus <= 2^30 (with h0 < 2^20)
        return (1 << 20) + max_len * mx + s["end_bonus"] <= 1 << 30
    if path == "global32":                        # (len1 + len2 + 2) * c + o_del + o_ins <= 2^29
        c = max(mx, s["e_del"], s["e_ins"])
        return (2 * max_len + 2) * c + s["o_del"] + s["o_ins"] <= 1 << 29
    if path == "global":                          # g2::scores_ok: every table score a signed byte
        return all(-127 <= v <= 127 for v in (s["match"], -s["mismatch"], s["ambig"]))
    return True                                   # bsw_extend: h0 + len2 * match <= 32767 is the pairs' business


def schemes(seed: int, n: int, path: str = "extend", max_len: int = 1000) -> list:
    """n seeded schemes from the whole domain bsw_create accepts, narrowed only by the path's own domain."""
    rng = np.random.default_rng(seed)
    out = []
    while len(out) < n:
        match = _logint(rng, 1, 127)
        e_del, e_ins = _logint(rng, 1, 15999), _logint(rng, 1, 15999)
        s = _scheme(match, _logint(rng, 0, 127), int(rng.integers(-127, match + 1)),
                    _logint(rng, 0, 16000 - e_del), e_del, _logint(rng, 0, 16000 - e_ins), e_ins,
                    _logint(rng, 1, 32767), _logint(rng, 0, 16000), _logint(rng, 0, 500))
        if _fits(s, path, max_len):
            out.append(s)
    return out


def all_schemes(seed: int, n: int, path: str = "extend") -> dict:
    named = {f"r{k:02d}": s for k, s in enumerate(schemes(seed, n, path))}
    named.update({k: v for k, v in CORNERS.items() if _fits(v, path, 1000)})
    return named


def _seed(name: str) -> int:
    return zlib.crc32(name.encode()) & 0xFFFF


def oparams(s: dict, zmode: int = 0):
    return make_params(**{k: s[k] for k in ("match", "mismatch", "ambig", "o_del", "e_del", "o_ins", "e_ins", "zdrop",
                                            "end_bonus")}, zdrop_mode=zmode)


def engine_kw(s: dict, zmode: int) -> dict:
    return dict({k: v for k, v in s.items() if k != "w"}, zdrop_mode=zmode)


# ---------------------------------------------------------------------------------------------------------------------
# Pairs
# ---------------------------------------------------------------------------------------------------------------------
def k16_eligible(match: int, len2, h0):
    return (h0.astype(np.int64) + len2.astype(np.int64) * match) * (1 + match) <= 32767


def _mutate(rng, s: np.ndarray, err: float) -> np.ndarray:
    out = []
    for b in s:
        u = rng.random()
        if u < err / 3:
            out.append((b + rng.integers(1, 4)) % 4)
        elif u < 2 * err / 3:
            out += [b, rng.integers(0, 4)]
        elif u >= err:
            out.append(b)
    return np.array(out or [0], dtype=np.uint8)


KINDS = ("similar", "k16_top", "k16_over", "ext16_top", "q255", "q256", "n_query", "n_ref", "junk_tail", "h0_zero")


def domain_pairs(s: dict, seed: int, n: int, qmax: int = 300):
    """Seeded pairs for scheme s, all inside bsw_extend's domain (h0 + len2 * match <= 32767), cycling through KINDS:
      similar     the target a mutated copy of the query, h0 anywhere in the domain
      k16_top     the largest h0 with (h0 + len2 * match) * (1 + match) <= 32767 (= 32767 when 1 + match divides it)
      k16_over    one more: the first h0 outside the packed kernels' domain (= 32768 when 1 + match divides that)
      ext16_top   h0 + len2 * match = 32767, the top of bsw_extend's domain
      q255, q256  queries of 255 and 256 bases (w16::MAX_QLEN and one more), where the match score allows them
      n_query     a run of N in the query only;  n_ref: in the reference only
      junk_tail   the target's tail unrelated to the query (the scores fall, z-drop fires)
      h0_zero     h0 = 0
    -> (pairs, ref, qer)"""
    from genomicsbench_b200 import SEQPAIR_DTYPE
    rng = np.random.default_rng(seed)
    m = s["match"]
    lmax_ext = max(1, min(qmax, EXT16_TOP // m - 1))       # len2 that leaves room for h0 >= 1
    lmax_k16 = max(1, (32767 // (1 + m)) // m)             # len2 that leaves room for a non-negative k16_top h0
    pairs = np.zeros(n, dtype=SEQPAIR_DTYPE)
    qs, ts = [], []
    qo = ro = 0
    for k in range(n):
        kind = KINDS[k % len(KINDS)]
        if kind in ("k16_top", "k16_over"):
            L = int(rng.integers(1, min(lmax_k16, qmax) + 1))
            h0 = 32767 // (1 + m) - L * m + (kind == "k16_over")
        elif kind == "ext16_top":
            L = int(rng.integers(1, lmax_ext + 1))
            h0 = EXT16_TOP - L * m
        elif kind in ("q255", "q256"):
            L = 255 if kind == "q255" else 256
            if L * m >= EXT16_TOP:
                L = lmax_ext
            h0 = int(rng.integers(0, min(EXT16_TOP - L * m, 400) + 1))
        else:
            L = int(rng.integers(1, lmax_ext + 1))
            h0 = 0 if kind == "h0_zero" else int(rng.integers(1, min(EXT16_TOP - L * m, 3 * L * m + 50) + 1))
        q = rng.integers(0, 4, L).astype(np.uint8)
        t = _mutate(rng, q, float(rng.uniform(0.0, 0.15)))
        if kind == "junk_tail" and len(t) > 2:
            cut = int(rng.integers(1, len(t)))
            t[cut:] = rng.integers(0, 4, len(t) - cut)
        if kind == "n_query":
            a = int(rng.integers(0, L)); q[a: a + int(rng.integers(1, 20))] = 4
        if kind == "n_ref":
            a = int(rng.integers(0, len(t))); t[a: a + int(rng.integers(1, 20))] = 4
        assert h0 >= 0 and h0 + L * m <= EXT16_TOP
        pairs[k]["idq"], pairs[k]["idr"], pairs[k]["len2"], pairs[k]["len1"], pairs[k]["h0"] = qo, ro, L, len(t), h0
        qs.append(q); ts.append(t)
        qo += L; ro += len(t)
    pairs["id"] = np.arange(n)
    for f in PAIR_FIELDS:
        pairs[f] = -7
    return pairs, np.concatenate(ts + [np.zeros(64, np.uint8)]), np.concatenate(qs + [np.zeros(64, np.uint8)])


def has_n(pairs, ref, qer) -> np.ndarray:
    return np.array([(qer[p["idq"]: p["idq"] + p["len2"]] > 3).any() or (ref[p["idr"]: p["idr"] + p["len1"]] > 3).any()
                     for p in pairs])


def oracle_run(oracle, s, zmode, pairs, ref, qer, w=None):
    want = pairs.copy()
    cells = oracle.batch(oparams(s, zmode), want, ref, qer, s["w"] if w is None else w)
    return want, cells


def test_pair_generator_hits_the_boundaries():
    """The boundary kinds land where they claim: exactly 32767 / 32768 for the corner matches that allow it."""
    for name, prod in (("match6", 32767), ("match63", 32768), ("match127", 32768)):
        s = CORNERS[name]
        pairs, ref, qer = domain_pairs(s, 5, 4 * len(KINDS))
        m = s["match"]
        v = (pairs["h0"].astype(np.int64) + pairs["len2"].astype(np.int64) * m) * (1 + m)
        assert (v == prod).any(), name
        top = pairs["h0"].astype(np.int64) + pairs["len2"].astype(np.int64) * m
        assert (top == EXT16_TOP).any() and (top <= EXT16_TOP).all()
        assert k16_eligible(m, pairs["len2"], pairs["h0"]).any() and not k16_eligible(m, pairs["len2"], pairs["h0"]).all()
    pairs, ref, qer = domain_pairs(CORNERS["ambig0"], 5, 4 * len(KINDS))
    assert (pairs["len2"] == 255).any() and (pairs["len2"] == 256).any() and (pairs["h0"] == 0).any()
    nq = np.array([(qer[p["idq"]: p["idq"] + p["len2"]] > 3).any() for p in pairs])
    nr = np.array([(ref[p["idr"]: p["idr"] + p["len1"]] > 3).any() for p in pairs])
    assert (nq & ~nr).any() and (nr & ~nq).any()


# ---------------------------------------------------------------------------------------------------------------------
# CPU: emulations
# ---------------------------------------------------------------------------------------------------------------------
CPU_SCHEMES = all_schemes(0x5C0E1, 60)


def _prm(s: dict, zmode: int, ambig: bool = False) -> np.ndarray:
    v = [s["match"], s["mismatch"], s["o_del"], s["e_del"], s["o_ins"], s["e_ins"], s["zdrop"], s["end_bonus"], zmode]
    return np.array(v + ([s["ambig"]] if ambig else []), dtype=np.int32)


@pytest.fixture(scope="module")
def k16():
    from emu.build import build
    lib = C.CDLL(str(build(name="k16")))
    lib.k16_emu_batch2.restype = C.c_longlong
    lib.k16_emu_batch2.argtypes = [C.c_void_p] * 4 + [C.c_longlong, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return lib


@pytest.fixture(scope="module")
def w16():
    from emu.build import build
    lib = C.CDLL(str(build(name="w16")))
    lib.w16_emu_batch.restype = C.c_longlong
    lib.w16_emu_batch.argtypes = [C.c_void_p] * 4 + [C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return lib


@pytest.fixture(scope="module")
def l32():
    from emu.build import build
    lib = C.CDLL(str(build(name="l32")))
    lib.l32_emu_batch.restype = C.c_longlong
    lib.l32_emu_batch.argtypes = [C.c_void_p] * 4 + [C.c_longlong, C.c_int, C.c_int]
    return lib


@pytest.fixture(scope="module")
def g2():
    from emu.build import build
    lib = C.CDLL(str(build(name="g2")))
    lib.g2_emu_global.restype = C.c_int
    lib.g2_emu_global.argtypes = [C.c_void_p] * 4 + [C.c_longlong, C.c_void_p, C.c_int, C.c_longlong, C.c_longlong] + \
        [C.c_void_p] * 3 + [C.c_longlong, C.c_void_p, C.c_void_p]
    return lib


def run_k16(lib, s, zmode, pairs, ref, qer, circ, fill):
    skipped = np.zeros(len(pairs), dtype=np.uint8)
    ovf = C.c_longlong(0)
    cells = lib.k16_emu_batch2(_prm(s, zmode).ctypes.data, pairs.ctypes.data, ref.ctypes.data, qer.ctypes.data,
                               len(pairs), s["w"], circ, fill, skipped.ctypes.data, C.byref(ovf))
    return int(cells), skipped.astype(bool)


def run_w16(lib, s, zmode, pairs, ref, qer, fill):
    skipped = np.zeros(len(pairs), dtype=np.uint8)
    ovf = C.c_longlong(0)
    cells = lib.w16_emu_batch(_prm(s, zmode).ctypes.data, pairs.ctypes.data, ref.ctypes.data, qer.ctypes.data,
                              len(pairs), s["w"], fill, skipped.ctypes.data, C.byref(ovf))
    assert cells >= 0, "the lanes of a warp disagreed"
    return int(cells), skipped.astype(bool)


def _plain(pairs, ref, qer):
    """The pairs without N (those run on the byte kernels, not the 2-bit packed ones)."""
    return pairs[~has_n(pairs, ref, qer)].copy()


@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("name", sorted(CPU_SCHEMES))
def test_k16_emulation_across_the_domain(k16, oracle, name, zmode):
    """The packed kernel's sweep, whole rows and circular rows, with three shared-memory fill bytes: it runs exactly the
    pairs k16::eligible admits, and on those its results and effective cells are the oracle's whatever the fill."""
    s = CPU_SCHEMES[name]
    pairs, ref, qer = domain_pairs(s, _seed(name), 300)
    pairs = _plain(pairs, ref, qer)
    elig = k16_eligible(s["match"], pairs["len2"], pairs["h0"])
    assert elig.any() and not elig.all()
    want, cells_o = oracle_run(oracle, s, zmode, pairs[elig], ref, qer)
    for circ in (0, 1):
        first = None
        for fill in FILLS:
            got = pairs.copy()
            cells, skipped = run_k16(k16, s, zmode, got, ref, qer, circ, fill)
            assert np.array_equal(skipped, ~elig), (circ, fill)
            r = results_matrix(got[elig])
            if first is None:
                first = r
            assert np.array_equal(r, first), f"circ {circ}: fill {fill:#x} changed {(r != first).any(axis=1).sum()} pairs"
            bad = (r != results_matrix(want)).any(axis=1)
            assert not bad.any(), f"circ {circ} fill {fill:#x}: {bad.sum()} pairs differ from the oracle"
            assert cells == cells_o, (circ, fill)


def _w16_ok(s, pairs):
    return (7 * s["e_ins"] <= 32767) & k16_eligible(s["match"], pairs["len2"], pairs["h0"]) & (pairs["len2"] <= W16_MAX_QLEN)


@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("name", sorted(CPU_SCHEMES))
def test_w16_emulation_across_the_domain(w16, oracle, name, zmode):
    """The warp-per-pair register kernel's sweep, three fill bytes: it runs exactly the pairs w16::scoring_ok,
    k16::eligible and w16::MAX_QLEN admit, with the oracle's results and effective cells whatever the fill."""
    s = CPU_SCHEMES[name]
    pairs, ref, qer = domain_pairs(s, _seed(name), 120)
    pairs = _plain(pairs, ref, qer)
    ok = _w16_ok(s, pairs)
    assert not ok.all()
    if 7 * s["e_ins"] <= 32767:                 # schemes w16::scoring_ok refuses check the refusal alone
        assert ok.any()
    want, cells_o = oracle_run(oracle, s, zmode, pairs[ok], ref, qer)
    first = None
    for fill in FILLS:
        got = pairs.copy()
        cells, skipped = run_w16(w16, s, zmode, got, ref, qer, fill)
        assert np.array_equal(skipped, ~ok), fill
        r = results_matrix(got[ok])
        if first is None:
            first = r
        assert np.array_equal(r, first), f"fill {fill:#x} changed {(r != first).any(axis=1).sum()} pairs"
        bad = (r != results_matrix(want)).any(axis=1)
        assert not bad.any(), f"fill {fill:#x}: {bad.sum()} pairs differ from the oracle"
        assert cells == cells_o, fill


@pytest.mark.parametrize("e_ins", [4681, 4682])
def test_w16_guard_boundary(w16, oracle, e_ins):
    """w16::scoring_ok: at e_ins = 4681 (7 e_ins = 32767) the warp kernel runs and equals the oracle; at 4682 it
    refuses every pair, so the engine keeps such schemes on the other kernels."""
    s = CORNERS[f"e_ins_{e_ins}"]
    pairs, ref, qer = domain_pairs(s, 77, 150)
    pairs = _plain(pairs, ref, qer)
    pairs = pairs[k16_eligible(s["match"], pairs["len2"], pairs["h0"]) & (pairs["len2"] <= W16_MAX_QLEN)].copy()
    assert len(pairs) > 30
    for zmode in (0, 1):
        got = pairs.copy()
        cells, skipped = run_w16(w16, s, zmode, got, ref, qer, 0xA5)
        if e_ins == 4682:
            assert skipped.all() and cells == 0
            continue
        want, cells_o = oracle_run(oracle, s, zmode, pairs, ref, qer)
        assert not skipped.any()
        assert np.array_equal(results_matrix(got), results_matrix(want)) and cells == cells_o


@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("name", sorted(CPU_SCHEMES))
def test_l32_emulation_across_the_domain(l32, oracle, name, zmode):
    """The int32 ring kernel's sweep (bsw_extend32) on every pair of the scheme, N included (ambig is read here)."""
    s = CPU_SCHEMES[name]
    pairs, ref, qer = domain_pairs(s, (_seed(name)) + 1, 60, qmax=200)
    want, cells_o = oracle_run(oracle, s, zmode, pairs, ref, qer)
    got = pairs.copy()
    cells = l32.l32_emu_batch(_prm(s, zmode, ambig=True).ctypes.data, got.ctypes.data, ref.ctypes.data,
                              qer.ctypes.data, len(got), s["w"], 0)
    assert cells >= 0, "the lanes of a warp disagreed"
    bad = (results_matrix(got) != results_matrix(want)).any(axis=1)
    assert not bad.any(), f"{bad.sum()} pairs differ from the oracle"
    assert cells == cells_o


def global_cases(s: dict, seed: int, n: int, lmax: int = 150):
    """Pairs for global alignment: similar and unrelated sequences, N on either side, bands from 0 to wider than both.
    -> (queries, targets, bands)"""
    rng = np.random.default_rng(seed)
    qs, ts, ws = [], [], []
    for k in range(n):
        L = int(rng.integers(1, lmax + 1))
        q = rng.integers(0, 4, L).astype(np.uint8)
        t = _mutate(rng, q, 0.1) if k % 3 else rng.integers(0, 4, int(rng.integers(1, lmax + 1))).astype(np.uint8)
        if k % 4 == 1:
            a = int(rng.integers(0, len(q))); q[a: a + int(rng.integers(1, 12))] = 4
        if k % 4 == 2:
            a = int(rng.integers(0, len(t))); t[a: a + int(rng.integers(1, 12))] = 4
        d = abs(len(q) - len(t))
        ws.append(d + (0 if k % 7 == 0 else int(rng.integers(0, 20)) if k % 11 else int(rng.integers(100, 300))))
        qs.append(q); ts.append(t)
    return qs, ts, ws


G2_SCHEMES = {k: v for k, v in all_schemes(0x5C0E2, 25, "global").items() if not k.startswith("e_ins")}


@pytest.mark.parametrize("name", sorted(G2_SCHEMES))
def test_g2_emulation_across_the_domain(g2, oracle, name):
    """bsw_global's second kernel, with the slot width the engine would pick, against the oracle: ambig from -127 to
    match (a positive score against N), mismatch 0, match up to 127, heavy gaps."""
    from test_g2_emulation import run_emu
    s = G2_SCHEMES[name]
    P = {k: s[k] for k in ("o_del", "e_del", "o_ins", "e_ins", "match", "mismatch", "ambig")}
    qs, ts, ws = global_cases(s, _seed(name), 80)
    rc, score, ncig, cigar, off, info = run_emu(g2, P, [len(t) for t in ts], [len(q) for q in qs], np.concatenate(ts),
                                                np.concatenate(qs), ws)
    assert rc == 0
    Po = oparams(s)
    for k in range(len(qs)):
        sc, cg = oracle.global_align(Po, qs[k], ts[k], ws[k])
        assert sc == score[k] and np.array_equal(cg, cigar[off[k]: off[k + 1]]), (k, sc, int(score[k]))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
GPU_SCHEMES = all_schemes(0x5C0E3, 10)
# bsw_extend's chunks (run_pipeline, bsw_engine.cu): the first is CHUNK_MIN pairs when more than 4 CHUNK_MIN pairs
# remain; a packed batch starts at 2 CHUNK_MIN, so it needs more than 8 CHUNK_MIN pairs for a second chunk
CHUNK_MIN = 1 << 15


def _tile(pairs, reps):
    big = np.tile(pairs, reps)
    big["id"] = np.arange(len(big))
    return big


@pytest.mark.gpu
@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("name", sorted(GPU_SCHEMES))
def test_gpu_extend_routes_across_the_domain(lib, oracle, name, zmode):
    """bsw_extend on every route, bsw_extend_packed in both record forms: the oracle's six fields and effective cells."""
    s = GPU_SCHEMES[name]
    w = s["w"]
    base, ref, qer = domain_pairs(s, (_seed(name)) + 2, 1000)
    want, cells_o = oracle_run(oracle, s, zmode, base, ref, qer)
    wm = results_matrix(want)
    kw = engine_kw(s, zmode)

    def check(got, wmat, what):
        bad = (results_matrix(got) != wmat).any(axis=1)
        assert not bad.any(), f"{what}: {bad.sum()} pairs differ; first {np.flatnonzero(bad)[:3] % len(wmat)}"

    reps = 4 * CHUNK_MIN // len(base) + 2
    big = _tile(base, reps)                       # several chunks on pageable and on page-locked buffers
    for extra, pinned in (({}, False), ({}, True), ({"short_variant": 1}, False), ({"long_min_qlen": 1}, False),
                          ({"warp_max_pairs": 1 << 20}, False)):
        with lib.Engine(**kw, **extra) as eng:
            got = lib.pinned_copy(big) if pinned else big.copy()
            eng.extend(got, lib.pinned_copy(ref) if pinned else ref, lib.pinned_copy(qer) if pinned else qer, w)
            st = eng.stats()
        check(got, np.tile(wm, (reps, 1)), (extra, pinned))
        assert st["cells_effective"] == reps * cells_o, (extra, pinned)
        if "long_min_qlen" in extra:
            assert st["n_long"] == len(big)
        elif not extra:
            assert st["n_short"] > 0

    # the latency route (tiny_batch): one call, one kernel.  A call whose pairs are all plain (no N, inside
    # k16::eligible, queries of at most w16::MAX_QLEN bases) runs a 16-bit kernel on 2-bit words: the warp-per-pair
    # register kernel while the device's warp budget lasts, else (warp_max_pairs = 1: a budget of one pair) the
    # thread-per-pair packed kernel; with warp_max_pairs = -1 or a scheme w16::scoring_ok refuses, and for any call
    # with one other pair, the whole call runs the byte-reading warp-per-pair kernel.
    plain_mask = ~has_n(base, ref, qer) & k16_eligible(s["match"], base["len2"], base["h0"]) & \
        (base["len2"] <= W16_MAX_QLEN)
    plain = base[plain_mask].copy()
    assert len(plain) > 0 and not plain_mask.all()
    plain_cells = oracle_run(oracle, s, zmode, plain, ref, qer)[1]
    for batch, wmat, cells, is_plain in ((base, wm, cells_o, False), (plain, wm[plain_mask], plain_cells, True)):
        for wmp in (-1, 0, 1):
            for pinned in (False, True):
                what = ("tiny", "plain" if is_plain else "mixed", wmp, pinned)
                with lib.Engine(**kw, tiny_batch=len(batch), warp_max_pairs=wmp) as eng:
                    got = lib.pinned_copy(batch) if pinned else batch.copy()
                    eng.extend(got, lib.pinned_copy(ref) if pinned else ref, lib.pinned_copy(qer) if pinned else qer, w)
                    st = eng.stats()
                check(got, wmat, what)
                assert st["cells_effective"] == cells and st["kernel_launches"] == 1, what
                sixteen = is_plain and wmp >= 0 and 7 * s["e_ins"] <= 32767
                assert (st["n_short"], st["n_long"]) == ((len(batch), 0) if sixteen else (0, len(batch))), what

    preps = 8 * CHUNK_MIN // len(base) + 2
    b = lib.PackedBatch.from_pairs(_tile(base, preps), ref, qer)
    with lib.Engine(**kw) as eng:
        for compact in (False, True):
            out = eng.extend_packed(b, w, compact=compact)
            m = np.stack([out[f] for f in PAIR_FIELDS], axis=1).astype(np.int32)
            bad = (m != np.tile(wm, (preps, 1))).any(axis=1)
            assert not bad.any(), f"packed compact={compact}: {bad.sum()} pairs differ"


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GPU_SCHEMES))
def test_gpu_extend32_and_retry_across_the_domain(lib, oracle, name):
    """bsw_extend32 on pairs beyond bsw_extend's 16-bit domain (h0 + len2 * match > 32767), and bsw_extend_retry
    against the oracle's band-doubling loop."""
    from test_extend32 import long_pairs
    s = GPU_SCHEMES[name]
    m = s["match"]
    pairs, ref, qer = long_pairs(_seed(name), 40, 50, 1500, (0, 0), err=0.1, n_rate=0.003, junk_tail=0.3)
    rng = np.random.default_rng(_seed(name))
    pairs["h0"] = np.maximum(1, EXT16_TOP + 1 - pairs["len2"].astype(np.int64) * m) + rng.integers(0, 60000, len(pairs))
    assert ((pairs["h0"].astype(np.int64) + pairs["len2"].astype(np.int64) * m) > EXT16_TOP).all()
    for zmode in (0, 1):
        want, cells_o = oracle_run(oracle, s, zmode, pairs, ref, qer)
        got = pairs.copy()
        with lib.Engine(**engine_kw(s, zmode)) as eng:
            eng.extend32(got, ref, qer, s["w"])
            st = eng.stats()
        assert np.array_equal(results_matrix(got), results_matrix(want)), zmode
        assert st["cells_effective"] == cells_o
    base, ref, qer = domain_pairs(s, (_seed(name)) + 3, 2000)
    w = max(1, s["w"] // 4)
    for zmode in (0, 1):
        want = base.copy()
        band_o = oracle.band_retry(oparams(s, zmode), want, ref, qer, w)
        got = base.copy()
        with lib.Engine(**engine_kw(s, zmode)) as eng:
            band = eng.extend_retry(got, ref, qer, w)
        assert np.array_equal(results_matrix(got), results_matrix(want)), zmode
        assert np.array_equal(band, band_o), zmode


GLOBAL_GPU_SCHEMES = {k: v for k, v in all_schemes(0x5C0E4, 8, "global").items()
                      if k in ("match127_amb", "mismatch0", "ambig_m127", "ambig0", "ambig_match", "samegap_diff_e",
                               "open_max", "match63") or k.startswith("r")}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GLOBAL_GPU_SCHEMES))
def test_gpu_global_across_the_domain(lib, oracle, name):
    """bsw_global and bsw_global32 against the oracle's ksw_global2, scores and CIGARs."""
    from genomicsbench_b200 import SEQPAIR_DTYPE
    s = GLOBAL_GPU_SCHEMES[name]
    qs, ts, ws = global_cases(s, (_seed(name)) + 4, 300, lmax=400)
    pairs = np.zeros(len(qs), dtype=SEQPAIR_DTYPE)
    pairs["len1"], pairs["len2"] = [len(t) for t in ts], [len(q) for q in qs]
    pairs["idr"] = np.concatenate([[0], np.cumsum(pairs["len1"])[:-1]])
    pairs["idq"] = np.concatenate([[0], np.cumsum(pairs["len2"])[:-1]])
    ref, qer = np.concatenate(ts + [np.zeros(64, np.uint8)]), np.concatenate(qs + [np.zeros(64, np.uint8)])
    Po = oparams(s)
    want = [oracle.global_align(Po, qs[k], ts[k], ws[k]) for k in range(len(qs))]
    with lib.Engine(**engine_kw(s, 0)) as eng:
        for fn in (eng.global_align, eng.global_align32):
            score, cigar, off = fn(pairs, ref, qer, np.array(ws, dtype=np.int32))
            for k, (sc, cg) in enumerate(want):
                assert sc == score[k] and np.array_equal(cg, cigar[off[k]: off[k + 1]]), (fn.__name__, k)


REG2ALN_SCHEMES = {
    "match3_amb0": dict(match=3, mismatch=5, o_del=6, e_del=1, o_ins=6, e_ins=1, ambig=0),
    "match2_amb_pos": dict(match=2, mismatch=3, o_del=5, e_del=2, o_ins=4, e_ins=3, ambig=2),
    "asym_amb_neg": dict(match=1, mismatch=4, o_del=9, e_del=1, o_ins=3, e_ins=2, ambig=-5),
    "large_e_del": dict(match=2, mismatch=4, o_del=10, e_del=40, o_ins=6, e_ins=1, ambig=-1),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(REG2ALN_SCHEMES))
def test_gpu_reg2aln_across_the_domain(lib, name):
    """bsw_reg2aln against aln_oracle.c with match > 1, ambig != -1 (the MD pass's fast-path score), asymmetric gaps and
    a large e_del (band inference and the band-doubling loop on non-default arithmetic); N runs in the reads."""
    from test_reg2aln import AlnOracle, assert_equal_oracle, loop_cases
    aln = AlnOracle()
    P = REG2ALN_SCHEMES[name]
    regs, query, D, l_pac, _ = loop_cases(seed=91 + len(name), n=3000)
    rng = np.random.default_rng(92)
    q = query.copy()
    for _ in range(200):
        a = int(rng.integers(0, len(q) - 64)); q[a: a + int(rng.integers(1, 30))] = 4
    regs["reg"]["truesc"] *= P["match"]
    for w in (1, 100):
        want = aln.reg2aln(make_params(**P), regs, q, D, l_pac, w)
        with lib.Engine(**P) as eng:
            got = eng.reg2aln(regs, q, D, l_pac, w)
        assert_equal_oracle(got, want)
        assert want["info"][:, 2].sum() > 0

"""bsw_extend across the whole length domain it accepts: 1 <= len1, len2 <= 32767 (include/bsw.h).  Lengths pick the
kernel, the row form, the shared-memory class and the chunk layout just as the scores do, so every test here builds
pairs at the length boundaries the engine steps at:
  queries  1-9 (tails of the groups of 4), 127-129 and 511-513 (the shared-memory classes of stride_for), 255/256
           (w16::MAX_QLEN), 823-825 (SHORT_MAX_QLEN: the packed kernels' last query), 3063-3065 (the warp-per-pair
           kernel's rows leave shared memory for HBM), 8191, 16383 and 32766;
  targets  1, len2 - 1, len2, len2 + 1, 2 len2 and 32767, related to the query or not (z-drop fires or does not);
  bands    0, 1, 100, 4096 (the last circular-row band), 4097, wider than the query, 2^31 - 1 (the clamp at the top);
  h0       0 up to the top of the domain, h0 + len2 * match = 32767 (an exact match there scores 32767).
CPU: the packed (k16) and warp register (w16) sweeps on the pairs they admit, with long targets.
GPU: bsw_extend through every route, the latency route at its row limit, the HBM row form, bsw_extend_packed,
bsw_stage, bsw_extend_retry and bsw_extend32 against the oracle, and calls whose chunks hold more than 2^30 bytes of
sequence."""
from __future__ import annotations

import numpy as np
import pytest

from conftest import results_matrix
from test_extend32 import mutate
from test_scoring_domain import (EXT16_TOP, FILLS, PAIR_FIELDS, W16_MAX_QLEN, _scheme, _tile, engine_kw, has_n,
                                 k16, k16_eligible, oparams, oracle_run, run_k16, run_w16, w16)  # noqa: F401 (fixtures)

# ---------------------------------------------------------------------------------------------------------------------
# The boundaries, derived from the engine's own rules
# ---------------------------------------------------------------------------------------------------------------------
SHORT_MAX_QLEN = 824                   # bsw_engine.cu: the longest query of the packed kernels
LONG_WARPS = 4                         # bsw_kernels.cuh: warps per block of bsw_long_kernel
SMEM_ROWS = 48 * 1024                  # bsw_long_kernel keeps its rows in shared memory up to this many bytes
CIRC_MAX_W = 4096                      # device_prepare: circular rows only for w <= 4096
RAW_LIMIT = 0x3FFFFFFF                 # 32-bit chunk offsets: at most 2^30 - 1 bytes of a side per chunk


def long_row_bytes(qmax: int) -> int:
    """Shared memory of bsw_long_kernel's rows for a chunk's longest query (launch_bytes, run_tiny):
    LONG_WARPS rows of long_stride = (qmax + 12) & ~3 four-byte cells."""
    return LONG_WARPS * ((qmax + 12) & ~3) * 4


HBM_QLEN = next(q for q in range(1, 32768) if long_row_bytes(q) > SMEM_ROWS)     # first query whose rows live in HBM


def stride_class(qmax: int) -> int:
    """stride_for's rounding step for a query: 4 words up to 128 bases, 16 up to 512, 32 beyond."""
    need = qmax + 8
    return 4 if need <= 136 else 16 if need <= 520 else 32


QLENS = list(range(1, 10)) + [127, 128, 129, 255, 256, 511, 512, 513, SHORT_MAX_QLEN - 1, SHORT_MAX_QLEN,
                              SHORT_MAX_QLEN + 1, HBM_QLEN - 1, HBM_QLEN, HBM_QLEN + 1, 8191, 16383, 32766]
BANDS = {"w0": 0, "w1": 1, "w100": 100, "w4096": CIRC_MAX_W, "w4097": CIRC_MAX_W + 1, "wide": 32767,
         "w_int32_top": (1 << 31) - 1}

SCHEMES = {
    "bwa": _scheme(1, 4, -1, 6, 1, 6, 1, 100, 5, 0),
    "match2_asym": _scheme(2, 5, -1, 8, 1, 5, 2, 200, 10, 0),
    "large_e_del": _scheme(1, 4, -1, 6, 60, 6, 1, 100, 5, 0),       # bsw_clamp_band: w <= (qlen * 4 - 1) / 60 + 1
    # the band clamp allows len2 * match / e_del and z-drop never fires: past the query's end the deletions run down
    # the target for len2 * match rows.  With (h0 + len2 * match) * (1 + match) <= 32767, match = 5 takes the packed
    # kernel to its deepest rows, about 4950 (824 * 6)
    "deep_rows": _scheme(5, 4, -1, 6, 1, 6, 1, 32767, 5, 0),
}
# without z-drop an unrelated tail runs as far as the score lasts: queries up to the HBM boundary keep the oracle cheap
QLENS_OF = {"deep_rows": [q for q in QLENS if q <= 3065]}


def target_lengths(L: int) -> list:
    return sorted({t for t in (1, L - 1, L, L + 1, 2 * L, 32767) if 1 <= t <= 32767})


def length_pairs(s: dict, seed: int, qlens=None):
    """Seeded pairs at the length boundaries for scheme s, all inside bsw_extend's domain.  Per query length L (those
    with L * match <= 32767) one pair per target length of target_lengths(L), the target alternately a mutated copy of
    the query padded with random bases (related: the score climbs along the whole query, and with a large h0 the
    deletions past its end keep the sweep going down a long target) and one whose tail turns unrelated (z-drop
    fires), the two alternating between neighbouring query lengths too.  Queries of 8191 bases and more have one related pair each (a full band over them costs
    up to a gigacell in the oracle); their other targets turn unrelated within the first 3000 bases.  h0 cycles through
    0, the top of the domain (h0 + L * match = 32767), the packed kernels' top and values between.  Then:
      exact     the longest query the scheme allows with h0 = 32767 - L * match, the target the query plus one base:
                it scores exactly 32767, tle and qle at the top of int16
      deepest   the longest queries the packed kernels admit at h0 = 0, against related 32767-base targets: the
                deletions past the query's end take the sweep furthest down the target
      k16_top   short queries against 32767-base targets at the largest h0 with (h0 + L * match) * (1 + match) <= 32767,
      k16_over  and at one more
      n_query   N in the query only (a 3064-base query and a short one against a 32767-base target);
      n_ref     N in the target only
    -> (pairs, ref, qer)"""
    from genomicsbench_b200 import SEQPAIR_DTYPE
    rng = np.random.default_rng(seed)
    m = s["match"]
    qlens = QLENS if qlens is None else qlens
    rows = []                                                       # (q, t, h0)

    def h0_for(L, k):
        top, k16_top = EXT16_TOP - L * m, 32767 // (1 + m) - L * m
        return (0, top, k16_top if k16_top >= 0 else int(rng.integers(0, top + 1)), int(rng.integers(0, top + 1)),
                min(top, int(rng.integers(0, 3 * L * m + 50))))[k % 5]

    k = 0
    for li, L in enumerate(qlens):
        if L * m > EXT16_TOP:
            continue
        q = rng.integers(0, 4, L).astype(np.uint8)
        for j, T in enumerate(target_lengths(L)):
            related = ((j + li) % 2 == 0) if L < 8191 else T == L + 1
            t = mutate(rng, q, 0.03)[:T]
            if len(t) < T:
                t = np.concatenate([t, rng.integers(0, 4, T - len(t)).astype(np.uint8)])
            if not related and T > 1:
                cut = int(rng.integers(1, min(T, 3000)))
                t[cut:] = rng.integers(0, 4, T - cut)
            rows.append((q, t, h0_for(L, k)))
            k += 1
    L = min(32766, EXT16_TOP // m - (1 if EXT16_TOP % m == 0 else 0))
    q = rng.integers(0, 4, L).astype(np.uint8)
    rows.append((q, np.concatenate([q, [1]]).astype(np.uint8), EXT16_TOP - L * m))                  # exact
    for L in (min(SHORT_MAX_QLEN, 32767 // ((1 + m) * m)), min(W16_MAX_QLEN, 32767 // ((1 + m) * m))):
        q = rng.integers(0, 4, L).astype(np.uint8)
        t = np.concatenate([mutate(rng, q, 0.02), rng.integers(0, 4, 32767).astype(np.uint8)])[:32767]
        rows.append((q, t, 0))                                                                       # deepest
    for L in (7, 128, 200, 255, 256, 700):
        if L * m > 32767 // (1 + m):
            continue
        q = rng.integers(0, 4, L).astype(np.uint8)
        t = np.concatenate([mutate(rng, q, 0.02), rng.integers(0, 4, 32767).astype(np.uint8)])[:32767]
        top = 32767 // (1 + m) - L * m
        rows.append((q, t, top)); rows.append((q, t.copy(), top + 1))                                # k16_top / over
    for L, T in ((HBM_QLEN, HBM_QLEN + 40), (150, 32767)):
        q = rng.integers(0, 4, L).astype(np.uint8)
        t = np.concatenate([mutate(rng, q, 0.03), rng.integers(0, 4, T).astype(np.uint8)])[:T]
        qn = q.copy(); a = int(rng.integers(0, L - 10)); qn[a: a + 10] = 4
        tn = t.copy(); a = int(rng.integers(0, min(T, L) - 10)); tn[a: a + 10] = 4
        rows.append((qn, t, 10)); rows.append((q, tn, 10))                                           # n_query / n_ref
    n = len(rows)
    pairs = np.zeros(n, dtype=SEQPAIR_DTYPE)
    pairs["len2"] = [len(r[0]) for r in rows]
    pairs["len1"] = [len(r[1]) for r in rows]
    pairs["h0"] = [r[2] for r in rows]
    pairs["idq"] = np.concatenate([[0], np.cumsum(pairs["len2"], dtype=np.int64)[:-1]])
    pairs["idr"] = np.concatenate([[0], np.cumsum(pairs["len1"], dtype=np.int64)[:-1]])
    pairs["id"] = np.arange(n)
    for f in PAIR_FIELDS:
        pairs[f] = -7
    qer = np.concatenate([r[0] for r in rows] + [np.zeros(64, np.uint8)])
    ref = np.concatenate([r[1] for r in rows] + [np.zeros(64, np.uint8)])
    assert (pairs["h0"] >= 0).all() and (pairs["h0"].astype(np.int64) + pairs["len2"].astype(np.int64) * m <= EXT16_TOP).all()
    return pairs, ref, qer


def _seed(name: str) -> int:
    import zlib
    return zlib.crc32(name.encode()) & 0xFFFF


def test_length_generator_hits_the_boundaries():
    """The derived boundaries are where the engine steps, and the pairs land on every one of them."""
    assert long_row_bytes(HBM_QLEN - 1) <= SMEM_ROWS < long_row_bytes(HBM_QLEN)
    assert (stride_class(128), stride_class(129), stride_class(512), stride_class(513)) == (4, 16, 16, 32)
    for name, s in SCHEMES.items():
        pairs, ref, qer = length_pairs(s, _seed(name), QLENS_OF.get(name))
        m = s["match"]
        L, T, h0 = pairs["len2"], pairs["len1"], pairs["h0"].astype(np.int64)
        for q in QLENS_OF.get(name, QLENS):
            if q * m <= EXT16_TOP:
                assert (L == q).any(), (name, q)
                for t in target_lengths(q):
                    assert ((L == q) & (T == t)).any(), (name, q, t)
        assert (T == 32767).any() and (h0 == 0).any()
        top = h0 + L.astype(np.int64) * m
        assert (top == EXT16_TOP).any() and (top <= EXT16_TOP).all()
        assert (L * m >= EXT16_TOP - m).any(), name                          # the exact-match pair at the top
        k16v = (h0 + L * m) * (1 + m)
        long_t = T == 32767
        assert ((k16v == 32767 // (1 + m) * (1 + m)) & long_t).any() and (~k16_eligible(m, L, h0) & long_t).any()
        nq = np.array([(qer[p["idq"]: p["idq"] + p["len2"]] > 3).any() for p in pairs])
        nr = np.array([(ref[p["idr"]: p["idr"] + p["len1"]] > 3).any() for p in pairs])
        assert (nq & ~nr).any() and (nr & ~nq).any()
        assert ((L == HBM_QLEN) & nq).any()
    assert max(BANDS.values()) == (1 << 31) - 1 and CIRC_MAX_W in BANDS.values() and CIRC_MAX_W + 1 in BANDS.values()


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the emulated sweeps with long targets
# ---------------------------------------------------------------------------------------------------------------------
def _with(s: dict, w: int) -> dict:
    return dict(s, w=w)


@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("name", sorted(SCHEMES))
def test_k16_emulation_length_domain(k16, oracle, name, zmode):
    """The packed kernel's sweep on every query the engine gives it (1..824 bases) against targets up to 32767 bases,
    over all bands: whole rows, and circular rows where the engine uses them (w <= 4096), with three fill bytes.  It
    runs exactly the pairs k16::eligible admits, with the oracle's results and effective cells."""
    s0 = SCHEMES[name]
    pairs, ref, qer = length_pairs(s0, _seed(name))
    pairs = pairs[(pairs["len2"] <= SHORT_MAX_QLEN) & ~has_n(pairs, ref, qer)].copy()
    elig = k16_eligible(s0["match"], pairs["len2"], pairs["h0"])
    assert elig.any() and not elig.all() and (pairs["len1"][elig] == 32767).any()
    for bname, w in BANDS.items():
        s = _with(s0, w)
        want, cells_o = oracle_run(oracle, s, zmode, pairs[elig], ref, qer)
        for circ in ((0, 1) if w <= CIRC_MAX_W else (0,)):
            first = None
            for fill in FILLS:
                got = pairs.copy()
                cells, skipped = run_k16(k16, s, zmode, got, ref, qer, circ, fill)
                assert np.array_equal(skipped, ~elig), (bname, circ, fill)
                r = results_matrix(got[elig])
                if first is None:
                    first = r
                assert np.array_equal(r, first), f"{bname} circ {circ}: fill {fill:#x} changed {(r != first).any(axis=1).sum()} pairs"
                bad = (r != results_matrix(want)).any(axis=1)
                assert not bad.any(), f"{bname} circ {circ} fill {fill:#x}: pairs {np.flatnonzero(bad)[:5]} differ"
                assert cells == cells_o, (bname, circ, fill)


@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("name", sorted(SCHEMES))
def test_w16_emulation_length_domain(w16, oracle, name, zmode):
    """The warp-per-pair register kernel's sweep on queries up to w16::MAX_QLEN against targets up to 32767 bases, over
    all bands, three fill bytes: it runs exactly the pairs it admits, with the oracle's results and cells."""
    s0 = SCHEMES[name]
    pairs, ref, qer = length_pairs(s0, _seed(name))
    pairs = pairs[(pairs["len2"] <= W16_MAX_QLEN + 1) & ~has_n(pairs, ref, qer)].copy()
    ok = k16_eligible(s0["match"], pairs["len2"], pairs["h0"]) & (pairs["len2"] <= W16_MAX_QLEN)
    assert ok.any() and not ok.all() and (pairs["len1"][ok] == 32767).any()
    for bname, w in BANDS.items():
        s = _with(s0, w)
        want, cells_o = oracle_run(oracle, s, zmode, pairs[ok], ref, qer)
        first = None
        for fill in FILLS:
            got = pairs.copy()
            cells, skipped = run_w16(w16, s, zmode, got, ref, qer, fill)
            assert np.array_equal(skipped, ~ok), (bname, fill)
            r = results_matrix(got[ok])
            if first is None:
                first = r
            assert np.array_equal(r, first), f"{bname}: fill {fill:#x} changed {(r != first).any(axis=1).sum()} pairs"
            bad = (r != results_matrix(want)).any(axis=1)
            assert not bad.any(), f"{bname} fill {fill:#x}: pairs {np.flatnonzero(bad)[:5]} differ"
            assert cells == cells_o, (bname, fill)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _check(got, want, what):
    bad = (results_matrix(got) != results_matrix(want)).any(axis=1)
    assert not bad.any(), f"{what}: {bad.sum()} pairs differ; first {np.flatnonzero(bad)[:5]}"


def _pin(lib, a, pinned):
    return lib.pinned_copy(a) if pinned else a.copy()


@pytest.mark.gpu
@pytest.mark.parametrize("bname", list(BANDS))
@pytest.mark.parametrize("name", sorted(SCHEMES))
def test_gpu_extend_length_domain(lib, oracle, name, bname):
    """bsw_extend on every route, pageable and page-locked, both z-drop modes: the oracle's six fields and cells.
    Every query longer than SHORT_MAX_QLEN runs on the warp-per-pair byte kernel (its rows in HBM here: the batch
    holds 3064-base and longer queries); with long_min_qlen = 1 every pair does."""
    s = _with(SCHEMES[name], BANDS[bname])
    w = s["w"]
    base, ref, qer = length_pairs(s, _seed(name), QLENS_OF.get(name))
    n_long = int((base["len2"] > SHORT_MAX_QLEN).sum())
    for zmode in (0, 1):
        want, cells_o = oracle_run(oracle, s, zmode, base, ref, qer)
        kw = engine_kw(s, zmode)
        for extra, pinned in (({}, False), ({}, True), ({"short_variant": 1}, False), ({"long_min_qlen": 1}, True),
                              ({"warp_max_pairs": 1 << 20}, False)):
            what = (zmode, extra, pinned)
            with lib.Engine(**kw, **extra) as eng:
                got = _pin(lib, base, pinned)
                eng.extend(got, _pin(lib, ref, pinned), _pin(lib, qer, pinned), w)
                st = eng.stats()
            _check(got, want, what)
            assert st["cells_effective"] == cells_o, what
            assert st["n_long"] == (len(base) if "long_min_qlen" in extra else n_long), what
        # bsw_extend32 promises bsw_extend's results inside the 16-bit domain
        with lib.Engine(**kw) as eng:
            got = base.copy()
            eng.extend32(got, ref, qer, w)
        _check(got, want, ("extend32", zmode))
        # bsw_extend_packed, both record forms: RAW long queries and N pairs, 2-bit short pairs with long targets
        b = lib.PackedBatch.from_pairs(base, ref, qer)
        with lib.Engine(**kw) as eng:
            for compact in (False, True):
                out = eng.extend_packed(b, w, compact=compact)
                mat = np.stack([out[f] for f in PAIR_FIELDS], axis=1).astype(np.int32)
                bad = (mat != results_matrix(want)).any(axis=1)
                assert not bad.any(), f"packed compact={compact} zmode {zmode}: pairs {np.flatnonzero(bad)[:5]} differ"
        # the resident form
        with lib.Engine(**kw) as eng:
            got = base.copy()
            eng.stage(got, ref, qer, w)
            eng.run_staged()
            eng.fetch(got)
        _check(got, want, ("stage", zmode))


@pytest.mark.gpu
def test_gpu_exact_match_at_the_top(lib, oracle):
    """A 32766-base exact match with h0 = 1: score 32767, qle 32766, tle 32766, on every route and both packed forms."""
    s = _with(SCHEMES["bwa"], 100)
    pairs, ref, qer = length_pairs(s, 5)
    top = pairs[(pairs["len2"] == 32766) & (pairs["h0"] == 1) & (pairs["len1"] == 32767)]
    top = top[[(ref[p["idr"]: p["idr"] + 32766] == qer[p["idq"]: p["idq"] + 32766]).all() for p in top]].copy()
    assert len(top) == 1
    want, _ = oracle_run(oracle, s, 0, top, ref, qer)
    assert (want["score"][0], want["qle"][0], want["tle"][0]) == (32767, 32766, 32766)
    for extra in ({}, {"long_min_qlen": 1}, {"tiny_batch": 1}):
        with lib.Engine(**engine_kw(s, 0), **extra) as eng:
            got = top.copy()
            eng.extend(got, ref, qer, 100)
        _check(got, want, extra)
    with lib.Engine(**engine_kw(s, 0)) as eng:
        for compact in (False, True):
            out = eng.extend_packed(lib.PackedBatch.from_pairs(top, ref, qer), 100, compact=compact)
            assert [int(out[f][0]) for f in PAIR_FIELDS] == [int(want[f][0]) for f in PAIR_FIELDS], compact


def _long_batch(rng, qlens, tpad=40):
    """Pairs with the given query lengths, targets mutated copies (+ tpad random bases), h0 in [0, 50]."""
    from genomicsbench_b200 import SEQPAIR_DTYPE
    qs, ts = [], []
    for L in qlens:
        q = rng.integers(0, 4, int(L)).astype(np.uint8)
        t = np.concatenate([mutate(rng, q, 0.05), rng.integers(0, 4, tpad).astype(np.uint8)])
        qs.append(q); ts.append(t)
    n = len(qs)
    pairs = np.zeros(n, dtype=SEQPAIR_DTYPE)
    pairs["len2"] = [len(q) for q in qs]; pairs["len1"] = [len(t) for t in ts]
    pairs["h0"] = rng.integers(0, 51, n)
    pairs["idq"] = np.concatenate([[0], np.cumsum(pairs["len2"], dtype=np.int64)[:-1]])
    pairs["idr"] = np.concatenate([[0], np.cumsum(pairs["len1"], dtype=np.int64)[:-1]])
    pairs["id"] = np.arange(n)
    return pairs, np.concatenate(ts + [np.zeros(64, np.uint8)]), np.concatenate(qs + [np.zeros(64, np.uint8)])


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_gpu_tiny_route_row_limit(lib, oracle, pinned):
    """The latency route keeps a call while bsw_long_kernel's rows fit shared memory: a call whose longest query is
    HBM_QLEN - 1 runs as one kernel; one more base moves it to the general route, which gives the same results."""
    s = _with(SCHEMES["bwa"], 100)
    rng = np.random.default_rng(31)
    for qmax, one_launch in ((HBM_QLEN - 1, True), (HBM_QLEN, False)):
        pairs, ref, qer = _long_batch(rng, list(rng.integers(SHORT_MAX_QLEN + 1, qmax, 63)) + [qmax])
        want, cells_o = oracle_run(oracle, s, 0, pairs, ref, qer)
        with lib.Engine(**engine_kw(s, 0), tiny_batch=len(pairs)) as eng:
            got = _pin(lib, pairs, pinned)
            eng.extend(got, _pin(lib, ref, pinned), _pin(lib, qer, pinned), 100)
            st = eng.stats()
        _check(got, want, (qmax, pinned))
        assert st["cells_effective"] == cells_o and st["n_long"] == len(pairs), qmax
        assert (st["kernel_launches"] == 1) == one_launch, (qmax, st["kernel_launches"])


@pytest.mark.gpu
@pytest.mark.parametrize("w", [100, 4097])
def test_gpu_hbm_rows_for_the_whole_chunk(lib, oracle, w):
    """One query of HBM_QLEN bases among many of 825..HBM_QLEN - 1: the chunk's longest query sets the row stride, so
    every long pair of the chunk runs the HBM row form, on both routes and on bsw_extend_retry."""
    s = _with(SCHEMES["match2_asym"], w)
    rng = np.random.default_rng(32 + w)
    pairs, ref, qer = _long_batch(rng, list(rng.integers(SHORT_MAX_QLEN + 1, HBM_QLEN, 1500)) + [HBM_QLEN])
    for zmode in (0, 1):
        want, cells_o = oracle_run(oracle, s, zmode, pairs, ref, qer)
        for pinned in (False, True):
            with lib.Engine(**engine_kw(s, zmode)) as eng:
                got = _pin(lib, pairs, pinned)
                eng.extend(got, _pin(lib, ref, pinned), _pin(lib, qer, pinned), w)
                st = eng.stats()
            _check(got, want, (zmode, pinned))
            assert st["cells_effective"] == cells_o and st["n_long"] == len(pairs)
        want = pairs.copy()
        band_o = oracle.band_retry(oparams(s, zmode), want, ref, qer, w)
        with lib.Engine(**engine_kw(s, zmode)) as eng:
            got = pairs.copy()
            band = eng.extend_retry(got, ref, qer, w)
        _check(got, want, ("retry", zmode))
        assert np.array_equal(band, band_o)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(SCHEMES))
def test_gpu_retry_length_domain(lib, oracle, name):
    """bsw_extend_retry on the boundary pairs, against the oracle's band-doubling loop."""
    s0 = SCHEMES[name]
    base, ref, qer = length_pairs(s0, _seed(name) + 1, QLENS_OF.get(name))
    for w in (1, 100, CIRC_MAX_W):
        for zmode in (0, 1):
            want = base.copy()
            band_o = oracle.band_retry(oparams(s0, zmode), want, ref, qer, w)
            with lib.Engine(**engine_kw(s0, zmode)) as eng:
                got = base.copy()
                band = eng.extend_retry(got, ref, qer, w)
            _check(got, want, (w, zmode))
            assert np.array_equal(band, band_o), (w, zmode)


# ---- chunks with more than 2^30 bytes of sequence ---------------------------------------------------------------------
N_BIG = 40_000                         # pairs: 40 000 targets of 32767 bases are 1.31e9 bytes, in one chunk of pairs
QLEN_BIG = 900                         # > SHORT_MAX_QLEN: RAW bytes on the staged route


def big_batch(kind: str, layout: str, seed: int = 41):
    """N_BIG pairs against 32767-base targets.  kind "long": 900-base queries (the queries' pairs go RAW); "n_short":
    150-base queries with an N (the N pairs go RAW).  layout "shared": every pair reads target 0 (idr = 0; 33 MB of
    input, but the staged pass gathers 1.31 GB); "consecutive": one target per pair, 1.31 GB of host input.  Each query
    is a mutated window of the target's first 1100 bases.  -> (pairs, ref, qer)"""
    from genomicsbench_b200 import SEQPAIR_DTYPE
    rng = np.random.default_rng(seed)
    T = 32767
    L = QLEN_BIG if kind == "long" else 150
    t = rng.integers(0, 4, T).astype(np.uint8)
    start = rng.integers(0, 200, N_BIG)
    qer = t[start[:, None] + np.arange(L)[None, :]]
    sub = rng.random(qer.shape) < 0.04
    qer[sub] = (qer[sub] + rng.integers(1, 4, int(sub.sum()))) % 4
    if kind == "n_short":
        qer[np.arange(N_BIG), rng.integers(0, L, N_BIG)] = 4
    qer = np.concatenate([qer.ravel(), np.zeros(64, np.uint8)])
    pairs = np.zeros(N_BIG, dtype=SEQPAIR_DTYPE)
    pairs["len2"], pairs["len1"] = L, T
    pairs["h0"] = rng.integers(0, 200, N_BIG)
    pairs["idq"] = np.arange(N_BIG, dtype=np.int64) * L
    if layout == "shared":
        ref = np.concatenate([t, np.zeros(64, np.uint8)])
    else:
        ref = np.concatenate([np.tile(t, N_BIG), np.zeros(64, np.uint8)])
        pairs["idr"] = np.arange(N_BIG, dtype=np.int64) * T
    pairs["id"] = np.arange(N_BIG)
    for f in PAIR_FIELDS:
        pairs[f] = -7
    assert N_BIG * T > RAW_LIMIT
    return pairs, ref, qer


@pytest.mark.gpu
@pytest.mark.parametrize("kind,layout,pinned", [("long", "shared", False), ("long", "shared", True),
                                                ("long", "consecutive", False), ("long", "consecutive", True),
                                                ("n_short", "shared", False), ("n_short", "consecutive", True)])
def test_gpu_chunk_bytes_beyond_2_30(lib, oracle, kind, layout, pinned):
    """A batch inside the domain whose chunk of pairs holds more than 2^30 bytes of a side runs: the staged pass ends
    such a chunk where its bytes still fit 32-bit offsets, and the direct route's retry lands there.  The results equal
    the oracle on a seeded sample, and the same pairs run in calls of one chunk each; bsw_stage runs it too."""
    s = _with(SCHEMES["bwa"], 100)
    pairs, ref, qer = big_batch(kind, layout)
    kw = engine_kw(s, 0)
    with lib.Engine(**kw) as eng:
        got = _pin(lib, pairs, pinned)
        eng.extend(got, lib.pinned_copy(ref) if pinned else ref, lib.pinned_copy(qer) if pinned else qer, s["w"])
        st = eng.stats()
    assert st["pairs"] == N_BIG
    sample = np.sort(np.random.default_rng(42).choice(N_BIG, 2000, replace=False))
    want, _ = oracle_run(oracle, s, 0, pairs[sample], ref, qer)
    _check(got[sample], want, "oracle sample")
    part = 1 << 14                                           # 16384 * 32767 < 2^30: one chunk per call
    small = pairs.copy()
    with lib.Engine(**kw) as eng:
        for a in range(0, N_BIG, part):
            sub = small[a: a + part]
            eng.extend(sub, ref, qer, s["w"])
            small[a: a + part] = sub
    _check(got, small, "one-chunk calls")
    if not pinned:
        with lib.Engine(**kw) as eng:
            staged = pairs.copy()
            eng.stage(staged, ref, qer, s["w"])
            eng.run_staged()
            eng.fetch(staged)
        _check(staged, small, "bsw_stage")

"""bsw_global32: ksw_global2 (tools/bwa/ksw.c:502-606) for alignment regions beyond bsw_global's 32767-base lengths,
one warp per alignment (csrc/bsw_global32.cuh).

CPU: the kernel's row sweep and backtrack (g32::sweep, g32::backtrack) run with the lanes as coroutines
(tests/emu/g32_emu.cu), against every golden case and against oracle/global_oracle.c on alignments outside
bsw_global's domain.
GPU: the entry point against the goldens, bsw_global inside its domain, the oracle on long alignments, chunking, its
domain and call contract, and long-read regions from bsw_extend_chains end to end."""
from __future__ import annotations

import ctypes as C
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from conftest import GOLDEN_DIR
from oracle.pyoracle import make_params
from test_extend32 import LONG_SCORING, _chain_batch, long_reads, mutate      # noqa: F401  (long_reads: fixture)

GOLDEN = sorted(str(p.relative_to(GOLDEN_DIR).with_suffix("")) for d in ("global", "global_emu")
                for p in (GOLDEN_DIR / d).glob("*.npz"))
DEFAULT = dict(match=1, mismatch=4, o_del=6, e_del=1, o_ins=6, e_ins=1, ambig=-1)
ASYM = dict(match=2, mismatch=5, o_del=5, e_del=3, o_ins=4, e_ins=2, ambig=-1)
EDGE = dict(match=1, mismatch=4, o_del=0, e_del=16000, o_ins=0, e_ins=16000, ambig=-1)   # value bound: sum <= 33552
G32_Z_CAP = 2 << 30                           # direction-matrix bytes per chunk
G32_CHUNK_PAIRS = 1 << 16                     # alignments per chunk


def _prm(P: dict) -> np.ndarray:
    return np.array([P["o_del"], P["e_del"], P["o_ins"], P["e_ins"], P["match"], P["mismatch"], P.get("ambig", -1)],
                    dtype=np.int32)


def load_golden(name):
    """-> (P, pairs, ref, qer, w, score, n_cigar, cigar) of tests/golden/<name>.npz (global / global_emu)"""
    from genomicsbench_b200 import SEQPAIR_DTYPE
    z = np.load(GOLDEN_DIR / f"{name}.npz")
    P = dict(zip(("o_del", "e_del", "o_ins", "e_ins", "match", "mismatch", "ambig"), (int(v) for v in z["params"])))
    pairs = np.zeros(len(z["w"]), dtype=SEQPAIR_DTYPE)
    pairs["len1"], pairs["len2"] = z["len1"], z["len2"]
    pairs["idr"] = np.concatenate([[0], np.cumsum(z["len1"])[:-1]])
    pairs["idq"] = np.concatenate([[0], np.cumsum(z["len2"])[:-1]])
    return (P, pairs, np.ascontiguousarray(z["target"]), np.ascontiguousarray(z["query"]), z["w"].astype(np.int32),
            z["score"], z["n_cigar"], z["cigar"])


def make_batch(qs, ts):
    """(queries, targets) -> (pairs, ref, qer) with the sequences laid out one after the other"""
    from genomicsbench_b200 import SEQPAIR_DTYPE
    pairs = np.zeros(len(qs), dtype=SEQPAIR_DTYPE)
    pairs["len2"], pairs["len1"] = [len(q) for q in qs], [len(t) for t in ts]
    pairs["idq"] = np.concatenate([[0], np.cumsum(pairs["len2"].astype(np.int64))[:-1]])
    pairs["idr"] = np.concatenate([[0], np.cumsum(pairs["len1"].astype(np.int64))[:-1]])
    pad = [np.zeros(64, np.uint8)]
    return pairs, np.concatenate(list(ts) + pad), np.concatenate(list(qs) + pad)


def long_set(seed, n, lmin, lmax, err=0.08, wx=(0, 50), n_runs=0, lead=0, w=None):
    """n seeded alignments: a random query, the target a mutated copy (err: substitutions, insertions, deletions),
    optional runs of N in both, optional unrelated leading / trailing pieces (long end indels).  w = |len1 - len2| plus
    a draw from wx, or the fixed w (both are then trimmed to |len1 - len2| <= w / 2).  -> (qs, ts, w int32[n])"""
    rng = np.random.default_rng(seed)
    qs, ts, ws = [], [], []
    for _ in range(n):
        L = int(rng.integers(lmin, lmax + 1))
        q = rng.integers(0, 4, L).astype(np.uint8)
        t = mutate(rng, q, err)
        for _ in range(n_runs):
            a = int(rng.integers(0, L - 100))
            ln = int(rng.integers(5, 80))
            q[a: a + ln] = 4
            t[a: a + ln // 2] = 4
        if lead:
            t = np.concatenate([rng.integers(0, 4, int(rng.integers(lead // 2, lead))).astype(np.uint8), t])
            q = np.concatenate([q, rng.integers(0, 4, int(rng.integers(lead // 2, lead))).astype(np.uint8)])
        if w is not None:
            m = min(len(q), len(t))
            q, t = q[:m + int(rng.integers(0, w // 2 + 1))], t[:m + int(rng.integers(0, w // 2 + 1))]
            ws.append(w)
        else:
            ws.append(abs(len(q) - len(t)) + int(rng.integers(*wx)))
        qs.append(q); ts.append(t)
    return qs, ts, np.array(ws, dtype=np.int32)


def oracle_all(oracle, P: dict, qs, ts, ws, idx=None):
    """oracle.global_align on alignments idx (default all), in parallel -> list of (score, cigar)"""
    Po = make_params(**P)
    idx = range(len(qs)) if idx is None else idx
    with ThreadPoolExecutor(max_workers=16) as ex:
        return list(ex.map(lambda k: oracle.global_align(Po, qs[k], ts[k], int(ws[k])), idx))


def check(score, cigar, off, want, idx):
    for j, k in enumerate(idx):
        sc, cg = want[j]
        assert score[k] == sc, f"alignment {k}: score {score[k]}, oracle {sc}"
        assert np.array_equal(cigar[off[k]: off[k + 1]], cg), f"alignment {k}: cigar differs"


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the emulated sweep and backtrack
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emu(lib, tmp_path_factory):                 # (lib: the product library, which the oracle's build links against)
    """tests/emu/g32_emu.cu compiled as host code (nvcc) into a temporary directory, fresh for every session."""
    import os
    import subprocess
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    out = tmp_path_factory.mktemp("g32_emu") / "libg32_emu.so"
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    env = dict(os.environ)
    env["PATH"] = "/usr/bin:" + env.get("PATH", "")
    subprocess.run([nvcc, "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "-shared",
                    "-Xcompiler", "-fPIC,-pthread", "-I", str(root / "include"), "-o", str(out),
                    str(root / "tests" / "emu" / "g32_emu.cu"), "-lpthread"], check=True, env=env)
    so = C.CDLL(str(out))
    so.g32_emu_batch.restype = C.c_int
    so.g32_emu_batch.argtypes = [C.c_void_p] * 4 + [C.c_longlong, C.c_void_p, C.c_int] + [C.c_void_p] * 4
    so.g32_ring_slots.restype = C.c_int
    so.g32_ring_slots.argtypes = [C.c_int, C.c_int, C.c_int]
    return so


def run_emu(so, P: dict, pairs, ref, qer, w, ring_k=0):
    """-> (score, cigar, off) in global_align's layout"""
    n = len(pairs)
    wv = np.ascontiguousarray(np.broadcast_to(np.asarray(w, dtype=np.int32), (n,)))
    room = np.concatenate([[0], np.cumsum(pairs["len1"].astype(np.int64) + pairs["len2"])]).astype(np.int64)
    buf = np.zeros(int(room[-1]) + 1, np.uint32)
    score, ncig = np.zeros(n, np.int32), np.zeros(n, np.int32)
    rc = so.g32_emu_batch(_prm(P).ctypes.data, pairs.ctypes.data, ref.ctypes.data, qer.ctypes.data, n, wv.ctypes.data,
                          ring_k, score.ctypes.data, ncig.ctypes.data, buf.ctypes.data, room.ctypes.data)
    assert rc == 0, "the lanes of a warp disagreed"
    off = np.concatenate([[0], np.cumsum(ncig)]).astype(np.int64)
    cigar = np.concatenate([buf[room[k]: room[k] + ncig[k]] for k in range(n)] + [np.zeros(0, np.uint32)])
    return score, cigar, off


@pytest.mark.parametrize("name", GOLDEN)
def test_emulated_matches_golden(emu, name):
    P, pairs, ref, qer, w, score_g, ncig_g, cigar_g = load_golden(name)
    score, cigar, off = run_emu(emu, P, pairs, ref, qer, w)
    assert np.array_equal(score, score_g)
    assert np.array_equal(np.diff(off), ncig_g)
    assert np.array_equal(cigar, cigar_g)


# alignments outside bsw_global's domain: (scoring, long_set arguments)
OUTSIDE = {
    "default_33k": (DEFAULT, dict(seed=1, n=8, lmin=33000, lmax=45000, wx=(0, 30))),
    "band_exact": (DEFAULT, dict(seed=2, n=8, lmin=33000, lmax=40000, wx=(0, 1))),             # w = |len1 - len2|
    "band_500": (DEFAULT, dict(seed=3, n=8, lmin=33000, lmax=34000, w=500)),
    "to_200k": (DEFAULT, dict(seed=4, n=2, lmin=150000, lmax=200000, err=0.05, wx=(0, 8))),
    "pacbio": (LONG_SCORING, dict(seed=5, n=8, lmin=33000, lmax=40000, err=0.12, wx=(0, 60))),
    "asym_gaps": (ASYM, dict(seed=6, n=8, lmin=33000, lmax=40000, wx=(0, 60))),
    "n_runs": (DEFAULT, dict(seed=7, n=8, lmin=33000, lmax=40000, n_runs=8, wx=(5, 40))),
    "end_indels": (DEFAULT, dict(seed=8, n=8, lmin=33000, lmax=36000, lead=1000, wx=(0, 40))),
}


@pytest.mark.parametrize("case", sorted(OUTSIDE))
def test_emulated_matches_oracle_outside_global_domain(emu, oracle, case):
    P, kw = OUTSIDE[case]
    qs, ts, ws = long_set(**kw)
    pairs, ref, qer = make_batch(qs, ts)
    assert (np.maximum(pairs["len1"], pairs["len2"]) > 32767).all()
    score, cigar, off = run_emu(emu, P, pairs, ref, qer, ws)
    check(score, cigar, off, oracle_all(oracle, P, qs, ts, ws), range(len(qs)))


def test_emulated_band_edges(emu, oracle):
    """w >= qlen (the whole row, a band wider than both sequences), and w = 0 on equal lengths (the diagonal)."""
    qs, ts, _ = long_set(11, 8, 1500, 2500, err=0.1)
    ws = np.array([max(len(q), len(t)) + 100 * k for k, (q, t) in enumerate(zip(qs, ts))], np.int32)
    ws[-1] = 2 ** 31 - 1
    pairs, ref, qer = make_batch(qs, ts)
    score, cigar, off = run_emu(emu, DEFAULT, pairs, ref, qer, ws)
    check(score, cigar, off, oracle_all(oracle, DEFAULT, qs, ts, np.minimum(ws, 10 ** 6)), range(len(qs)))
    rng = np.random.default_rng(12)
    qs = [rng.integers(0, 5, int(rng.integers(33000, 40000))).astype(np.uint8) for _ in range(6)]
    ts = [np.where(rng.random(len(q)) < 0.1, rng.integers(0, 4, len(q)), q).astype(np.uint8) for q in qs]
    pairs, ref, qer = make_batch(qs, ts)
    score, cigar, off = run_emu(emu, DEFAULT, pairs, ref, qer, 0)
    check(score, cigar, off, oracle_all(oracle, DEFAULT, qs, ts, np.zeros(6, np.int32)), range(6))


def test_emulated_larger_ring(emu, oracle):
    """Any ring of at least the alignment's slots (a multiple of 128) gives the same results: a launch sizes its ring
    for the widest band of the chunk, in shared memory or in the global scratch."""
    qs, ts, ws = long_set(13, 8, 33000, 36000, wx=(0, 100))
    pairs, ref, qer = make_batch(qs, ts)
    want = oracle_all(oracle, DEFAULT, qs, ts, ws)
    need = max(emu.g32_ring_slots(int(p["len2"]), int(p["len1"]), int(w)) for p, w in zip(pairs, ws))
    for k in (need + 128, 4096):
        score, cigar, off = run_emu(emu, DEFAULT, pairs, ref, qer, ws, ring_k=k)
        check(score, cigar, off, want, range(len(qs)))


def test_emulated_value_bound_edge(emu, oracle):
    """(len1 + len2 + 2) * 16000 = 2^29 - 6912: scores near -2^29, still equal to the oracle's."""
    rng = np.random.default_rng(14)
    q = rng.integers(0, 4, 600).astype(np.uint8)
    t = rng.integers(0, 4, 32952).astype(np.uint8)
    t[:600] = q
    pairs, ref, qer = make_batch([q], [t])
    assert (32952 + 600 + 2) * 16000 <= 1 << 29
    score, cigar, off = run_emu(emu, EDGE, pairs, ref, qer, 32952)
    check(score, cigar, off, oracle_all(oracle, EDGE, [q], [t], [32952]), [0])
    assert score[0] < -(1 << 28)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the entry point
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", GOLDEN)
def test_global32_matches_golden(lib, name):
    P, pairs, ref, qer, w, score_g, ncig_g, cigar_g = load_golden(name)
    with lib.Engine(**P) as eng:
        score, cigar, off = eng.global_align32(pairs, ref, qer, w)
        st = eng.stats()
    assert np.array_equal(score, score_g)
    assert np.array_equal(np.diff(off), ncig_g)
    assert np.array_equal(cigar, cigar_g)
    assert st["kernel_launches"] == 4 and st["n_long"] == len(pairs) and st["pairs"] == len(pairs)


@pytest.mark.gpu
def test_global32_equals_global_tiled_goldens(lib):
    """global_default tiled 300 times (210 000 alignments, several chunks): bsw_global's results, the goldens."""
    P, pairs, ref, qer, w, score_g, ncig_g, cigar_g = load_golden("global/global_default")
    big, wb = np.tile(pairs, 300), np.tile(w, 300)
    with lib.Engine(**P) as eng:
        s1, c1, o1 = eng.global_align(big, ref, qer, wb)
        s2, c2, o2 = eng.global_align32(big, ref, qer, wb)
        st = eng.stats()
    assert np.array_equal(s2, s1) and np.array_equal(o2, o1) and np.array_equal(c2, c1)
    assert np.array_equal(s2, np.tile(score_g, 300)) and np.array_equal(c2, np.tile(cigar_g, 300))
    assert st["kernel_launches"] == 4 * -(-len(big) // G32_CHUNK_PAIRS)
    l1, l2, wc = big["len1"].astype(np.int64), big["len2"].astype(np.int64), wb.astype(np.int64)
    cells = sum(int(((np.minimum(i + wc + 1, l2) - np.maximum(i - wc, 0)) * (i < l1)).sum()) for i in range(int(l1.max())))
    assert st["cells_effective"] == cells and st["cells_nominal"] == int((l1 * l2).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("params", [DEFAULT, ASYM, LONG_SCORING])
def test_global32_equals_global_in_domain(lib, params):
    """Random alignments up to 32 767 bases with bands up to 1 500 (bsw_global's first kernel, rows in HBM)."""
    rng = np.random.default_rng(0xB5B23200 + params["e_del"])
    qs, ts, ws = [], [], []
    for _ in range(120):
        L = int(rng.integers(50, 32000))
        q = rng.integers(0, 5 if rng.random() < 0.2 else 4, L).astype(np.uint8)
        t = mutate(rng, q, float(rng.uniform(0.01, 0.2)))[:32767]
        d = abs(len(q) - len(t))
        assert d <= 1500
        qs.append(q); ts.append(t); ws.append(int(rng.integers(d, 1501)))
    pairs, ref, qer = make_batch(qs, ts)
    with lib.Engine(**params) as eng:
        s1, c1, o1 = eng.global_align(pairs, ref, qer, ws)
        s2, c2, o2 = eng.global_align32(pairs, ref, qer, ws)
    assert np.array_equal(s2, s1) and np.array_equal(o2, o1) and np.array_equal(c2, c1)


# (seed, n, lmin, lmax, w): long alignments against the oracle; "wide_ring" has K = 8064 ring slots, 4 rings of which
# exceed a block's shared memory: the global-scratch variant
LONG = {
    "to_2e5": dict(seed=31, n=6, lmin=100000, lmax=200000, w=100),
    "mega": dict(seed=32, n=1, lmin=1000000, lmax=1000000, w=100),
    "wide_ring": dict(seed=33, n=4, lmin=30000, lmax=40000, w=4000),
    "mixed": dict(seed=34, n=40, lmin=5000, lmax=80000, wx=(0, 300), n_runs=3),
}


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("case", sorted(LONG))
def test_global32_matches_oracle_long(lib, oracle, case, pinned):
    qs, ts, ws = long_set(**LONG[case])
    pairs, ref, qer = make_batch(qs, ts)
    if pinned:
        pairs, ref, qer = lib.pinned_copy(pairs), lib.pinned_copy(ref), lib.pinned_copy(qer)
    with lib.Engine(**DEFAULT) as eng:
        score, cigar, off = eng.global_align32(pairs, ref, qer, ws)
    idx = range(len(qs)) if len(qs) <= 8 else range(0, len(qs), 5)
    check(score, cigar, off, oracle_all(oracle, DEFAULT, qs, ts, ws, idx), idx)
    if case == "mega":
        assert len(qs[0]) >= 10 ** 6


@pytest.mark.gpu
def test_global32_cut_by_matrix_bytes(lib, oracle):
    """60 alignments of ~100 kb at w = 2000 (~205 MB of directions each): a call cut into several chunks by the
    per-chunk matrix cap gives the results of one call per chunk, and the oracle's on a sample."""
    qs, ts, ws = long_set(41, 60, 98000, 102000, err=0.05, w=2000)
    pairs, ref, qer = make_batch(qs, ts)
    zb = pairs["len1"].astype(np.int64) * 64 * ((np.minimum(pairs["len2"], 2 * ws + 1).astype(np.int64) + 3 + 127) // 128)
    cuts, acc = [0], 0
    for k, b in enumerate(zb):
        if acc + b > G32_Z_CAP:
            cuts.append(k); acc = 0
        acc += int(b)
    cuts.append(len(qs))
    assert len(cuts) - 1 >= 5
    with lib.Engine(**DEFAULT) as eng:
        score, cigar, off = eng.global_align32(pairs, ref, qer, ws)
        st = eng.stats()
        assert st["kernel_launches"] == 4 * (len(cuts) - 1)
        for a, b in zip(cuts[:-1], cuts[1:]):
            s, c, o = eng.global_align32(pairs[a:b], ref, qer, ws[a:b])
            assert np.array_equal(s, score[a:b])
            assert np.array_equal(c, cigar[off[a]: off[b]]) and np.array_equal(o + off[a], off[a: b + 1])
    idx = list(range(0, 60, 12))
    check(score, cigar, off, oracle_all(oracle, DEFAULT, qs, ts, ws, idx), idx)


@pytest.mark.gpu
def test_global32_contract(lib):
    P, pairs, ref, qer, w, score_g, ncig_g, cigar_g = load_golden("global/global_default")
    big, wb = np.tile(pairs, 300), np.tile(w, 300)
    n = len(big)
    with lib.Engine(**P) as eng:
        # a cigar buffer that holds the first chunk but not the call: refused after the first chunk's results are out
        cap = int(np.tile(ncig_g, 300)[:G32_CHUNK_PAIRS].sum())
        out = (np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(cap, np.uint32), np.zeros(n + 1, np.int64))
        with pytest.raises(lib.BswError) as ei:
            eng.global_align32(big, ref, qer, wb, out=out)
        assert ei.value.code == -1 and "cigar buffer too small" in str(ei.value)
        assert np.array_equal(out[0][:G32_CHUNK_PAIRS], np.tile(score_g, 300)[:G32_CHUNK_PAIRS])
        assert np.array_equal(out[2], np.tile(cigar_g, 300)[:cap])
        score, cigar, off = eng.global_align32(big, ref, qer, wb)
        assert np.array_equal(score, np.tile(score_g, 300)) and np.array_equal(cigar, np.tile(cigar_g, 300))
        # the empty batch
        s0, c0, o0 = eng.global_align32(big[:0], ref, qer, 10)
        assert len(s0) == 0 and len(c0) == 0 and list(o0) == [0]
        assert eng.stats()["pairs"] == 0
        # the domain: |len1 - len2| > w, lengths beyond 2^24 - 1, a negative band
        for field, value, wv in (("len1", int(big["len2"][2]) + 11, 10), ("len1", 1 << 24, 1 << 24), ("len2", 1 << 24, 1 << 24),
                                 ("len1", 0, 300), ("idr", -1, 300), ("len1", 100, -1)):
            bad = big[:4].copy()
            bad[2][field] = value
            if field == "len1" and value == 1 << 24:
                bad[2]["len2"] = (1 << 24) - 1
            with pytest.raises(lib.BswError) as ei:
                eng.global_align32(bad, ref, qer, wv)
            assert ei.value.code == -2, (field, value)
        # bad arguments
        assert eng._lib.bsw_global32(eng._h, None, None, None, 3, None, None, None, None, 0, None) == -1
        assert eng._lib.bsw_global32(eng._h, big.ctypes.data, ref.ctypes.data, qer.ctypes.data, 3, wb.ctypes.data,
                                     out[0].ctypes.data, out[1].ctypes.data, out[2].ctypes.data, -1, out[3].ctypes.data) == -1
        assert eng._lib.bsw_global32(None, None, None, None, 0, None, None, None, None, 0, None) == -1
    # the value bound: (len1 + len2 + 2) * 16000 <= 2^29 holds for 600 + 32952 bases and fails for one more
    rng = np.random.default_rng(15)
    q = rng.integers(0, 4, 600).astype(np.uint8)
    t = rng.integers(0, 4, 32953).astype(np.uint8)
    pairs, ref, qer = make_batch([q, q], [t[:32952], t])
    with lib.Engine(**EDGE) as eng:
        s, c, o = eng.global_align32(pairs[:1], ref, qer, 32952)
        assert s[0] < -(1 << 28)
        with pytest.raises(lib.BswError) as ei:
            eng.global_align32(pairs, ref, qer, 32953)
        assert ei.value.code == -2


@pytest.mark.gpu
def test_global32_long_read_regions(lib, oracle, long_reads):
    """bsw_extend_chains on the 20-120 kb reads, then every region's CIGAR (bwa_gen_cigar2's ksw_global2 call) with
    w = max(region w, |len1 - len2| + 3): equal to the oracle; bsw_global refuses the regions beyond 32 767 bases."""
    L, D, reads = long_reads
    w = 100
    with lib.Engine(end_bonus=0, zdrop_mode=lib.BSW_ZDROP_SCALAR, **LONG_SCORING) as eng:
        chains, seeds, query, ref = _chain_batch(lib, eng, reads, D, L, w, 1)
        regs, count = eng.extend_chains(chains, seeds, query, ref, w, 0, 0, 2)
        qs, ts, ws = [], [], []
        for k, ch in enumerate(chains):
            read = query[int(ch["query_off"]): int(ch["query_off"]) + int(ch["l_query"])]
            for r in regs[int(ch["seed_first"]): int(ch["seed_first"]) + int(count[k])]:
                q, t = read[int(r["qb"]): int(r["qe"])], D[int(r["rb"]): int(r["re"])]
                if len(q) == 0 or len(t) == 0:
                    continue
                qs.append(q); ts.append(t); ws.append(max(int(r["w"]), abs(len(q) - len(t)) + 3))
        ws = np.array(ws, np.int32)
        pairs, rseq, qseq = make_batch(qs, ts)
        score, cigar, off = eng.global_align32(pairs, rseq, qseq, ws)
        longest = int(np.argmax(np.maximum(pairs["len1"], pairs["len2"])))
        assert max(pairs["len1"][longest], pairs["len2"][longest]) > 32767
        with pytest.raises(lib.BswError) as ei:
            eng.global_align(pairs[longest: longest + 1], rseq, qseq, ws[longest: longest + 1])
        assert ei.value.code == -2
    check(score, cigar, off, oracle_all(oracle, LONG_SCORING, qs, ts, ws), range(len(qs)))

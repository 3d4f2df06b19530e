"""bsw_extend32: ksw_extend2 with int32 scores for pairs outside bsw_extend's 16-bit domain (long-read flanks), and
bsw_extend_chains on reads beyond that domain.

CPU: the kernel's row sweep (l32::sweep, bsw_long32.cuh) run with the lanes as coroutines (tests/emu/l32_emu.cu),
against every golden set and against the int32 oracle (oracle/ksw_oracle.c) on pairs outside the 16-bit domain.
GPU: the entry point against the goldens, bsw_extend, the oracle, its domain and contract; long-read chains against
oracle/chain_oracle.c."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from conftest import GOLDEN_CASES, load_golden, results_matrix

DEFAULT = dict(match=1, mismatch=4, o_del=6, e_del=1, o_ins=6, e_ins=1, zdrop=100, end_bonus=5, ambig=-1)


@pytest.fixture(scope="module")
def emu(lib, tmp_path_factory):                 # (lib: the product library, which the oracle's build links against)
    """tests/emu/l32_emu.cu compiled as host code (nvcc) into a temporary directory, fresh for every session: the sweep
    it runs is the kernel header's own source."""
    import os
    import subprocess
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    out = tmp_path_factory.mktemp("l32_emu") / "libl32_emu.so"
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    env = dict(os.environ)
    env["PATH"] = "/usr/bin:" + env.get("PATH", "")
    subprocess.run([nvcc, "-std=c++17", "-O2", "-gencode", "arch=compute_100a,code=sm_100a", "-shared",
                    "-Xcompiler", "-fPIC,-pthread", "-I", str(root / "include"), "-o", str(out),
                    str(root / "tests" / "emu" / "l32_emu.cu"), "-lpthread"], check=True, env=env)
    so = C.CDLL(str(out))
    so.l32_emu_batch.restype = C.c_longlong
    so.l32_emu_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int]
    so.l32_ring_slots.restype = C.c_int
    so.l32_ring_slots.argtypes = [C.c_void_p, C.c_int, C.c_int]
    return so


def _prm_array(prm: dict, zmode: int) -> np.ndarray:
    return np.array([prm["match"], prm["mismatch"], prm["o_del"], prm["e_del"], prm["o_ins"], prm["e_ins"],
                     prm["zdrop"], prm["end_bonus"], zmode, prm.get("ambig", -1)], dtype=np.int32)


def run_emu(lib, prm: dict, pairs, ref, qer, w, zmode=0, ring_k=0) -> int:
    cells = lib.l32_emu_batch(_prm_array(prm, zmode).ctypes.data, pairs.ctypes.data, ref.ctypes.data, qer.ctypes.data,
                              len(pairs), w, ring_k)
    assert cells >= 0, "the lanes of a warp disagreed"
    return int(cells)


def oracle_params(prm: dict, zmode: int):
    from oracle.pyoracle import make_params
    return make_params(**prm, zdrop_mode=zmode)


def mutate(rng, s: np.ndarray, err: float, n_rate: float = 0.0) -> np.ndarray:
    """s with substitutions, single-base insertions and deletions at rate err in total (a third each)."""
    u = rng.random(len(s) + len(s) // 2 + 8)
    kind = np.where(u < err / 3, 1, np.where(u < 2 * err / 3, 2, np.where(u < err, 3, 0)))    # match, sub, ins, del
    adv = (kind != 2).astype(np.int64)
    pos = np.cumsum(adv) - adv
    keep = pos < len(s)
    kind, pos = kind[keep], pos[keep]
    base = s[pos].astype(np.int64)
    base = np.where(kind == 1, (base + rng.integers(1, 4, len(kind))) % 4, base)
    base = np.where(kind == 2, rng.integers(0, 4, len(kind)), base)
    a = base[kind != 3].astype(np.uint8)
    if n_rate > 0:
        a[rng.random(len(a)) < n_rate] = 4
    return a


def long_pairs(seed: int, n: int, lmin: int, lmax: int, h0=(0, 100), err=0.08, n_rate=0.0, n_runs=0, junk_tail=0.0):
    """Seeded pairs: a random query, the target a mutated copy of it (so scores grow along the band), optional runs
    of N, optional unrelated tails (the window shrinks, z-drop fires).  -> (pairs, ref, qer)"""
    from genomicsbench_b200 import SEQPAIR_DTYPE
    rng = np.random.default_rng(seed)
    pairs = np.zeros(n, dtype=SEQPAIR_DTYPE)
    qs, ts = [], []
    qo = ro = 0
    for k in range(n):
        L = int(rng.integers(lmin, lmax + 1))
        q = rng.integers(0, 4, L).astype(np.uint8)
        t = mutate(rng, q, err, n_rate)
        if junk_tail and rng.random() < junk_tail:
            cut = int(rng.integers(len(t) // 3, len(t)))
            t[cut:] = rng.integers(0, 4, len(t) - cut)
        for _ in range(n_runs):
            a = int(rng.integers(0, len(q)))
            q[a: a + int(rng.integers(5, 60))] = 4
        t = t[:max(1, len(t))]
        pairs[k]["idq"], pairs[k]["idr"] = qo, ro
        pairs[k]["len2"], pairs[k]["len1"] = len(q), len(t)
        pairs[k]["h0"] = int(rng.integers(h0[0], h0[1] + 1))
        qs.append(q); ts.append(t)
        qo += len(q); ro += len(t)
    qer = np.concatenate(qs + [np.zeros(64, np.uint8)])
    ref = np.concatenate(ts + [np.zeros(64, np.uint8)])
    pairs["id"] = np.arange(n)
    for f in ("score", "qle", "tle", "gtle", "gscore", "max_off"):
        pairs[f] = -7
    return pairs, ref, qer


def in16(pairs, match) -> np.ndarray:
    return ((pairs["len1"] <= 32767) & (pairs["len2"] <= 32767) &
            (pairs["h0"].astype(np.int64) + pairs["len2"].astype(np.int64) * match <= 32767))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the emulated sweep
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_emulated_sweep_matches_golden(emu, name, zmode):
    pairs, ref, qer, w, prm, expect, scalar = load_golden(name)
    if zmode == 0 and prm["zdrop"] < 1:
        pytest.skip("vector z-drop needs zdrop >= 1")
    want = expect if zmode == 0 else scalar
    step = max(1, len(pairs) // 200)
    pairs, want = pairs[::step].copy(), want[::step]
    run_emu(emu, prm, pairs, ref, qer, w, zmode=zmode)
    got = results_matrix(pairs)
    assert np.array_equal(got, want), f"{name}: {(got != want).any(axis=1).sum()} pairs differ"


# item 2 of the sets outside the 16-bit domain: (seed, n, lmin, lmax, h0 range, w, extra generator args)
OUTSIDE = {
    "h0_high": (11, 40, 200, 3000, (30000, 200000), 100, {}),
    "long_w1": (12, 2, 33000, 70000, (0, 50), 1, {}),
    "long_w8": (13, 2, 33000, 70000, (0, 50), 8, {}),
    "long_w50": (14, 2, 33000, 70000, (0, 50), 50, {}),
    "w_ge_qlen": (15, 6, 100, 900, (33000, 90000), 1000, {}),
    "n_runs": (16, 3, 33000, 45000, (0, 50), 50, dict(n_runs=6, n_rate=0.002)),
    "virgin": (17, 30, 300, 4000, (60000, 200000), 3, {}),
    "stale": (18, 20, 2000, 9000, (40000, 60000), 20, dict(junk_tail=0.7, err=0.15)),
}


@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("case", sorted(OUTSIDE))
def test_emulated_sweep_matches_oracle_outside_16bit(emu, oracle, case, zmode):
    seed, n, lmin, lmax, h0, w, kw = OUTSIDE[case]
    pairs, ref, qer = long_pairs(seed, n, lmin, lmax, h0, **kw)
    assert not in16(pairs, 1).any()
    want = pairs.copy()
    cells_o = oracle.batch(oracle_params(DEFAULT, zmode), want, ref, qer, w)
    cells = run_emu(emu, DEFAULT, pairs, ref, qer, w, zmode=zmode)
    assert np.array_equal(results_matrix(pairs), results_matrix(want))
    assert cells == cells_o
    if case == "virgin":
        # the first row's non-zero prefix (h0 / e_ins columns) is longer than the ring: the virgin-cell rule is exercised
        k = np.array([emu.l32_ring_slots(_prm_array(DEFAULT, zmode).ctypes.data, int(l2), w) for l2 in pairs["len2"]])
        assert ((pairs["h0"] - 7) > k).all()


@pytest.mark.parametrize("e_del,e_ins", [(1, 1), (2, 3), (3, 2)])
@pytest.mark.parametrize("zdrop", [1, 20, 100, 32767])
@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("match", [1, 2])
def test_emulated_sweep_scorings_outside_16bit(emu, oracle, e_del, e_ins, zdrop, zmode, match):
    prm = dict(DEFAULT, match=match, e_del=e_del, e_ins=e_ins, zdrop=zdrop)
    pairs, ref, qer = long_pairs(100 + 7 * e_del + e_ins + zdrop + match, 6, 300, 2500, (33000, 80000), err=0.1,
                                 n_rate=0.003, junk_tail=0.3)
    want = pairs.copy()
    cells_o = oracle.batch(oracle_params(prm, zmode), want, ref, qer, 30)
    cells = run_emu(emu, prm, pairs, ref, qer, 30, zmode=zmode)
    assert np.array_equal(results_matrix(pairs), results_matrix(want))
    assert cells == cells_o


def test_emulated_sweep_forced_larger_ring(emu, oracle):
    """Any ring of at least ring_slots slots (a multiple of the chunk width) gives the same results: the launch sizes
    its ring for the widest band of a chunk."""
    pairs, ref, qer = long_pairs(21, 8, 500, 3000, (40000, 90000), junk_tail=0.5)
    want = pairs.copy()
    oracle.batch(oracle_params(DEFAULT, 1), want, ref, qer, 10)
    for k in (128, 384, 1024):
        got = pairs.copy()
        run_emu(emu, DEFAULT, got, ref, qer, 10, zmode=1, ring_k=k)
        assert np.array_equal(results_matrix(got), results_matrix(want)), k


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the entry point
# ---------------------------------------------------------------------------------------------------------------------
def _engine(lib, prm: dict, zmode: int):
    return lib.Engine(zdrop_mode=zmode, **prm)


@pytest.mark.gpu
@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_extend32_matches_golden(lib, name, zmode):
    pairs, ref, qer, w, prm, expect, scalar = load_golden(name)
    if zmode == 0 and prm["zdrop"] < 1:
        pytest.skip("vector z-drop needs zdrop >= 1")
    with _engine(lib, prm, zmode) as eng:
        eng.extend32(pairs, ref, qer, w)
    got = results_matrix(pairs)
    want = expect if zmode == 0 else scalar
    assert np.array_equal(got, want), f"{name}: {(got != want).any(axis=1).sum()} pairs differ"


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("config,w", [("short8", 100), ("long16", 100), ("large", 100), ("sweep", 500)])
def test_extend32_equals_extend_inside_16bit(lib, oracle, config, w, zmode, pinned):
    cfg = lib.gen_named_config(config)
    pairs, ref, qer = lib.gen_pairs(cfg, 4242, 20000)
    if pinned:
        pairs, ref, qer = lib.pinned_copy(pairs), lib.pinned_copy(ref), lib.pinned_copy(qer)
    a, b, want = pairs.copy(), pairs.copy(), pairs.copy()
    cells_o = oracle.batch(oracle_params(DEFAULT, zmode), want, ref, qer, w)
    with _engine(lib, DEFAULT, zmode) as eng:
        eng.extend(a, ref, qer, w)
        if pinned:
            b = lib.pinned_copy(b)
        eng.extend32(b, ref, qer, w)
        st = eng.stats()
    assert np.array_equal(results_matrix(b), results_matrix(a))
    assert np.array_equal(results_matrix(b), results_matrix(want))
    assert st["cells_effective"] == cells_o
    assert st["pairs"] == len(pairs) and st["kernel_launches"] >= 1
    assert st["cells_nominal"] == int((pairs["len1"].astype(np.int64) * pairs["len2"]).sum())


LARGER = {
    "to_2e5": (31, 6, 100000, 200000, (0, 100), 100, {}),
    "mega": (32, 1, 1000000, 1000000, (0, 50), 100, {}),
}


@pytest.mark.gpu
@pytest.mark.parametrize("zmode", [0, 1])
@pytest.mark.parametrize("case", sorted(OUTSIDE) + sorted(LARGER))
def test_extend32_matches_oracle_outside_16bit(lib, oracle, case, zmode):
    seed, n, lmin, lmax, h0, w, kw = {**OUTSIDE, **LARGER}[case]
    pairs, ref, qer = long_pairs(seed, n, lmin, lmax, h0, **kw)
    want = pairs.copy()
    cells_o = oracle.batch(oracle_params(DEFAULT, zmode), want, ref, qer, w)
    with _engine(lib, DEFAULT, zmode) as eng:
        eng.extend32(pairs, ref, qer, w)
        st = eng.stats()
    assert np.array_equal(results_matrix(pairs), results_matrix(want))
    assert st["cells_effective"] == cells_o
    if case == "mega":
        assert pairs["len2"][0] >= 10 ** 6 and pairs["score"][0] > 32767


@pytest.mark.gpu
def test_extend32_global_ring(lib, oracle):
    """A band whose ring does not fit shared memory (4 rings of 2 K ints > 200 KB for K > 6400) runs the global-ring
    variant: same results and cells as the oracle, with a ring narrower than the row (w = 4000) and the whole row."""
    pairs, ref, qer = long_pairs(41, 12, 9000, 20000, (33000, 60000), err=0.12, junk_tail=0.4)
    for w in (4000, 1 << 14):
        for zmode in (0, 1):
            want = pairs.copy()
            cells_o = oracle.batch(oracle_params(DEFAULT, zmode), want, ref, qer, w)
            got = pairs.copy()
            with _engine(lib, DEFAULT, zmode) as eng:
                eng.extend32(got, ref, qer, w)
                assert eng.stats()["cells_effective"] == cells_o
            assert np.array_equal(results_matrix(got), results_matrix(want)), (w, zmode)


@pytest.mark.gpu
def test_extend32_domain_and_contract(lib):
    pairs, ref, qer = long_pairs(51, 20, 100, 3000, (0, 40000))
    with _engine(lib, DEFAULT, 0) as eng:
        for field, value in (("len1", 0), ("len2", 0), ("len1", 1 << 24), ("len2", 1 << 24), ("h0", -1),
                             ("h0", (1 << 30) - 5 - 100)):
            bad = pairs.copy()
            bad[3][field] = value
            if field == "h0" and value > 0:
                bad[3]["len2"] = 101                               # h0 + len2 * 1 + end_bonus = 2^30 + 1
            before = bad.copy()
            with pytest.raises(lib.BswError) as ei:
                eng.extend32(bad, ref, qer, 50)
            assert ei.value.code == lib._lib.BSW_ERR_DOMAIN
            assert np.array_equal(bad, before)                    # nothing written on a refusal
        eng.extend32(pairs[:0], ref, qer, 50)                     # n = 0
        assert eng.stats()["pairs"] == 0
        # the engine is usable afterwards; records beyond n and the input fields are untouched
        buf = pairs.copy()
        buf["seqid"], buf["regid"] = 11, 22
        before = buf.copy()
        eng.extend32(buf[:15], ref, qer, 50)
        assert np.array_equal(buf[15:], before[15:])
        for f in ("idr", "idq", "id", "len1", "len2", "h0", "seqid", "regid"):
            assert np.array_equal(buf[f], before[f]), f
        assert (buf["score"][:15] >= 0).all()
        with pytest.raises(lib.BswError):
            eng.extend32(buf, ref, qer, -1)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: bsw_extend_chains on long reads
# ---------------------------------------------------------------------------------------------------------------------
def make_long_reads(rng, D, L, n_reads, lmin, lmax, err):
    """Reads of lmin..lmax bases cut from either strand of D with substitutions, insertions and deletions (a third of
    err each), a few N; seeds = the exact runs of at least 19 bases of the true alignment plus contained (same
    diagonal) and shifted-diagonal extras -- the seeds of tests/golden/make_golden_chain.make_reads at long-read
    lengths.  -> list of (read codes, seeds[(rbeg, qbeg, len)])."""
    out = []
    for _ in range(n_reads):
        rl = int(rng.integers(lmin, lmax + 1))
        strand = int(rng.integers(0, 2))
        lo, hi = strand * L, (strand + 1) * L
        start = int(rng.integers(lo, hi - 2 * rl))
        r = float(rng.uniform(*err))
        u = rng.random(2 * rl)
        kind = np.where(u < r / 3, 1, np.where(u < 2 * r / 3, 2, np.where(u < r, 3, 0)))   # match, sub, ins, del
        adv = (kind != 2).astype(np.int64)
        pos = start + np.cumsum(adv) - adv
        emit = kind != 3
        base = D[pos].astype(np.int64)
        base = np.where(kind == 1, (base + 1 + rng.integers(0, 3, len(kind))) % 4, base)
        base = np.where(kind == 2, rng.integers(0, 4, len(kind)), base)
        read = base[emit][:rl].astype(np.uint8)
        qidx = np.cumsum(emit) - 1
        k_e, p_e, q_e = kind[emit][:rl], pos[emit][:rl], qidx[emit][:rl]
        m = (k_e == 0).astype(np.int8)
        edges = np.flatnonzero(np.diff(np.concatenate([[0], m, [0]])))
        seeds = []
        for a, b in zip(edges[0::2], edges[1::2]):
            if b - a >= 19:
                seeds.append((int(p_e[a]), int(q_e[a]), int(b - a)))
        extra = []
        for rb, qb, ln in seeds:
            v = rng.random()
            if ln >= 30 and v < 0.25:
                off = int(rng.integers(1, ln - 20))
                extra.append((rb + off, qb + off, int(rng.integers(15, ln - off + 1))))
            elif ln >= 24 and v < 0.40:
                sh = int(rng.choice([-3, -2, -1, 1, 2, 3]))
                if lo <= rb + sh and rb + sh + ln <= hi:
                    extra.append((rb + sh, qb, ln - int(rng.integers(0, 3))))
        seeds = sorted(set(seeds + extra), key=lambda s: (s[1], s[0]))
        for p in rng.integers(0, len(read), size=int(rng.integers(0, 6))):
            read[p] = 4
        out.append((read, seeds))
    return out


def _chain_batch(lib, eng, reads, D, l_pac, w, match):
    """One chain per read in the C ABI's layout (windows from bsw_chain_window)."""
    chains = np.zeros(len(reads), dtype=lib.CHAIN_DTYPE)
    seeds = np.zeros(sum(len(s) for _, s in reads), dtype=lib.SEED_DTYPE)
    qparts, rparts, qo, ro, so = [], [], 0, 0, 0
    for k, (read, sd) in enumerate(reads):
        for i, (rb, qb, ln) in enumerate(sd):
            seeds[so + i] = (rb, qb, ln, ln * match, 0)
        r0, r1 = eng.chain_window(w, l_pac, seeds[so: so + len(sd)], len(read))
        chains[k] = (so, len(sd), len(read), qo, r0, r1, ro, 0, 0)
        qparts.append(read); rparts.append(D[r0:r1])
        qo += len(read); ro += r1 - r0; so += len(sd)
    return chains, seeds, np.concatenate(qparts), np.concatenate(rparts)


def _oracle_chains(oracle, P, chains, seeds, query, ref, w, clip, l_pac):
    from concurrent.futures import ThreadPoolExecutor
    from oracle.pyoracle import CHAIN_SEED_DTYPE

    def one(ch):
        sd = np.zeros(int(ch["n_seeds"]), dtype=CHAIN_SEED_DTYPE)
        src = seeds[int(ch["seed_first"]): int(ch["seed_first"]) + int(ch["n_seeds"])]
        for f in ("rbeg", "qbeg", "len", "score"):
            sd[f] = src[f]
        q = query[int(ch["query_off"]): int(ch["query_off"]) + int(ch["l_query"])]
        r0, r1 = int(ch["rmax0"]), int(ch["rmax1"])
        rs = ref[int(ch["ref_off"]): int(ch["ref_off"]) + r1 - r0]
        return oracle.chain(P, w, clip, clip, 2, q, sd, r0, r1, rs)

    with ThreadPoolExecutor(max_workers=16) as ex:
        return list(ex.map(one, chains))


def _check_chains(lib, chains, regs, count, want, skip=()):
    for k, ch in enumerate(chains):
        if k in skip:
            continue
        got = regs[int(ch["seed_first"]): int(ch["seed_first"]) + int(count[k])]
        assert int(count[k]) == len(want[k]), f"chain {k}: {count[k]} regions, oracle {len(want[k])}"
        gm = np.stack([got[f] for f in lib.ALNREG_FIELDS], axis=1).astype(np.int64).reshape(-1, len(lib.ALNREG_FIELDS))
        from oracle.pyoracle import CHAIN_REG_FIELDS
        wm = np.stack([want[k][f] for f in CHAIN_REG_FIELDS], axis=1).astype(np.int64).reshape(-1, len(CHAIN_REG_FIELDS))
        assert np.array_equal(gm, wm), f"chain {k}"


LONG_SCORING = dict(match=1, mismatch=1, o_del=1, e_del=1, o_ins=1, e_ins=1, zdrop=100)    # bwa -x pacbio (-L0)


@pytest.fixture(scope="module")
def long_reads():
    rng = np.random.default_rng(2026)
    L = 3_000_000
    G = rng.integers(0, 4, size=L, dtype=np.uint8)
    D = np.concatenate([G, (3 - G[::-1]).astype(np.uint8)])
    return L, D, make_long_reads(rng, D, L, 100, 20000, 120000, (0.05, 0.12))


@pytest.mark.gpu
@pytest.mark.parametrize("zmode", [1, 0])
def test_extend_chains_long_reads_match_oracle(lib, oracle, long_reads, zmode):
    """Reads of 20-120 kb: the flanks leave the 16-bit domain and run through bsw_extend32; every region equals
    chain_oracle's.  Scalar mode, and the vector mode, which agrees with it for unit gap extension."""
    from oracle.pyoracle import make_params
    L, D, reads = long_reads
    w, clip = 100, 0
    with lib.Engine(end_bonus=clip, zdrop_mode=zmode, **LONG_SCORING) as eng:
        chains, seeds, query, ref = _chain_batch(lib, eng, reads, D, L, w, 1)
        regs, count = eng.extend_chains(chains, seeds, query, ref, w, clip, clip, 2)
        st = eng.stats()
    want = _oracle_chains(oracle, make_params(end_bonus=clip, zdrop_mode=1, **LONG_SCORING), chains, seeds, query, ref,
                          w, clip, L)
    _check_chains(lib, chains, regs, count, want)
    assert (regs["score"][:int(count.sum())] > 32767).sum() > 0 or (regs["qe"] - regs["qb"] > 32767).any()
    assert st["n_long"] > 0


@pytest.mark.gpu
def test_extend_chains_mixed_short_and_long(lib, oracle, long_reads):
    """Golden short chains (repeated until the batch is cut into several lanes) and 30 long reads in one batch, with
    bwa's default scoring: the short chains keep their golden regions, the long ones equal the oracle."""
    from test_chain import _build_batch, load_chain_case
    from oracle.pyoracle import make_params
    c = load_chain_case("chain_default")
    L, D, reads = long_reads
    P = c["P"]
    w, clip = c["w"], c["clip5"]
    lreads = reads[:30]
    with lib.Engine(end_bonus=clip, zdrop_mode=lib.BSW_ZDROP_SCALAR, **P) as eng:
        gch, gseeds, gq, gr = _build_batch(lib, eng, c)
        lch, lseeds, lq, lr = _chain_batch(lib, eng, lreads, D, L, w, P["match"])
        reps = max(1, 25000 // len(gch))
        parts_ch, parts_sd = [], []
        for k in range(reps):
            ch = gch.copy(); ch["seed_first"] += k * len(gseeds)
            parts_ch.append(ch); parts_sd.append(gseeds)
        ch = lch.copy()
        ch["seed_first"] += reps * len(gseeds); ch["query_off"] += len(gq); ch["ref_off"] += len(gr)
        chains = np.concatenate(parts_ch + [ch])
        seeds = np.concatenate(parts_sd + [lseeds])
        query, ref = np.concatenate([gq, lq]), np.concatenate([gr, lr])
        regs, count = eng.extend_chains(chains, seeds, query, ref, w, clip, clip, 2)
        st = eng.stats()
    assert st["shards"] > 1
    ng = len(gch)
    reg_first = np.concatenate([[0], np.cumsum(c["reg_n"])])
    for k in range(reps):
        for j in range(ng):
            i = k * ng + j
            got = regs[int(chains[i]["seed_first"]): int(chains[i]["seed_first"]) + int(count[i])]
            gm = np.stack([got[f] for f in lib.ALNREG_FIELDS], axis=1).astype(np.int64).reshape(-1, len(lib.ALNREG_FIELDS))
            assert np.array_equal(gm, c["regs"][reg_first[j]: reg_first[j + 1]]), f"copy {k} chain {j}"
    want = _oracle_chains(oracle, make_params(end_bonus=clip, zdrop_mode=1, **P), ch, seeds, query, ref, w, clip, L)
    _check_chains(lib, chains[reps * ng:], regs, count[reps * ng:], want)

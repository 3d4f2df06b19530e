"""bsw_reg2aln: alignment regions to alignment records -- band inference, the band-doubling loop, CIGAR with soft clips,
NM and MD (tools/bwa/bwamem.c mem_reg2aln, tools/bwa/bwa.c bwa_gen_cigar2).

CPU: oracle/aln_oracle.c on hand-worked regions, on every region of the chain goldens (bwa's own regions, both strands)
against properties a record must satisfy and a plain Python transcription of the NM / MD walk, the loop's exits; the
finishing pass's sweeps (md::md_sweep) emulated with the lanes as coroutines (tests/emu/md_emu.cu) against the oracle.
GPU: the entry point against the oracle on the golden regions, end to end from extend_chains, long reads, a seeded
stress set and the call contract."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from oracle.pyoracle import make_params
from test_chain import _build_batch, load_chain_case, CHAIN_CASES
from test_extend32 import LONG_SCORING, _chain_batch, long_reads, mutate      # noqa: F401  (long_reads: fixture)

class AlnOracle:
    """ctypes access to oracle/aln_oracle.c (mem_reg2aln's alignment part) and the global_oracle.c it calls.  TEST
    INFRASTRUCTURE ONLY: compiled on first use into a temporary directory, never into the tree."""
    _so = None

    def __init__(self):
        if AlnOracle._so is None:
            import os
            import shutil
            import subprocess
            import tempfile
            from pathlib import Path
            root = Path(__file__).resolve().parent.parent / "oracle"
            out = Path(tempfile.mkdtemp(prefix="aln_oracle_")) / "libaln_oracle.so"
            cc = shutil.which("gcc") or shutil.which("cc") or "cc"
            subprocess.run([cc, "-O2", "-fPIC", "-shared", "-fopenmp", "-std=c11", "-Wall", "-o", str(out),
                            str(root / "global_oracle.c"), str(root / "aln_oracle.c")], check=True)
            AlnOracle._so = C.CDLL(str(out))
            AlnOracle._threads = os.cpu_count() or 1
        self.lib = AlnOracle._so

    def max_threads(self) -> int:
        return AlnOracle._threads

    def global_align(self, params, query: np.ndarray, target: np.ndarray, w: int):
        """ksw_global2 (global_oracle.c) -> (score, cigar uint32[n])"""
        query = np.ascontiguousarray(query); target = np.ascontiguousarray(target)
        cig = np.zeros(len(query) + len(target) + 1, dtype=np.uint32)
        n = C.c_int(0)
        fn = self.lib.bsw_oracle_global
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        score = fn(C.byref(params), query.ctypes.data, len(query), target.ctypes.data, len(target), w, cig.ctypes.data,
                   C.byref(n))
        return int(score), cig[:n.value].copy()

    def reg2aln(self, params, regs_in: np.ndarray, query: np.ndarray, ref: np.ndarray, l_pac: int, w: int,
                nthreads: int = 0):
        """mem_reg2aln's alignment part for bsw_reg_in records (72 bytes, REG_IN_DTYPE) -> dict(pos int64[n],
        rec int32[n, 5] = is_rev n_cigar NM gscore w, cigar list of uint32 arrays, md list of bytes, info int32[n, 3] =
        tries, exit (1 score == last, 2 w2 == w << 2, 3 three tries, 4 score >= truesc - a), fast path).  Raises
        ValueError for a region bwa_gen_cigar2 rejects."""
        regs_in = np.ascontiguousarray(regs_in)
        assert regs_in.dtype.itemsize == 72
        n = len(regs_in)
        r = regs_in["reg"]
        mapped = (r["rb"] >= 0) & (r["re"] >= 0)
        ql = np.where(mapped, r["qe"].astype(np.int64) - r["qb"], 0)
        rl = np.where(mapped, r["re"] - r["rb"], 0)
        croom = np.concatenate([[0], np.cumsum(ql + rl + 2)]).astype(np.int64)
        mroom = np.concatenate([[0], np.cumsum(4 * ql + rl + 2)]).astype(np.int64)
        pos = np.zeros(max(n, 1), np.int64); rec = np.zeros((max(n, 1), 5), np.int32)
        info = np.zeros((max(n, 1), 3), np.int32); lmd = np.zeros(max(n, 1), np.int32)
        cig = np.zeros(int(croom[-1]) + 1, np.uint32); md = np.zeros(int(mroom[-1]) + 1, np.uint8)
        query = np.ascontiguousarray(query); ref = np.ascontiguousarray(ref)
        fn = self.lib.bsw_oracle_reg2aln_batch
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p] + \
            [C.c_void_p] * 8 + [C.c_int]
        rc = fn(C.byref(params), w, C.c_int64(l_pac), regs_in.ctypes.data, n, query.ctypes.data, ref.ctypes.data,
                pos.ctypes.data, rec.ctypes.data, cig.ctypes.data, croom.ctypes.data, md.ctypes.data, mroom.ctypes.data,
                lmd.ctypes.data, info.ctypes.data, nthreads if nthreads > 0 else self.max_threads())
        if rc:
            raise ValueError("a region bwa_gen_cigar2 rejects (strand-bridging, empty)")
        return dict(pos=pos[:n], rec=rec[:n], info=info[:n],
                    cigar=[cig[croom[k]: croom[k] + rec[k, 1]].copy() for k in range(n)],
                    md=[md[mroom[k]: mroom[k] + lmd[k]].tobytes() for k in range(n)])


@pytest.fixture(scope="module")
def aln():
    return AlnOracle()


ENC = {c: i for i, c in enumerate("ACGTN")}
DEFAULT = dict(match=1, mismatch=4, o_del=6, e_del=1, o_ins=6, e_ins=1, ambig=-1)
ASYM = dict(match=1, mismatch=4, o_del=6, e_del=1, o_ins=5, e_ins=2, ambig=-1)


def s2c(s: str) -> np.ndarray:
    return np.array([ENC[c] for c in s], np.uint8)


def revcomp(a: np.ndarray) -> np.ndarray:
    return np.where(a < 4, 3 - a, 4).astype(np.uint8)[::-1].copy()


def oparams(P: dict):
    return make_params(**{k: P[k] for k in ("match", "mismatch", "o_del", "e_del", "o_ins", "e_ins")}, ambig=P.get("ambig", -1))


def one_region(G, read, rb, re, qb, qe, truesc, reg_w=100):
    """-> (regs_in[1], read, D, l_pac) for one region over genome G (strings or codes), D = G + revcomp(G)"""
    import genomicsbench_b200 as gb
    G = s2c(G) if isinstance(G, str) else G
    read = s2c(read) if isinstance(read, str) else read
    D = np.concatenate([G, revcomp(G)])
    r = np.zeros(1, gb.REG_IN_DTYPE)
    g = r["reg"]
    g["rb"], g["re"], g["qb"], g["qe"], g["truesc"], g["w"] = rb, re, qb, qe, truesc, reg_w
    r["ref_off"], r["l_query"] = max(rb, 0), len(read)
    return r, read, D, len(G)


def oracle_one(aln, P, *a, w=100):
    import genomicsbench_b200 as gb
    regs, read, D, L = one_region(*a)
    o = aln.reg2aln(oparams(P), regs, read, D, L, w)
    return dict(pos=int(o["pos"][0]), is_rev=int(o["rec"][0, 0]), NM=int(o["rec"][0, 2]), gscore=int(o["rec"][0, 3]),
                cigar=gb.cigar_string(o["cigar"][0]), md=o["md"][0].decode(), info=tuple(int(v) for v in o["info"][0]))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: hand-worked records
# ---------------------------------------------------------------------------------------------------------------------
R20 = "GGTTCAGTACTTGCAGGTTC"


def test_hand_worked_records(aln):
    P = DEFAULT
    o = oracle_one(aln, P, "ACTT", "ACGT", 0, 4, 0, 4, 2)                # forward: the reference base of the mismatch
    assert (o["cigar"], o["md"], o["NM"], o["pos"], o["is_rev"]) == ("4M", "2T1", 1, 0, 0)
    assert o["info"][2] == 1 and o["gscore"] == -1                          # fast path: 1 + 1 - 4 + 1, no DP
    o = oracle_one(aln, P, "AAGT", "ACGT", 4, 8, 0, 4, 2)                # D[4:8] = ACTT on the reverse strand
    assert (o["cigar"], o["md"], o["NM"], o["pos"], o["is_rev"]) == ("4M", "1A2", 1, 0, 1)     # "TGCAN": T -> A
    o = oracle_one(aln, P, R20, R20[:8] + R20[10:], 0, 20, 0, 18, 10)    # an internal deletion
    assert (o["cigar"], o["md"], o["NM"]) == ("8M2D10M", "8^AC10", 2)
    ri = R20[:8] + "GG" + R20[8:]
    ri = ri[:17] + "A" + ri[18:]                                             # and a mismatch 7 bases after the insertion
    o = oracle_one(aln, P, R20, ri, 0, 20, 0, 22, 10)
    assert (o["cigar"], o["md"], o["NM"]) == ("8M2I12M", "15G4", 3)         # the insertion does not reset the run
    o = oracle_one(aln, P, "TT" + R20, R20, 0, 22, 0, 20, 12)            # a leading D: pos moves, not in MD / NM
    assert (o["cigar"], o["md"], o["NM"], o["pos"]) == ("20M", "20", 0, 2)
    o = oracle_one(aln, P, "TT" + R20 + "AA", R20, 0, 24, 0, 20, 12)     # both ends D: only the leading one goes
    assert (o["cigar"], o["md"], o["NM"], o["pos"]) == ("20M2D", "20", 0, 2)
    read = "AC" + R20 + "GTA"
    o = oracle_one(aln, P, R20, read, 0, 20, 2, 22, 20)
    assert o["cigar"] == "2S20M3S"
    o = oracle_one(aln, P, "".join("TGCA"["ACGT".index(c)] for c in R20[::-1]), read, 20, 40, 2, 22, 20)
    assert (o["cigar"], o["is_rev"]) == ("3S20M2S", 1)                       # clips swap on the reverse strand
    rn = R20[:5] + "N" + R20[6:]
    o = oracle_one(aln, P, rn, rn, 0, 20, 0, 20, 18)                      # N against N: an MD match
    assert (o["cigar"], o["md"], o["NM"], o["gscore"]) == ("20M", "20", 0, 18)
    o = oracle_one(aln, P, R20, R20, -1, -1, 0, 20, 18)                   # the unmapped record
    assert (o["pos"], o["cigar"], o["md"], o["NM"]) == (-1, "", "", 0)


def test_reverse_strand_homopolymer_deletion_is_leftmost(aln):
    """One A fewer in the run AAAAA of the forward genome, read on the reverse strand: the deletion sits at the run's
    first base in forward coordinates (bwa_gen_cigar2 reverses both sequences; without that it lands at the last)."""
    F = "GCATGCCGTAAAAAGCTTGACG"
    fd = F[:9] + F[10:]
    read = "".join("TGCA"["ACGT".index(c)] for c in fd[::-1])
    L = len(F)
    o = oracle_one(aln, DEFAULT, F, read, L, 2 * L, 0, len(read), len(read) - 8)
    assert (o["cigar"], o["md"], o["NM"], o["is_rev"], o["pos"]) == ("9M1D12M", "9^A12", 1, 1, 0)


# ---------------------------------------------------------------------------------------------------------------------
# the golden chain regions and properties every record satisfies
# ---------------------------------------------------------------------------------------------------------------------
def golden_regions(name):
    """-> (P, regs_in, query, D, l_pac, w) for every region of tests/golden/chain/<name>.npz (bwa's own regions)"""
    import genomicsbench_b200 as gb
    c = load_chain_case(name)
    ch = np.repeat(np.arange(len(c["reg_n"])), c["reg_n"])
    regs = np.zeros(len(ch), gb.REG_IN_DTYPE)
    for k, f in enumerate(("rb", "re", "qb", "qe", "score", "truesc", "w", "seedcov", "seedlen0")):
        regs["reg"][f] = c["regs"][:, k]
    regs["query_off"] = c["query_off"][ch]
    regs["l_query"] = c["l_query"][ch]
    regs["ref_off"] = regs["reg"]["rb"]
    P = dict(c["P"], ambig=-1)
    P.pop("zdrop")
    return P, regs, np.ascontiguousarray(c["query"]), c["D"], c["l_pac"], c["w"]


def oriented(regs, k, query, D, l_pac):
    g = regs["reg"][k]
    qo, lq = int(regs["query_off"][k]), int(regs["l_query"][k])
    q = query[qo + int(g["qb"]): qo + int(g["qe"])]
    r = D[int(g["rb"]): int(g["re"])]
    rev = int(g["rb"]) >= l_pac
    return (q[::-1].copy(), r[::-1].copy(), 1) if rev else (q.copy(), r.copy(), 0)


def core_and_presqueeze(ops, pos, rb, re, l_pac, rev, rlen):
    """The record's operations without the clips, and the operation list before the squeeze (the leading D from pos,
    the trailing one from the reference span)"""
    core = [int(c) for c in ops if (int(c) & 0xf) != 3]
    base = 2 * l_pac - 1 - (re - 1) if rev else rb
    lead = pos - base
    used = sum(int(c) >> 4 for c in core if (int(c) & 0xf) in (0, 2))
    pre = ([lead << 4 | 2] if lead else []) + core
    trail = rlen - lead - used
    if trail:
        pre = pre + [trail << 4 | 2]
    return core, pre, lead


def md_walk(q, r, ops, rev):
    """bwa_gen_cigar2's NM / MD walk (bwa.c), transcribed plainly -> (md bytes, NM)"""
    i2b = "TGCAN" if rev else "ACGTN"
    out, x, y, u, nmm, ngap = [], 0, 0, 0, 0, 0
    for k, c in enumerate(ops):
        op, ln = c & 0xf, c >> 4
        if op == 0:
            for i in range(ln):
                if q[x + i] != r[y + i]:
                    out.append(f"{u}{i2b[min(int(r[y + i]), 4)]}"); nmm += 1; u = 0
                else:
                    u += 1
            x += ln; y += ln
        elif op == 2:
            if 0 < k < len(ops) - 1:
                out.append(f"{u}^" + "".join(i2b[min(int(b), 4)] for b in r[y: y + ln])); u = 0; ngap += ln
            y += ln
        elif op == 1:
            x += ln; ngap += ln
    out.append(str(u))
    return "".join(out).encode(), nmm + ngap


def dp_band(P, lq, rlen, w_):
    half = ((lq + 1) >> 1) * P["match"]
    mg = max(int((half - P["o_ins"]) / P["e_ins"] + 1.), int((half - P["o_del"]) / P["e_del"] + 1.), 1)
    return max(min((mg + abs(rlen - lq) + 1) >> 1, w_), abs(rlen - lq) + 3)


def check_record_properties(aln, P, regs, query, D, l_pac, o, sample=None):
    for k in (range(len(regs)) if sample is None else sample):
        g = regs["reg"][k]
        rb, re = int(g["rb"]), int(g["re"])
        if rb < 0 or re < 0:
            assert o["pos"][k] == -1 and len(o["cigar"][k]) == 0 and o["md"][k] == b""
            continue
        q, r, rev = oriented(regs, k, query, D, l_pac)
        ops = o["cigar"][k]
        core, pre, lead = core_and_presqueeze(ops, int(o["pos"][k]), rb, re, l_pac, rev, len(r))
        # the query span with the clips is the read
        assert sum(int(c) >> 4 for c in ops if (int(c) & 0xf) in (0, 1, 3)) == int(regs["l_query"][k])
        # the MD expanded against the operations and the query rebuilds the reference
        md = o["md"][k].decode()
        i2b = "TGCAN" if rev else "ACGTN"
        toks, j = [], 0
        while j < len(md):
            if md[j].isdigit():
                e = j
                while e < len(md) and md[e].isdigit():
                    e += 1
                toks.append(int(md[j:e])); j = e
            elif md[j] == "^":
                e = j + 1
                while e < len(md) and not md[e].isdigit():
                    e += 1
                toks.append(("^", md[j + 1:e])); j = e
            else:
                toks.append(("x", md[j])); j += 1
        built, x, ti, left = [], 0, 0, 0
        for kk, c in enumerate(core):
            op, ln = c & 0xf, c >> 4
            if op == 0:
                for i in range(ln):
                    while left == 0 and ti < len(toks) and isinstance(toks[ti], int):
                        left = toks[ti]; ti += 1
                    if left > 0:
                        built.append(int(q[x + i])); left -= 1
                    else:
                        assert toks[ti][0] == "x", (k, md)
                        built.append(i2b.index(toks[ti][1])); ti += 1
                x += ln
            elif op == 1:
                x += ln
            elif op == 2:
                if kk == len(core) - 1:                  # a D left at the end (both ends were D): not in MD
                    built.extend(int(b) for b in r[lead + len(built): lead + len(built) + ln])      # trailing D kept, not in MD
                    continue
                while ti < len(toks) and toks[ti] == 0:
                    ti += 1
                assert toks[ti][0] == "^", (k, md)
                built.extend(i2b.index(ch) for ch in toks[ti][1]); ti += 1
        assert np.array_equal(np.array(built, np.uint8), r[lead: lead + len(built)]), k
        # the plain transcription of the walk: MD byte for byte, and NM
        want_md, want_nm = md_walk(q, r, pre, rev)
        assert o["md"][k] == want_md, (k, o["md"][k], want_md)
        assert o["rec"][k, 2] == want_nm
        # gscore: global_oracle on the same inputs and band
        wl = int(o["rec"][k, 4])
        if o["info"][k, 2]:
            sc = sum(P["ambig"] if a >= 4 or b >= 4 else (P["match"] if a == b else -P["mismatch"]) for a, b in zip(q, r))
        else:
            sc, _ = aln.global_align(oparams(P), q, r, dp_band(P, len(q), len(r), wl))
        assert o["rec"][k, 3] == sc, k


@pytest.mark.parametrize("case", CHAIN_CASES)
def test_oracle_records_on_golden_regions(aln, case):
    P, regs, query, D, l_pac, w = golden_regions(case)
    o = aln.reg2aln(oparams(P), regs, query, D, l_pac, w)
    assert len(regs) > 100 and (regs["reg"]["rb"] >= l_pac).any() and (regs["reg"]["rb"] < l_pac).any()
    check_record_properties(aln, P, regs, query, D, l_pac, o)


def loop_cases(seed=5, n=400, L=200):
    """Regions built to drive every exit of the band-doubling loop: paired opposite indels that a narrow band cannot
    reach, local scores (truesc) from far below to far above the global score, opt w from 1 to 100, equal-length
    regions on the fast path.  -> (regs_in, query, D, l_pac, ws)"""
    import genomicsbench_b200 as gb
    rng = np.random.default_rng(seed)
    G = rng.integers(0, 4, 200000).astype(np.uint8)
    D = np.concatenate([G, revcomp(G)])
    l_pac = len(G)
    regs = np.zeros(n, gb.REG_IN_DTYPE)
    reads, qo = [], 0
    for k in range(n):
        rb = int(rng.integers(0, 2 * l_pac - 2 * L))
        if rb < l_pac < rb + 2 * L:
            rb = l_pac
        r = D[rb: rb + L]
        kind = k % 4
        if kind == 0:                                            # exact copy, equal lengths
            q = r.copy(); q[rng.integers(0, L, 3)] = rng.integers(0, 4, 3)
        elif kind == 1:                                          # a deletion and an insertion far apart
            a, b, g = int(rng.integers(20, 80)), int(rng.integers(120, 180)), int(rng.integers(5, 40))
            q = np.concatenate([r[:a], r[a + g: b], rng.integers(0, 4, g).astype(np.uint8), r[b:]])
        else:
            q = mutate(rng, r, 0.05)
        lq = len(q)
        regs["reg"][k]["rb"], regs["reg"][k]["re"] = rb, rb + L
        regs["reg"][k]["qb"], regs["reg"][k]["qe"] = 0, lq
        regs["reg"][k]["truesc"] = int(rng.integers(min(lq, L) - 80, min(lq, L) + 40))
        regs["reg"][k]["w"] = int(rng.integers(1, 200))
        regs["query_off"][k], regs["l_query"][k], regs["ref_off"][k] = qo, lq, rb
        reads.append(q); qo += lq
    ws = np.array([1, 2, 5, 16, 100])[np.arange(n) % 5]
    return regs, np.concatenate(reads + [np.zeros(64, np.uint8)]), D, l_pac, ws


def test_loop_exits_all_hit(aln):
    """Across the golden regions and the loop cases every exit is taken: one, two and three tries, score == last_sc,
    w2 == w << 2, the fast path."""
    seen_tries, seen_exit, fast = set(), set(), 0
    for case in CHAIN_CASES:
        P, regs, query, D, l_pac, w = golden_regions(case)
        o = aln.reg2aln(oparams(P), regs, query, D, l_pac, w)
        seen_tries |= set(o["info"][:, 0].tolist()); seen_exit |= set(o["info"][:, 1].tolist()); fast += int(o["info"][:, 2].sum())
    regs, query, D, l_pac, ws = loop_cases()
    for wv in np.unique(ws):
        sel = np.flatnonzero(ws == wv)
        o = aln.reg2aln(oparams(DEFAULT), regs[sel], query, D, l_pac, int(wv))
        seen_tries |= set(o["info"][:, 0].tolist()); seen_exit |= set(o["info"][:, 1].tolist()); fast += int(o["info"][:, 2].sum())
        check_record_properties(aln, DEFAULT, regs[sel], query, D, l_pac, o, sample=range(0, len(sel), 7))
    assert {1, 2, 3} <= seen_tries
    assert {1, 2, 3, 4} <= seen_exit
    assert fast > 0


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the finishing pass's sweeps, emulated
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def md_emu(lib, tmp_path_factory):
    """tests/emu/md_emu.cu compiled as host code (nvcc) into a temporary directory."""
    import os
    import subprocess
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    out = tmp_path_factory.mktemp("md_emu") / "libmd_emu.so"
    env = dict(os.environ)
    env["PATH"] = "/usr/bin:" + env.get("PATH", "")
    subprocess.run([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc"), "-std=c++17", "-O2", "-gencode",
                    "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC,-pthread", "-I", str(root / "include"),
                    "-o", str(out), str(root / "tests" / "emu" / "md_emu.cu"), "-lpthread"], check=True, env=env)
    so = C.CDLL(str(out))
    so.md_emu_batch.restype = C.c_int
    so.md_emu_batch.argtypes = [C.c_void_p, C.c_longlong] + [C.c_void_p] * 13
    return so


def run_md_emu(so, P, items):
    """items = [(q, r, pre-squeeze ops, rev)] -> (md list, nm, msc)"""
    n = len(items)
    cat = lambda xs, dt: np.concatenate([np.asarray(x, dt) for x in xs] + [np.zeros(64, dt)])  # noqa: E731
    offs = lambda xs: np.concatenate([[0], np.cumsum([len(x) for x in xs])]).astype(np.int64)  # noqa: E731
    qs, rs, cs = [it[0] for it in items], [it[1] for it in items], [it[2] for it in items]
    room = np.concatenate([[0], np.cumsum([4 * len(q) + len(r) + 1 for q, r in zip(qs, rs)])]).astype(np.int64)
    md = np.full(int(room[-1]) + 1, ord("#"), np.uint8)
    mdl, nm, msc = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32)
    ncig = np.array([len(c) for c in cs], np.int32)
    rev = np.array([it[3] for it in items], np.int32)
    sc = np.array([P["match"], P["mismatch"], P["ambig"]], np.int32)
    Q, Rr, Cc = cat(qs, np.uint8), cat(rs, np.uint8), cat(cs, np.uint32)
    qo, ro, co = offs(qs), offs(rs), offs(cs)
    rc = so.md_emu_batch(sc.ctypes.data, n, Q.ctypes.data, qo.ctypes.data, Rr.ctypes.data, ro.ctypes.data,
                         Cc.ctypes.data, co.ctypes.data, ncig.ctypes.data, rev.ctypes.data, md.ctypes.data,
                         room.ctypes.data, mdl.ctypes.data, nm.ctypes.data, msc.ctypes.data)
    assert rc == 0, "the lanes of a warp disagreed"
    for k in range(n):                                   # nothing written past the MD, nothing left unwritten
        assert md[room[k] + mdl[k]] == ord("#") and ord("#") not in md[room[k]: room[k] + mdl[k]].tolist()
    return [md[room[k]: room[k] + mdl[k]].tobytes() for k in range(n)], nm, msc


@pytest.mark.parametrize("case", CHAIN_CASES)
def test_md_emulated_matches_oracle_golden(md_emu, aln, case):
    P, regs, query, D, l_pac, w = golden_regions(case)
    o = aln.reg2aln(oparams(P), regs, query, D, l_pac, w)
    items, want = [], []
    for k in range(len(regs)):
        q, r, rev = oriented(regs, k, query, D, l_pac)
        g = regs["reg"][k]
        _, pre, _ = core_and_presqueeze(o["cigar"][k], int(o["pos"][k]), int(g["rb"]), int(g["re"]), l_pac, rev, len(r))
        items.append((q, r, pre, rev)); want.append(k)
    md, nm, msc = run_md_emu(md_emu, P, items)
    assert md == o["md"]
    assert np.array_equal(nm, o["rec"][:, 2])
    fast = o["info"][:, 2] == 1
    assert np.array_equal(msc[fast], o["rec"][fast, 3])


def synthetic_long(seed):
    """Long synthetic regions with their pre-squeeze operations: 100 kb with N runs, every base mismatched, alternating
    short indels near the MD bound."""
    rng = np.random.default_rng(seed)
    items = []
    r = rng.integers(0, 4, 100000).astype(np.uint8)
    q = r.copy()
    for _ in range(20):
        a = int(rng.integers(0, 99000)); ln = int(rng.integers(5, 300))
        q[a: a + ln] = 4
        r[a + ln // 3: a + ln] = 4
    q[rng.random(len(q)) < 0.03] = rng.integers(0, 4)
    items.append((q, r, [len(q) << 4], 0))
    r = rng.integers(0, 4, 5000).astype(np.uint8)
    items.append(((r + 1) % 4, r, [len(r) << 4], 1))                       # every base mismatched
    # alternating 1-base deletions and mismatches: "0^X0Y" per unit, 5 MD bytes per query base
    n = 3000
    r = rng.integers(0, 4, 2 * n + 2).astype(np.uint8)
    q = ((r[1:2 * n + 1:2] + 1) % 4).astype(np.uint8)
    ops = [1 << 4]
    qq = [int(r[0])]
    for i in range(n):
        ops += [1 << 4 | 2, 1 << 4]
        qq.append(int(q[i]))
    items.append((np.array(qq, np.uint8), r[: 2 * n + 1], ops, 0))
    # alternating 1-base insertions and deletions
    r = rng.integers(0, 4, 4001).astype(np.uint8)
    q = rng.integers(0, 4, 4001).astype(np.uint8)
    ops = [1 << 4] + [1 << 4 | 1, 1 << 4 | 2] * 2000 + [1 << 4]
    items.append((np.concatenate([q[:1], q[1:2001], q[2001:2002]]), np.concatenate([r[:1], r[1:2001], r[2001:2002]]), ops, 1))
    return items


def test_md_emulated_long_synthetic(md_emu):
    P = dict(DEFAULT)
    items = synthetic_long(9)
    md, nm, msc = run_md_emu(md_emu, P, items)
    for (q, r, ops, rev), m, n_ in zip(items, md, nm):
        want, wnm = md_walk(q, r, ops, rev)
        assert m == want and n_ == wnm
        assert len(m) <= 4 * len(q) + len(r) + 1                             # the documented MD bound
    assert len(md[2]) >= 4 * len(items[2][0]) - 10                           # close to it
    sc = lambda q, r: sum(P["ambig"] if a >= 4 or b >= 4 else (1 if a == b else -4) for a, b in zip(q.tolist(), r.tolist()))  # noqa: E731
    assert msc[0] == sc(items[0][0], items[0][1]) and msc[1] == -4 * len(items[1][0])


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the ABI
# ---------------------------------------------------------------------------------------------------------------------
def test_header_layout_matches_mirrors(lib, tmp_path):
    import shutil
    import subprocess
    from pathlib import Path
    cc = shutil.which("gcc") or shutil.which("cc")
    if not cc:
        pytest.skip("no C compiler")
    root = Path(__file__).resolve().parent.parent
    src = tmp_path / "layout.c"
    src.write_text('''
#include <stdio.h>
#include <stddef.h>
#include "bsw.h"
#define S(T) printf(#T " %zu\\n", sizeof(T))
#define O(T, F) printf(#T "." #F " %zu\\n", offsetof(T, F))
int main(void) {
    S(bsw_reg_in); O(bsw_reg_in, reg); O(bsw_reg_in, query_off); O(bsw_reg_in, ref_off); O(bsw_reg_in, l_query);
    S(bsw_aln); O(bsw_aln, pos); O(bsw_aln, is_rev); O(bsw_aln, n_cigar); O(bsw_aln, NM); O(bsw_aln, gscore); O(bsw_aln, w);
    return 0;
}
''')
    exe = tmp_path / "layout"
    subprocess.run([cc, "-std=c99", "-Wall", "-Werror", "-I", str(root / "include"), str(src), "-o", str(exe)], check=True)
    got = {k: int(v) for k, v in (line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True,
                                                                          text=True).stdout.splitlines())}
    for name, dt in (("bsw_reg_in", lib.REG_IN_DTYPE), ("bsw_aln", lib.ALN_DTYPE)):
        assert got[name] == dt.itemsize
        for f in dt.names:
            if f != "reserved":
                assert got[f"{name}.{f}"] == dt.fields[f][1], (name, f)
    assert got["bsw_reg_in"] == 72 and got["bsw_aln"] == 32                  # no padding holes


def test_product_does_not_name_aln_oracle():
    from pathlib import Path
    pkg = Path(__file__).resolve().parent.parent / "genomicsbench_b200"
    for p in [q for q in pkg.rglob("*") if q.suffix in (".py", ".cu", ".cpp", ".h", ".cuh", ".inl")]:
        assert "aln_oracle" not in p.read_text(), p


def test_cigar_string_and_capacity(lib):
    assert lib.cigar_string(np.array([2 << 4 | 3, 20 << 4, 1 << 4 | 1, 3 << 4 | 2], np.uint32)) == "2S20M1I3D"
    regs = np.zeros(3, lib.REG_IN_DTYPE)
    regs["reg"]["rb"], regs["reg"]["re"], regs["reg"]["qb"], regs["reg"]["qe"] = [0, -1, 10], [30, -1, 15], [0, 0, 2], [25, 0, 9]
    assert lib.reg2aln_capacity(regs) == (25 + 30 + 2 + 7 + 5 + 2, 4 * 25 + 30 + 1 + 4 * 7 + 5 + 1)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: the entry point against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def assert_equal_oracle(got, want, idx=None):
    aln, cigar, coff, md, moff = got
    idx = range(len(aln)) if idx is None else idx
    for k in idx:
        assert aln["pos"][k] == want["pos"][k], k
        rec = (aln["is_rev"][k], aln["n_cigar"][k], aln["NM"][k], aln["gscore"][k], aln["w"][k])
        assert rec == tuple(want["rec"][k]), (k, rec, tuple(want["rec"][k]))
        assert np.array_equal(cigar[coff[k]: coff[k + 1]], want["cigar"][k]), k
        assert md[moff[k]: moff[k + 1]].tobytes() == want["md"][k], k


@pytest.mark.gpu
@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("case", CHAIN_CASES)
def test_reg2aln_golden_regions(lib, aln, case, pinned):
    P, regs, query, D, l_pac, w = golden_regions(case)
    want = aln.reg2aln(oparams(P), regs, query, D, l_pac, w)
    if pinned:
        regs, query, D = lib.pinned_copy(regs), lib.pinned_copy(query), lib.pinned_copy(D)
    with lib.Engine(**P) as eng:
        got = eng.reg2aln(regs, query, D, l_pac, w)
        st = eng.stats()
    assert_equal_oracle(got, want)
    assert st["pairs"] == len(regs) and st["kernel_launches"] > 3 and st["ms_sort"] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", CHAIN_CASES)
def test_reg2aln_end_to_end_from_extend_chains(lib, aln, case):
    c = load_chain_case(case)
    P = dict(c["P"], ambig=-1)
    with lib.Engine(end_bonus=c["clip5"], zdrop_mode=lib.BSW_ZDROP_SCALAR, **c["P"]) as eng:
        chains, seeds, query, ref = _build_batch(lib, eng, c)
        regs, count = eng.extend_chains(chains, seeds, query, ref, c["w"], c["clip5"], c["clip3"], 2)
        rin = lib.reg_inputs(chains, regs, count)
        got = eng.reg2aln(rin, query, ref, c["l_pac"], c["w"])
    P.pop("zdrop")
    assert_equal_oracle(got, aln.reg2aln(oparams(P), rin, query, ref, c["l_pac"], c["w"]))


@pytest.mark.gpu
def test_reg2aln_long_reads(lib, aln, long_reads):
    L, D, reads = long_reads
    w = 100
    P = dict(LONG_SCORING, ambig=-1)
    P.pop("zdrop")
    with lib.Engine(end_bonus=0, zdrop_mode=lib.BSW_ZDROP_SCALAR, **LONG_SCORING) as eng:
        chains, seeds, query, ref = _chain_batch(lib, eng, reads, D, L, w, 1)
        regs, count = eng.extend_chains(chains, seeds, query, ref, w, 0, 0, 2)
        rin = lib.reg_inputs(chains, regs, count)
        got = eng.reg2aln(rin, query, ref, L, w)
        st = eng.stats()
    want = aln.reg2aln(oparams(P), rin, query, ref, L, w)
    assert_equal_oracle(got, want)
    g = rin["reg"]
    assert (np.maximum(g["qe"] - g["qb"], g["re"] - g["rb"]) > 32767).any() and st["n_long"] > 0
    assert (want["info"][:, 0] >= 2).any()


@pytest.mark.gpu
@pytest.mark.parametrize("scoring", ["default", "asym", "long"])
def test_reg2aln_stress(lib, aln, scoring):
    """About 200 000 seeded short regions (the loop cases tiled with fresh seeds): both strands, N runs, equal-length
    regions on the fast path, opt w from 1 to 100; several finishing-pass chunks."""
    P = {"default": DEFAULT, "asym": ASYM, "long": dict(LONG_SCORING, ambig=-1)}[scoring]
    P = {k: P[k] for k in ("match", "mismatch", "o_del", "e_del", "o_ins", "e_ins", "ambig")}
    regs, query, D, l_pac, _ = loop_cases(seed=77, n=70000 if scoring == "default" else 20000)
    rng = np.random.default_rng(78)
    q = query.copy()
    for _ in range(2000):
        a = int(rng.integers(0, len(q) - 64)); q[a: a + int(rng.integers(3, 40))] = 4
    for w in (1, 100):
        want = aln.reg2aln(oparams(P), regs, q, D, l_pac, w)
        with lib.Engine(**P) as eng:
            got = eng.reg2aln(regs, q, D, l_pac, w)
        assert_equal_oracle(got, want)
        assert want["info"][:, 2].sum() > 0


@pytest.mark.gpu
def test_reg2aln_contract(lib, aln):
    P, regs, query, D, l_pac, w = golden_regions("chain_default")
    want = aln.reg2aln(oparams(P), regs, query, D, l_pac, w)
    n = len(regs)
    with lib.Engine(**P) as eng:
        full = eng.reg2aln(regs, query, D, l_pac, w)
        ncig, nmd = int(full[2][n]), int(full[4][n])
        for cap_c, cap_m in ((ncig - 1, nmd), (ncig, nmd - 1)):              # one short of need: -1
            out = (np.zeros(n, lib.ALN_DTYPE), np.zeros(cap_c, np.uint32), np.zeros(n + 1, np.int64),
                   np.zeros(cap_m, np.uint8), np.zeros(n + 1, np.int64))
            with pytest.raises(lib.BswError) as ei:
                eng.reg2aln(regs, query, D, l_pac, w, out=out)
            assert ei.value.code == -1
            assert_equal_oracle(eng.reg2aln(regs, query, D, l_pac, w), want)   # the next call is complete
        out = (np.zeros(n, lib.ALN_DTYPE), np.zeros(ncig, np.uint32), np.zeros(n + 1, np.int64), np.zeros(nmd, np.uint8),
               np.zeros(n + 1, np.int64))
        assert_equal_oracle(eng.reg2aln(regs, query, D, l_pac, w, out=out), want)
        # n = 0
        a0, c0, o0, m0, mo0 = eng.reg2aln(regs[:0], query, D, l_pac, w)
        assert len(a0) == 0 and len(c0) == 0 and list(o0) == [0] and list(mo0) == [0]
        # unmapped regions mixed with mapped ones
        mix = regs.copy()
        mix["reg"]["rb"][::3] = -1
        mix["reg"]["re"][::3] = -1
        assert_equal_oracle(eng.reg2aln(mix, query, D, l_pac, w), aln.reg2aln(oparams(P), mix, query, D, l_pac, w))
        # the domain, nothing written
        k = int(np.flatnonzero(regs["reg"]["rb"] < l_pac)[0])
        cases = []
        for f, v in (("re", l_pac + 5), ("qb", -1), ("qe", 10 ** 6)):          # strand-bridging, qb < 0, qe > l_query
            b = regs.copy(); b["reg"][f][k] = v
            if f == "re":
                b["reg"]["rb"][k] = l_pac - 5
            cases.append((b, w))
        b = regs.copy(); b["reg"]["qe"][k] = b["reg"]["qb"][k]; cases.append((b, w))            # qb >= qe
        b = regs.copy(); b["reg"]["re"][k] = 2 * l_pac + 1; b["reg"]["rb"][k] = l_pac; cases.append((b, w))   # re > 2 l_pac
        b = regs.copy(); b["l_query"][k] = 1 << 24; b["reg"]["qe"][k] = (1 << 24); cases.append((b, w))      # length
        cases.append((regs, -1))                                                                  # w < 0
        for b, wv in cases:
            out = (np.full(n, 7, lib.ALN_DTYPE), np.full(ncig, 7, np.uint32), np.full(n + 1, 7, np.int64),
                   np.full(nmd, 7, np.uint8), np.full(n + 1, 7, np.int64))
            with pytest.raises(lib.BswError) as ei:
                eng.reg2aln(b, query, D, l_pac, wv, out=out)
            assert ei.value.code == -2
            assert (out[1] == 7).all() and (out[3] == 7).all() and (out[0]["pos"] == 7).all() and (out[2][1:] == 7).all()

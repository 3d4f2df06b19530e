#!/usr/bin/env python
"""Throughput of bsw_reg2aln (alignment regions -> CIGAR, NM, MD: mem_reg2aln + bwa_gen_cigar2).
Prints one JSON line (and writes it to OUT when given):
  short        N seeded regions of 151-bp and 250-bp reads on a 20 Mb synthetic genome, both strands (substitutions,
               short indels, a few N): call time, regions/s, DP kernel ms against finishing-pass ms (CUDA events, the
               engine's statistics), the share of regions that took 1, 2 or 3 tries
  long         the long-read regions of tests/test_extend32.py (100 reads of 20-120 kb, pacbio scoring) from
               bsw_extend_chains: the same figures
  oracle       oracle/aln_oracle.c (the project's CPU restatement, NOT bwa's code; compiled into a temporary directory)
               on the short regions: regions/s on one host thread and on all host threads
Every timed result is compared with the oracle inside the run; the card's name and power limit are read in the same run.
Usage: python scripts/reg2aln_bench.py [n_short=500000] [reps=3] [OUT]"""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import genomicsbench_b200 as gb
from oracle.pyoracle import make_params
from test_extend32 import LONG_SCORING, _chain_batch, make_long_reads, mutate
from test_reg2aln import AlnOracle

n_short = int(sys.argv[1]) if len(sys.argv) > 1 else 500000
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
out_path = sys.argv[3] if len(sys.argv) > 3 else None
DEFAULT = dict(match=1, mismatch=4, o_del=6, e_del=1, o_ins=6, e_ins=1, ambig=-1)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:                                 # the numbers still carry the torch device name
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def timed(eng, fn, *args):
    """best wall time of `reps` calls after one warm-up call, the stats of that call, and its results"""
    res = fn(*args)
    best, st = 1e30, None
    for _ in range(reps):
        t0 = time.perf_counter()
        res = fn(*args)
        dt = time.perf_counter() - t0
        if dt < best:
            best, st = dt, eng.stats()
    return best, st, res


def oparams(P):
    return make_params(**{k: P[k] for k in ("match", "mismatch", "o_del", "e_del", "o_ins", "e_ins")}, ambig=-1)


def short_regions(n, seed=2027, L=20_000_000):
    """n regions: a read of 151 or 250 bp taken from either strand of D = G + revcomp(G) and mutated (3 % substitutions,
    short indels, 1 % of reads with a run of N); the region spans the read's origin with 0-3 extra reference bases on each
    side, qb / qe clip 0-5 bases, truesc = the read's length minus 5 per difference."""
    rng = np.random.default_rng(seed)
    G = rng.integers(0, 4, L).astype(np.uint8)
    D = np.concatenate([G, (3 - G[::-1]).astype(np.uint8)])
    lens = np.where(rng.random(n) < 0.5, 151, 250)
    regs = np.zeros(n, gb.REG_IN_DTYPE)
    reads, qo = [], 0
    for k in range(n):
        ln = int(lens[k])
        strand = int(rng.integers(0, 2))
        rb = int(rng.integers(strand * L + 8, strand * L + L - ln - 16))
        src = D[rb: rb + ln + 8]
        q = mutate(rng, src, float(rng.choice([0.0, 0.01, 0.03, 0.06])))[:ln]
        if rng.random() < 0.01:
            a = int(rng.integers(0, ln - 20)); q[a: a + int(rng.integers(3, 20))] = 4
        e0, e1 = int(rng.integers(0, 4)), int(rng.integers(0, 4))
        qb, qe = int(rng.integers(0, 6)), len(q) - int(rng.integers(0, 6))
        g = regs["reg"][k]
        g["rb"], g["re"] = rb - e0, rb + qe + e1
        g["qb"], g["qe"] = qb, qe
        g["truesc"] = qe - qb - 5 * int((q[qb:qe] != src[qb:qe]).sum() // 4)
        g["w"] = 100
        regs["query_off"][k], regs["l_query"][k], regs["ref_off"][k] = qo, len(q), g["rb"]
        reads.append(q); qo += len(q)
    return regs, np.concatenate(reads + [np.zeros(64, np.uint8)]), D, L


def check(got, want):
    aln, cigar, coff, md, moff = got
    assert np.array_equal(aln["pos"], want["pos"])
    rec = np.stack([aln[f] for f in ("is_rev", "n_cigar", "NM", "gscore", "w")], axis=1)
    assert np.array_equal(rec, want["rec"])
    assert np.array_equal(cigar, np.concatenate(want["cigar"] + [np.zeros(0, np.uint32)]))
    assert md.tobytes() == b"".join(want["md"])


def figures(n, t, st, want):
    tries = np.bincount(want["info"][:, 0], minlength=4)[1:4]
    return {"regions": n, "call_s": t, "regions_per_s": n / t, "dp_kernel_ms": st["ms_kernel"] - st["ms_sort"],
            "finishing_pass_ms": st["ms_sort"], "host_pack_ms": st["ms_pack"], "kernel_launches": st["kernel_launches"],
            "dp_short": st["n_short"], "dp_long": st["n_long"],
            "tries_share": {str(k + 1): float(tries[k]) / max(1, int(tries.sum())) for k in range(3)},
            "fast_path_share": float(want["info"][:, 2].mean())}


oracle = AlnOracle()
line = {"bench": "reg2aln", "card": card()}

# ---- short reads -----------------------------------------------------------------------------------------------------
regs, query, D, L = short_regions(n_short)
W = 100
want = oracle.reg2aln(oparams(DEFAULT), regs, query, D, L, W)
with gb.Engine(**DEFAULT) as eng:
    t, st, got = timed(eng, eng.reg2aln, regs, query, D, L, W)
check(got, want)
line["short"] = figures(len(regs), t, st, want)
# the oracle on one host thread (a sample) and on all host threads
sub = regs[: min(len(regs), 50000)]
t0 = time.perf_counter(); oracle.reg2aln(oparams(DEFAULT), sub, query, D, L, W, nthreads=1); t1 = time.perf_counter() - t0
t0 = time.perf_counter(); oracle.reg2aln(oparams(DEFAULT), regs, query, D, L, W); ta = time.perf_counter() - t0
line["oracle_restated"] = {"regions_per_s_1thread": len(sub) / t1, "regions_per_s_all_threads": len(regs) / ta,
                           "threads": oracle.max_threads(), "host_cpus": os.cpu_count(),
                           "note": "oracle/aln_oracle.c + global_oracle.c (the project's restatement), not bwa's code"}

# ---- long reads ------------------------------------------------------------------------------------------------------
crng = np.random.default_rng(2026)
LL = 3_000_000
G = crng.integers(0, 4, size=LL, dtype=np.uint8)
DL = np.concatenate([G, (3 - G[::-1]).astype(np.uint8)])
reads = make_long_reads(crng, DL, LL, 100, 20000, 120000, (0.05, 0.12))
P = {k: LONG_SCORING[k] for k in ("match", "mismatch", "o_del", "e_del", "o_ins", "e_ins")}
with gb.Engine(end_bonus=0, zdrop_mode=gb.BSW_ZDROP_SCALAR, **LONG_SCORING) as eng:
    chains, seeds, lq, lref = _chain_batch(gb, eng, reads, DL, LL, W, 1)
    lregs, count = eng.extend_chains(chains, seeds, lq, lref, W, 0, 0, 2)
    rin = gb.reg_inputs(chains, lregs, count)
    t, st, got = timed(eng, eng.reg2aln, rin, lq, lref, LL, W)
lwant = oracle.reg2aln(oparams(dict(P, ambig=-1)), rin, lq, lref, LL, W)
check(got, lwant)
g = rin["reg"]
line["long"] = dict(figures(len(rin), t, st, lwant), reads=len(reads),
                    longest_region=int(np.maximum(g["qe"] - g["qb"], g["re"] - g["rb"]).max()))

s = json.dumps(line)
print(s)
if out_path:
    with open(out_path, "w") as f:
        f.write(s + "\n")

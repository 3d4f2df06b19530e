#!/usr/bin/env python
"""Long-read throughput of bsw_extend32 (ksw_extend2 in int32, bsw_long32.cuh) and of bsw_extend_chains on long reads.
Prints one JSON line (and writes it to OUT when given):
  extend32        seeded long flanks at w = 100 (N pairs of 5-60 kb, a mutated copy of the query as target, 8 % error):
                  call time, pairs/s, effective GCUPS over the call and over the kernel time (CUDA events)
  in_domain       bsw_extend32 against bsw_extend on the same pairs of the `large` config (inside the 16-bit domain):
                  what the int32 ring kernel costs where the 16-bit kernels apply
  chains          bsw_extend_chains on 100 reads of 20-120 kb (5-12 % error, both strands, a few N) with bwa's pacbio
                  scoring: chains/s and extensions/s
  oracle          oracle/ksw_oracle.c on one host thread on a subset of the flanks: ns per cell.  This is the project's
                  CPU restatement of ksw_extend2, NOT the reference's code.
Results are checked against the oracle on subsets inside the run; the card's name and power limit are read in the
same run.  Usage: python scripts/long_bench.py [n_pairs=20000] [reps=3] [OUT]"""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import genomicsbench_b200 as gb
from oracle.pyoracle import Oracle, make_params
from test_extend32 import LONG_SCORING, _chain_batch, _oracle_chains, long_pairs, make_long_reads

n_pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
out_path = sys.argv[3] if len(sys.argv) > 3 else None
W = 100
FIELDS = gb.RESULT_FIELDS


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as e:                                 # the numbers still carry the torch device name
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unknown ({e})"}


def best_of(fn):
    """best wall time of `reps` calls after one warm-up call (module load, buffers)"""
    fn()
    t_best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        t_best = min(t_best, time.perf_counter() - t0)
    return t_best


oracle = Oracle()
line = {"metric": "long_read_extension", "card": card(), "w": W}

# ---- bsw_extend32 on long flanks --------------------------------------------------------------------------------------
pairs, ref, qer = long_pairs(2026, n_pairs, 5000, 60000, (0, 100))
P = make_params(zdrop_mode=0)
with gb.Engine() as eng:
    work = pairs.copy()
    stats = []

    def run():
        work[:] = pairs
        eng.extend32(work, ref, qer, W)
        stats.append(eng.stats())
    t = best_of(run)
    st = min(stats[1:], key=lambda s: s["ms_total"])
    sub = pairs[::max(1, n_pairs // 60)].copy()
    want = sub.copy()
    oracle.batch(P, want, ref, qer, W)
    got = work[::max(1, n_pairs // 60)]
    assert all(np.array_equal(got[f], want[f]) for f in FIELDS), "bsw_extend32 differs from the oracle"
    line["extend32"] = {"pairs": n_pairs, "bases_query": int(pairs["len2"].sum()), "bases_target": int(pairs["len1"].sum()),
                        "call_s": t, "pairs_per_s": n_pairs / t, "cells_effective": int(st["cells_effective"]),
                        "gcups_call": st["cells_effective"] / t / 1e9, "kernel_ms": st["ms_kernel"],
                        "gcups_kernel": st["cells_effective"] / (st["ms_kernel"] * 1e-3) / 1e9,
                        "host_pack_ms": st["ms_pack"], "h2d_bytes": int(st["h2d_bytes"]), "checked_vs_oracle": len(sub)}
    # ---- the oracle, one host thread, on a subset of the same flanks
    sub = pairs[:40].copy()
    t0 = time.perf_counter()
    cells = oracle.batch(P, sub, ref, qer, W, nthreads=1)
    dt = time.perf_counter() - t0
    line["oracle_restated_1thread"] = {"pairs": len(sub), "cells": int(cells), "ns_per_cell": dt / cells * 1e9,
                                       "note": "oracle/ksw_oracle.c (the project's restatement of ksw_extend2), not the reference"}

    # ---- in-domain pairs: bsw_extend32 against bsw_extend
    cfg = gb.gen_named_config("large")
    ip, iref, iqer = gb.gen_pairs(cfg, 99, 200000)
    res = {}
    for name, fn in (("extend", eng.extend), ("extend32", eng.extend32)):
        wk = ip.copy()
        st_l = []

        def run_i():
            wk[:] = ip
            fn(wk, iref, iqer, W)
            st_l.append(eng.stats())
        ti = best_of(run_i)
        sti = min(st_l[1:], key=lambda s: s["ms_total"])
        res[name] = (wk.copy(), {"call_s": ti, "pairs_per_s": len(ip) / ti, "kernel_ms": sti["ms_kernel"],
                                 "gcups_call": sti["cells_effective"] / ti / 1e9,
                                 "gcups_kernel": sti["cells_effective"] / (sti["ms_kernel"] * 1e-3) / 1e9})
    assert all(np.array_equal(res["extend"][0][f], res["extend32"][0][f]) for f in FIELDS)
    line["in_domain_large"] = {"pairs": len(ip), "extend": res["extend"][1], "extend32": res["extend32"][1],
                               "extend32_over_extend_call": res["extend32"][1]["call_s"] / res["extend"][1]["call_s"]}

# ---- bsw_extend_chains on long reads ----------------------------------------------------------------------------------
rng = np.random.default_rng(2026)
L = 3_000_000
G = rng.integers(0, 4, size=L, dtype=np.uint8)
D = np.concatenate([G, (3 - G[::-1]).astype(np.uint8)])
reads = make_long_reads(rng, D, L, 100, 20000, 120000, (0.05, 0.12))
with gb.Engine(end_bonus=0, zdrop_mode=gb.BSW_ZDROP_SCALAR, **LONG_SCORING) as eng:
    chains, seeds, query, rseq = _chain_batch(gb, eng, reads, D, L, W, 1)
    out = (np.zeros(len(seeds), dtype=gb.ALNREG_DTYPE), np.zeros(len(chains), dtype=np.int32))
    stats = []

    def run_c():
        eng.extend_chains(chains, seeds, query, rseq, W, 0, 0, 2, out=out)
        stats.append(eng.stats())
    tc = best_of(run_c)
    stc = stats[-1]
    regs, count = out
    want = _oracle_chains(oracle, make_params(end_bonus=0, zdrop_mode=1, **LONG_SCORING), chains, seeds, query, rseq, W, 0, L)
    for k, ch in enumerate(chains):
        got = regs[int(ch["seed_first"]): int(ch["seed_first"]) + int(count[k])]
        assert len(got) == len(want[k]) and all(np.array_equal(got[f], want[k][f]) for f in ("rb", "re", "qb", "qe", "score", "truesc", "w")), k
    line["chains"] = {"reads": len(reads), "bases": int(len(query)), "seeds": int(len(seeds)), "regions": int(count.sum()),
                      "extensions": int(stc["pairs"]), "call_s": tc, "chains_per_s": len(chains) / tc,
                      "extensions_per_s": stc["pairs"] / tc, "cells_effective": int(stc["cells_effective"]),
                      "gcups_call": stc["cells_effective"] / tc / 1e9, "checked_vs_oracle": len(chains)}

s = json.dumps(line)
print(s)
if out_path:
    with open(out_path, "w") as f:
        f.write(s + "\n")

#!/usr/bin/env python
"""Throughput of bsw_global32 (ksw_global2 for long alignment regions, one warp per alignment, bsw_global32.cuh).
Prints one JSON line (and writes it to OUT when given):
  long_regions    N seeded regions of 5-100 kb (a mutated copy of the query as target, 8 % error) at w = 100-400: call
                  time, alignments/s, band GCUPS over the call and over the kernel time (CUDA events), and the DP and
                  backtrack kernels' shares from a separate torch.profiler run
  in_domain       bsw_global32 against bsw_global on the same alignments: the 210 000 short alignments of the tiled
                  global_default goldens, and 20-32 kb alignments at w = 100-400
  chains          the long-read chains of tests/test_extend32.py (100 reads of 20-120 kb, pacbio scoring) ->
                  bsw_extend_chains -> regions -> bsw_global32 CIGARs: regions/s
  oracle          oracle/global_oracle.c on one host thread: ns per band cell.  This is the project's CPU restatement of
                  ksw_global2, NOT the reference's code.
A sample of every timed result is checked against the oracle inside the run; the card's name and power limit are read
in the same run.  Usage: python scripts/long_global_bench.py [n_regions=2000] [reps=3] [OUT]"""
import json, os, subprocess, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import genomicsbench_b200 as gb
from oracle.pyoracle import Oracle, make_params
from test_extend32 import LONG_SCORING, _chain_batch, make_long_reads
from test_global32 import DEFAULT, check, load_golden, long_set, make_batch, oracle_all

n_regions = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
out_path = sys.argv[3] if len(sys.argv) > 3 else None


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


def rates(n, t, st):
    return {"alignments": n, "call_s": t, "alignments_per_s": n / t, "cells_band": int(st["cells_effective"]),
            "gcups_call": st["cells_effective"] / t / 1e9, "kernel_ms": st["ms_kernel"],
            "gcups_kernel": st["cells_effective"] / (st["ms_kernel"] * 1e-3) / 1e9, "host_pack_ms": st["ms_pack"],
            "h2d_bytes": int(st["h2d_bytes"]), "d2h_bytes": int(st["d2h_bytes"])}


def kernel_split(fn):
    """device time of the DP and the backtrack kernels in one profiled call (torch.profiler, CUDA activities)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    tot = {"dp": 0.0, "backtrack": 0.0}
    for k in prof.key_averages():
        us = getattr(k, "device_time_total", None)
        us = k.cuda_time_total if us is None else us
        if "bsw_global32_dp_kernel" in k.key:
            tot["dp"] += us / 1e3
        elif "bsw_global32_bt_kernel" in k.key:
            tot["backtrack"] += us / 1e3
    return {"dp_ms": tot["dp"], "backtrack_ms": tot["backtrack"],
            "backtrack_share": tot["backtrack"] / max(1e-9, tot["dp"] + tot["backtrack"])}


oracle = Oracle()
line = {"metric": "long_read_global_alignment", "card": card()}

# ---- long regions ---------------------------------------------------------------------------------------------------
rng = np.random.default_rng(7)
qs, ts, _ = long_set(2027, n_regions, 5000, 100000, err=0.08, wx=(0, 1))
ws = np.array([max(abs(len(q) - len(t)) + 3, int(rng.integers(100, 401))) for q, t in zip(qs, ts)], np.int32)
pairs, ref, qer = make_batch(qs, ts)
with gb.Engine(**DEFAULT) as eng:
    t, st, (score, cigar, off) = timed(eng, eng.global_align32, pairs, ref, qer, ws)
    idx = list(range(0, n_regions, max(1, n_regions // 12)))
    check(score, cigar, off, oracle_all(oracle, DEFAULT, qs, ts, ws, idx), idx)
    line["long_regions"] = dict(rates(n_regions, t, st), bases=int(pairs["len1"].sum() + pairs["len2"].sum()),
                                w="100-400", checked_vs_oracle=len(idx),
                                profiled=kernel_split(lambda: eng.global_align32(pairs, ref, qer, ws)))
    # a call with few long alignments: one warp's row latency
    few = pairs[:8].copy()
    t8, st8, _ = timed(eng, eng.global_align32, few, ref, qer, ws[:8])
    rows = int(few["len1"].max())
    line["long_regions"]["few_8"] = dict(rates(8, t8, st8), longest_rows=rows,
                                         us_per_row_longest=st8["ms_kernel"] * 1e3 / rows)

# ---- in-domain: bsw_global32 against bsw_global ---------------------------------------------------------------------
P, gp, gref, gqer, gw, score_g, _, cigar_g = load_golden("global/global_default")
big, wb = np.tile(gp, 300), np.tile(gw, 300)
with gb.Engine(**P) as eng:
    res = {}
    for name, fn in (("global", eng.global_align), ("global32", eng.global_align32)):
        t, st, r = timed(eng, fn, big, gref, gqer, wb)
        res[name] = (r, rates(len(big), t, st))
    assert np.array_equal(res["global"][0][0], res["global32"][0][0]) and np.array_equal(res["global"][0][1], res["global32"][0][1])
    assert np.array_equal(res["global32"][0][0], np.tile(score_g, 300)) and np.array_equal(res["global32"][0][1], np.tile(cigar_g, 300))
    line["in_domain_short_210k"] = {"global": res["global"][1], "global32": res["global32"][1],
                                    "global32_over_global_call": res["global32"][1]["call_s"] / res["global"][1]["call_s"]}
    qs2, ts2, _ = long_set(2028, 1000, 20000, 32000, err=0.08, wx=(0, 1))
    ws2 = np.array([max(abs(len(q) - len(t)) + 3, int(rng.integers(100, 401))) for q, t in zip(qs2, ts2)], np.int32)
    keep = [k for k in range(len(qs2)) if len(qs2[k]) <= 32767 and len(ts2[k]) <= 32767]
    qs2, ts2, ws2 = [qs2[k] for k in keep], [ts2[k] for k in keep], ws2[keep]
    p2, r2, q2 = make_batch(qs2, ts2)
with gb.Engine(**DEFAULT) as eng:
    res = {}
    for name, fn in (("global", eng.global_align), ("global32", eng.global_align32)):
        t, st, r = timed(eng, fn, p2, r2, q2, ws2)
        res[name] = (r, rates(len(p2), t, st))
    assert all(np.array_equal(a, b) for a, b in zip(res["global"][0], res["global32"][0]))
    idx = list(range(0, len(p2), 100))
    check(*res["global32"][0], oracle_all(oracle, DEFAULT, qs2, ts2, ws2, idx), idx)
    line["in_domain_20_32kb"] = {"w": "100-400", "global": res["global"][1], "global32": res["global32"][1],
                                 "global_over_global32_call": res["global"][1]["call_s"] / res["global32"][1]["call_s"]}

# ---- long-read chains -> regions -> CIGARs ---------------------------------------------------------------------------
crng = np.random.default_rng(2026)                         # the long_reads fixture of tests/test_extend32.py
L = 3_000_000
G = crng.integers(0, 4, size=L, dtype=np.uint8)
D = np.concatenate([G, (3 - G[::-1]).astype(np.uint8)])
reads = make_long_reads(crng, D, L, 100, 20000, 120000, (0.05, 0.12))
W = 100
with gb.Engine(end_bonus=0, zdrop_mode=gb.BSW_ZDROP_SCALAR, **LONG_SCORING) as eng:
    chains, seeds, query, rseq = _chain_batch(gb, eng, reads, D, L, W, 1)
    t0 = time.perf_counter()
    regs, count = eng.extend_chains(chains, seeds, query, rseq, W, 0, 0, 2)
    t_chain = time.perf_counter() - t0
    cq, ct, cw = [], [], []
    for k, ch in enumerate(chains):
        read = query[int(ch["query_off"]): int(ch["query_off"]) + int(ch["l_query"])]
        for r in regs[int(ch["seed_first"]): int(ch["seed_first"]) + int(count[k])]:
            q, tt = read[int(r["qb"]): int(r["qe"])], D[int(r["rb"]): int(r["re"])]
            if len(q) and len(tt):
                cq.append(q); ct.append(tt); cw.append(max(int(r["w"]), abs(len(q) - len(tt)) + 3))
    cw = np.array(cw, np.int32)
    cp, cr, cqq = make_batch(cq, ct)
    t, st, (score, cigar, off) = timed(eng, eng.global_align32, cp, cr, cqq, cw)
    idx = list(range(0, len(cq), 10))
    check(score, cigar, off, oracle_all(oracle, LONG_SCORING, cq, ct, cw, idx), idx)
    line["chains"] = dict(rates(len(cq), t, st), reads=len(reads), regions=len(cq),
                          longest_region=int(max(cp["len1"].max(), cp["len2"].max())), regions_per_s=len(cq) / t,
                          extend_chains_s=t_chain, chains_to_cigars_per_s=len(chains) / (t_chain + t),
                          checked_vs_oracle=len(idx))

# ---- the oracle on one host thread ------------------------------------------------------------------------------------
Po = make_params(**DEFAULT)
cells, dt = 0, 0.0
for k in range(3):
    T, Q, Wk = len(ts[k]), len(qs[k]), int(ws[k])
    cells += sum(min(i + Wk + 1, Q) - max(i - Wk, 0) for i in range(T))
    t0 = time.perf_counter()
    oracle.global_align(Po, qs[k], ts[k], Wk)
    dt += time.perf_counter() - t0
line["oracle_restated_1thread"] = {"alignments": 3, "cells_band": cells, "ns_per_cell": dt / cells * 1e9,
                                   "note": "oracle/global_oracle.c (the project's restatement of ksw_global2), not the reference"}

s = json.dumps(line)
print(s)
if out_path:
    with open(out_path, "w") as f:
        f.write(s + "\n")

#!/usr/bin/env python
"""ONE engine, ONE call, N devices: strong scaling of the in-call partitioner (contiguous cost-balanced range per
device, one host thread each) on configs[4]'s divergent pairs and on the large mix.

    python scripts/multi_probe.py [--pairs 8000000] [--workload sweep] [--max-devices 8]
"""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import genomicsbench_b200 as gb  # noqa: E402
import torch  # noqa: E402


def timeit(fn, steps, warm=2):
    for _ in range(warm):
        fn()
    t = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        t.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(t))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=8_000_000)
    ap.add_argument("--workload", default="sweep")
    ap.add_argument("--max-devices", type=int, default=8)
    ap.add_argument("--steps", type=int, default=4)
    args = ap.parse_args()
    ngpu = min(torch.cuda.device_count(), args.max_devices)
    cfg = gb.gen_named_config(args.workload)
    pairs, ref, qer = gb.gen_pairs(cfg, 0, args.pairs)
    nominal = float((pairs["len1"].astype(np.int64) * pairs["len2"]).sum())
    pp, pr, pq = gb.pinned_copy(pairs), gb.pinned_copy(ref), gb.pinned_copy(qer)
    batch = gb.PackedBatch.from_pairs(pairs, ref, qer, pinned=True)
    out = gb.pinned_empty(len(pairs), gb.OUTSCORE_DTYPE)
    res = {"workload": args.workload, "pairs": args.pairs, "points": {}}
    base = None
    nd = 1
    while nd <= ngpu:
        with gb.Engine(devices=list(range(nd))) as eng:
            ms_pk = timeit(lambda: eng.extend_packed(batch, 100, out=out), args.steps)
            st = eng.stats()
            ms_di = timeit(lambda: eng.extend(pp, pr, pq, 100), args.steps)
            same = all(np.array_equal(out[f], pp[f]) for f in gb.RESULT_FIELDS)
            if base is None:
                base = {f: pp[f].copy() for f in gb.RESULT_FIELDS}
            same = same and all(np.array_equal(base[f], pp[f]) for f in gb.RESULT_FIELDS)
        res["points"][nd] = {"packed_ms": ms_pk, "packed_gcups": nominal / ms_pk / 1e6, "dropin_ms": ms_di,
                             "dropin_gcups": nominal / ms_di / 1e6, "shards": st["shards"], "kernel_ms_max_device": st["ms_kernel"],
                             "results_equal_single_device": bool(same)}
        print(nd, json.dumps(res["points"][nd]), flush=True)
        nd *= 2
    p1 = res["points"][1]
    for nd, p in res["points"].items():
        p["packed_speedup"] = p1["packed_ms"] / p["packed_ms"]
        p["dropin_speedup"] = p1["dropin_ms"] / p["dropin_ms"]
    print(json.dumps(res))


if __name__ == "__main__":
    main()

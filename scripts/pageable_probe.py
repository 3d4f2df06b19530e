"""Pageable (unmodified-driver) route: end-to-end time of bsw_extend on pageable numpy buffers, host pass times, PCIe bytes
per pair, and the resident kernel time of a batch staged from them."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, genomicsbench_b200 as gb
for name, idx in (("short8", 1), ("large", 3), ("long16", 2)):
    pairs, ref, qer = gb.gen_pairs(gb.gen_named_config(idx), 0, 1_000_000)
    with gb.Engine() as eng:
        for _ in range(3): eng.extend(pairs, ref, qer, 100)
        t=[]
        for _ in range(8):
            t0=time.perf_counter(); eng.extend(pairs, ref, qer, 100); t.append((time.perf_counter()-t0)*1e3)
        st=eng.stats()
        eng.stage(pairs, ref, qer, 100)
        ks=[]
        for _ in range(8):
            eng.run_staged(); ks.append(eng.stats()["ms_kernel"])
        print(name, "pageable e2e ms median %.3f min %.3f | host in %.2f out %.2f | h2d B/pair %.0f | resident kernel ms %.3f" % (np.median(t), np.min(t), st["ms_pack"], st["ms_scatter"], st["h2d_bytes"]/len(pairs), np.median(ks[2:])), flush=True)

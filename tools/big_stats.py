"""Reads-per-chain histogram of a workload after filtering, in bands of final reads per chain with each band's share of
sum n^3 (chains of up to 160 reads cluster in shared memory, longer ones in k_cluster_sparse).
python tools/big_stats.py --workload cfg3 --scale 0.25"""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ahsoka_b200 import api, synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="cfg3")
ap.add_argument("--scale", type=float, default=0.25)
a = ap.parse_args()
b = synth.generate(synth.config(a.workload, a.scale))
r = api.phase_batch(b, device=0, resident_iters=2, warmup=1)
n = np.diff(np.asarray(r.read_off))
print("chains", len(n), "reads/chain: mean %.1f" % n.mean(), "percentiles 50/90/99/max", np.percentile(n, [50, 90, 99, 100]))
for lo, hi in ((0, 128), (129, 168), (169, 256), (257, 512), (513, 10 ** 9)):
    m = (n >= lo) & (n <= hi)
    print("  %4d..%-6s chains %6d  sum n^3 share %.3f" % (lo, hi if hi < 10 ** 9 else "inf", m.sum(), (n[m].astype(float) ** 3).sum() / (n.astype(float) ** 3).sum()))
print({k: round(v, 2) for k, v in r.timings.items()})

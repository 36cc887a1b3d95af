"""Cost and effect of caller genotypes (ahs_phase_batch_genotyped) on the BASELINE workloads.

For each workload, in one process, three variants are called alternately: plain (no dosages), all-zero dosages (must give
the plain result bit for bit) and the generator's true dosages (synth.true_dosage).  2 warm-up calls of each, then 5 timed
calls of each; per variant the median and the spread (min, max) of ms_thread and ms_total_device (CUDA events of the
library).  Also per variant: the share of covered positions, over the chains of >= 10 positions, whose emitted hap_allele
multiset equals the truth.  Writes genotype_probe.json to --out with the GPU name, power limit and max SM clock.

    python tools/genotype_probe.py --out DIR [--workloads cfg2,cfg3,cfg4:0.1,cfg5cap:0.1]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ahsoka_b200 import api, synth  # noqa: E402

WARMUP, TIMED = 2, 5


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=60).stdout
    except (OSError, subprocess.TimeoutExpired) as e:
        out = f"nvidia-smi unavailable: {e}"
    return out.strip().splitlines()


def truth_agreement(batch, r):
    """share of the covered positions of chains with >= 10 positions whose hap_allele multiset is the true one"""
    p = batch.ploidy
    npos = np.diff(r.pos_off)
    keep = (r.status == 0) & (npos >= 10)
    chain = np.repeat(np.arange(batch.n_chains), npos)
    sel = keep[chain]
    gb = batch.bubble_off[chain[sel]] + r.pos[sel]
    truth = np.sort(batch.truth["hap_allele"].reshape(-1, p)[gb], axis=1)
    hap = np.sort(r.hap_allele.reshape(-1, p)[sel], axis=1)
    n = int(sel.sum())
    return {"positions": n, "agree": int((truth == hap).all(axis=1).sum()), "share": float((truth == hap).all(axis=1).mean()) if n else None}


def stats(xs):
    return {"median": float(np.median(xs)), "min": float(np.min(xs)), "max": float(np.max(xs)), "all": [float(x) for x in xs]}


def probe(name, scale):
    b = synth.generate(synth.config(name, scale))
    n_alleles = int(b.allele_off[-1])
    variants = {"plain": None, "zero": np.zeros(n_alleles, np.uint8), "true": synth.true_dosage(b)}
    times = {v: {"ms_thread": [], "ms_total_device": []} for v in variants}
    last = {}
    for it in range(WARMUP + TIMED):
        for v, d in variants.items():                               # alternate the variants
            b.allele_dosage = d
            r = api.phase_batch(b)
            if it >= WARMUP:
                for k in times[v]:
                    times[v][k].append(r.timings[k])
            last[v] = r
    b.allele_dosage = None
    bad = last["zero"].diff(last["plain"])
    assert not bad, f"{name}: all-zero dosages differ from the plain call in {bad}"
    out = {"workload": name, "scale": scale, "ploidy": int(b.ploidy), "chains": b.n_chains, "bubbles": int(b.bubble_off[-1]),
           "positions": int(last["plain"].pos_off[-1]), "zero_equals_plain": True,
           "true_differs_from_plain": last["true"].diff(last["plain"])}
    for v in variants:
        out[v] = {k: stats(x) for k, x in times[v].items()}
        out[v]["truth_agreement"] = truth_agreement(b, last[v])
    out["ms_thread_overhead_true_vs_plain"] = out["true"]["ms_thread"]["median"] - out["plain"]["ms_thread"]["median"]
    out["ms_thread_overhead_zero_vs_plain"] = out["zero"]["ms_thread"]["median"] - out["plain"]["ms_thread"]["median"]
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="directory for genotype_probe.json")
    ap.add_argument("--workloads", default="cfg2,cfg3,cfg4:0.1,cfg5cap:0.1", help="name[:scale],...")
    a = ap.parse_args()
    if api.load_library().ahs_device_count() < 1:
        raise SystemExit("no CUDA device: the phasing path has no CPU fallback")
    os.makedirs(a.out, exist_ok=True)
    res = {"gpu": gpu_info(), "warmup": WARMUP, "timed": TIMED, "workloads": []}
    for w in a.workloads.split(","):
        name, _, scale = w.partition(":")
        r = probe(name, float(scale) if scale else 1.0)
        res["workloads"].append(r)
        print(json.dumps({k: r[k] for k in ("workload", "scale", "ms_thread_overhead_true_vs_plain")} |
                         {v: (r[v]["ms_thread"]["median"], r[v]["ms_total_device"]["median"], r[v]["truth_agreement"]["share"])
                          for v in ("plain", "zero", "true")}), flush=True)
    with open(os.path.join(a.out, "genotype_probe.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py — read-bubble cells phased per second (BASELINE.json metric) on N B200s.

A "step" is one pass of the phasing hot path (projection -> scoring -> cluster editing ->
coverage/consensus -> threading DP) over one synthetic batch.  The workload at every N is
BASELINE.json configs[1] ("synthetic diploid human-scale graph: 50k chains, 2M bubbles, 30x
ultra-long reads"), one full batch PER GPU (chains are independent: weak scaling, no collective
on the data path; torch.distributed is only the barrier / max-over-ranks plumbing).

  value : cells/s with the batch resident in HBM, timed with CUDA events on the library's
          stream around each pass (ahs_phase_batch_resident), max over ranks.
  e2e   : cells/s through the public call ahs_phase_batch() with pinned HOST buffers; H2D of the
          whole CSR batch and D2H of every result array are inside the timed region.
  --impl reference : the reference's own sources compiled verbatim (+ WhatsHap API shim, see
          oracle/) run as `Ahsoka phase -t 1` on a bounded GFA/GAF sample of the same workload.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "read-bubble cells phased/sec"
UNIT = "cells/s"


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index, all_gpus=False):
        self.gpu, self.rows, self.proc, self.all_gpus = gpu_index, [], None, all_gpus

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi"] + ([] if self.all_gpus else ["-i", str(self.gpu)]) + ["--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        by_gpu, pw_gpu = {}, {}
        for r in self.rows:
            try:
                by_gpu.setdefault(int(r[0]), []).append(float(r[1])); pw_gpu.setdefault(int(r[0]), []).append(float(r[3]))
            except Exception:
                pass
        self.per_gpu = {"sm_mhz": [statistics.median(by_gpu[g]) for g in sorted(by_gpu)], "power_w": [round(statistics.median(pw_gpu[g]), 1) for g in sorted(pw_gpu)]}
        for r in self.rows:
            try:
                if int(r[0]) != self.gpu:
                    continue
                sm.append(float(r[1])); mx.append(float(r[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_batch(workload, scale, rank):
    from ahsoka_b200 import synth
    prm = synth.config(workload, scale)
    prm.seed = prm.seed + 1000 * rank          # every rank phases its own chains
    return synth.generate(prm)


WORKLOAD_NAMES = {"cfg1": "cfg1: BASELINE.json configs[0] one chain of 1k bubbles, 2k reads",
                  "cfg2": "cfg2: BASELINE.json configs[1] synthetic diploid human-scale graph",
                  "cfg3": "cfg3: BASELINE.json configs[2] synthetic triploid graph",
                  "cfg4": "cfg4: BASELINE.json configs[3] synthetic tetraploid graph",
                  "cfg5": "cfg5: BASELINE.json configs[4] synthetic hexaploid graph, Zipf-skewed chain sizes",
                  "cfg5cap": "cfg5cap: BASELINE.json configs[4] with chain length capped at 1000 bubbles",
                  "zipf2": "zipf2: diploid, Zipf-skewed chain sizes up to 10k bubbles (load-balancing stress)"}


def workload_desc(workload, scale, batch):
    return {"workload": WORKLOAD_NAMES.get(workload, workload),
            "scale": scale, "chains_per_gpu": batch.n_chains, "bubbles_per_gpu": int(batch.bubble_off[-1]),
            "reads_per_gpu": int(batch.read_off[-1]), "entry_nodes_per_gpu": int(batch.enode.shape[0]), "ploidy": int(batch.ploidy),
            "l2": "inputs (%.0f MB) and per-chain workspaces exceed the 126 MB L2; no explicit flush" % (batch.nbytes() / 1e6)}


def cpu_port_baseline(batch, seconds_target=15.0):
    """CPU oracle (restatement, all host threads) on a bounded prefix of the same workload."""
    from tests.oracle_binding import oracle_phase
    cores = os.cpu_count() or 1
    n = min(batch.n_chains, max(cores * 4, 64))
    sub = batch.select(np.arange(n))
    t0 = time.perf_counter(); r = oracle_phase(sub, cores); dt = time.perf_counter() - t0
    # grow the sample towards the time target (bounded)
    rate = max(r.n_cells / max(dt, 1e-6), 1.0)
    want = int(min(batch.n_chains, max(n, n * seconds_target / max(dt, 1e-3) * 0.8)))
    if want > 2 * n and dt < seconds_target / 4:
        sub = batch.select(np.arange(want))
        t0 = time.perf_counter(); r = oracle_phase(sub, cores); dt = time.perf_counter() - t0
        n = want
        rate = r.n_cells / max(dt, 1e-6)
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"first {n} chains of the batch ({r.n_cells} cells) in {dt:.2f} s, oracle/phase_oracle.cpp, {cores} threads",
            "chains_per_s": r.n_chains_ok / max(dt, 1e-6)}


def run_reference_arm(args):
    """Reference sources verbatim (+ WhatsHap shim) as `Ahsoka phase -t 1`, one process per host core, each on its own
    bounded sample of the workload (the reference is single-threaded: -t > 1 is an unfinished experiment, SURVEY 0.8)."""
    from ahsoka_b200 import synth
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    exe = os.path.join(ROOT, "oracle", "_ref", "Ahsoka_ref")
    cores = os.cpu_count() or 1
    # bounded sample: the reference-verbatim CLI costs ~2.6 s per cfg2 chain on one core (its projection is
    # O(bubbles x alleles x entries), SURVEY 0.7); keep the whole K+W run near 2-3 minutes
    n_chains = args.ref_chains if args.ref_chains > 0 else int(max(2, min(12, 150.0 / (2.6 * (args.steps + args.warmup)))))
    times, cells, chains = [], 0, 0
    kind, sample = "reference", ""
    with tempfile.TemporaryDirectory() as td:
        if os.path.exists(exe):
            from tests.oracle_binding import oracle_phase
            n_proc = cores
            for i in range(n_proc):
                prm = synth.config(args.workload, 1.0)
                prm.n_chains = n_chains; prm.seed = prm.seed + 7919 * i
                batch = synth.generate(prm, os.path.join(td, f"s{i}"))
                want = oracle_phase(batch)           # only to count the cells the CLI runs phase (not timed)
                cells += want.n_cells; chains += want.n_chains_ok
            for it in range(args.warmup + args.steps):
                t0 = time.perf_counter()
                procs = [subprocess.Popen([exe, "phase", "-g", os.path.join(td, f"s{i}.gfa"), "-a", os.path.join(td, f"s{i}.gaf"),
                                           "-o", os.path.join(td, f"o{it}_{i}"), "-t", "1"], cwd=td, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                         for i in range(n_proc)]
                rcs = [p.wait() for p in procs]
                dt = time.perf_counter() - t0
                if any(rcs):
                    raise SystemExit("bench.py: the reference binary failed on the sample")
                if it >= args.warmup:
                    times.append(dt)
            sample = (f"{n_proc} concurrent `Ahsoka phase -t 1` processes (one per host core), each on its own {n_chains}-chain GFA+GAF sample of "
                      f"{args.workload} (reference src/*.cpp verbatim at -O2 + WhatsHap API shim), whole CLI runs incl. parsing")
        else:
            from tests.oracle_binding import oracle_phase
            kind = "port"
            prm = synth.config(args.workload, 1.0)
            prm.n_chains = n_chains * cores * 8
            batch = synth.generate(prm)
            for it in range(args.warmup + args.steps):
                t0 = time.perf_counter(); r = oracle_phase(batch, cores); dt = time.perf_counter() - t0
                cells, chains = r.n_cells, r.n_chains_ok
                if it >= args.warmup:
                    times.append(dt)
            sample = f"{prm.n_chains} chains of {args.workload}, CPU oracle port, {cores} threads (reference-verbatim binary not built)"
    dt = sum(times) / len(times)
    val = cells / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32/i64 fixed point",
            "data": "synthetic", "config": {"workload": WORKLOAD_NAMES.get(args.workload, args.workload), "sample_chains": n_chains * (cores if kind == "reference" else cores * 8),
                                            "cells": cells, "ploidy": int(synth.config(args.workload, 1.0).ploidy)},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "chains_per_s": chains / dt},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    _emit(line)
    return 0


DUMP_MAX_ELEMS = 1 << 19          # per array: 15 arrays x 4 MB of float64 stay under 64 MB


def dump_outputs(res, out_dir):
    """Every array of the result as <out_dir>/<name>.npy in float64 (the integer values are exact there), plus the three
    counts.  An array above DUMP_MAX_ELEMS elements is replaced by the elements at a fixed, seeded, sorted sample of
    indices, so that two builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: getattr(res, k) for k in res.ARRAYS}
    arrays.update({k: np.array([getattr(res, k)]) for k in ("n_cells", "n_pairs", "n_chains_ok")})
    for name, a in arrays.items():
        a = np.ascontiguousarray(a).reshape(-1)
        if a.size > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(20261020).choice(a.size, DUMP_MAX_ELEMS, replace=False))
            a = a[idx]
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def _emit(line):
    """The ONE JSON line goes to the real stdout; everything else a library prints there (NCCL's version banner,
    torchrun notices) was redirected to stderr at start-up."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed passes of every single-device leg (the N > 1 multi-device check times 3 calls)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--ref-chains", type=int, default=0, help="chains in the reference-arm sample (0 = sized from steps + warmup)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result arrays of the last timed pass as DIR/<name>.npy (float64; rank 0's batch when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the result of the b200 path")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        return run_reference_arm(args)

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    from ahsoka_b200 import api
    lib = api.load_library()
    if lib.ahs_device_count() <= local:
        raise SystemExit("bench.py: no CUDA device for this rank; the phasing path has no CPU fallback")

    # one rank = one GPU = one share of the host cores (the ranks of a box would otherwise all run on the same CPUs)
    try:
        cpus = sorted(os.sched_getaffinity(0))
        if world > 1 and len(cpus) >= world:
            per = len(cpus) // world
            os.sched_setaffinity(0, set(cpus[local * per:(local + 1) * per]))
    except (AttributeError, OSError):
        pass

    batch = make_batch(args.workload, args.scale, rank)
    api.pin_batch(batch)

    def barrier():
        if dist is not None:
            import torch
            dist.barrier(); torch.cuda.synchronize()

    sampler = ClockSampler(local, all_gpus=world > 1)
    # ---- device-resident timing: W warm-up passes, K timed passes, CUDA events inside the library
    barrier()
    if rank == 0:
        sampler.start()
    res = api.phase_batch(batch, device=local, resident_iters=args.steps, warmup=args.warmup)
    barrier()
    t = res.timings
    ms_step = t["ms_total_device"]
    # ---- end to end through the public call: host buffers in, host buffers out
    # (results are numpy views of the library's pinned output buffers: the C ABI contract, no extra host copy)
    for _ in range(2):
        api.phase_batch(batch, device=local, copy=False).release()
    barrier()
    e2e_times, d2h = [], 0
    for _ in range(args.steps):
        t0 = time.perf_counter(); r2 = api.phase_batch(batch, device=local, copy=False); e2e_times.append(time.perf_counter() - t0)
        d2h = sum(getattr(r2, k).nbytes for k in r2.ARRAYS)
        assert r2.n_cells == res.n_cells and int(r2.read_cluster.shape[0]) == int(res.read_off[-1])
        r2.release()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    e2e_ms = 1e3 * sum(e2e_times) / len(e2e_times)
    ahead_ms = None
    if os.environ.get("BENCH_AHEAD_LEG"):          # diagnostic: the same loop with the look-ahead upload order of the library
        os.environ["AHS_UPLOAD_AHEAD"] = "1"
        api.phase_batch(batch, device=local, copy=False).release()
        barrier()
        ta = []
        for _ in range(args.steps):
            t0 = time.perf_counter(); api.phase_batch(batch, device=local, copy=False).release(); ta.append(time.perf_counter() - t0)
        barrier()
        os.environ["AHS_UPLOAD_AHEAD"] = "0"
        ahead_ms = 1e3 * sum(ta) / len(ta)
    # ---- N > 1: the north-star split, checked once outside the timed regions.  Rank 0 deals ITS batch over all N
    # devices of the box inside one process (ahs_phase_batch_multi: one contiguous, cost-balanced share of the chains
    # per device; no inter-GPU traffic; every device writes its ranges straight into the output arrays)
    # and compares every output array with the single-device result; the other ranks idle at the barrier.
    def multi_leg(single_ms):
        devs = list(range(world))
        single = api.phase_batch(batch, device=local)
        api.phase_batch(batch, devices=devs, copy=False).release()          # contexts + pools of the other devices
        mt, ms_dev = [], 0.0
        for _ in range(3):
            t0 = time.perf_counter(); rm = api.phase_batch(batch, devices=devs, copy=False); mt.append(time.perf_counter() - t0)
            bad = rm.diff(single)
            ms_dev = rm.timings["ms_total_device"]
            rm.release()
            if bad:
                raise RuntimeError(f"multi-device result differs from the single-device result in {bad}")
        return {"ms_per_call": 1e3 * min(mt), "single_device_ms_same_inputs": single_ms, "speedup": single_ms / (1e3 * min(mt)),
                "slowest_device_first_to_last_kernel_ms": ms_dev}

    def checked_multi_leg(single_ms):
        # the check runs outside the timed regions: a failure is reported in the line (and on stderr), loudly, without
        # discarding the per-rank measurement the other ranks are waiting to reduce
        try:
            return multi_leg(single_ms)
        except Exception as e:            # noqa: BLE001
            multi["equal_to_single_device"] = False
            print(f"bench.py: MULTI-DEVICE CHECK FAILED: {e}", file=sys.stderr, flush=True)
            return {"error": str(e)}

    # While rank 0 uses every GPU, the other ranks must be off theirs: an NCCL barrier spins ON the device (and two processes
    # time-slice one GPU), so they wait on the rendezvous store instead — a CPU wait.
    store = None
    if dist is not None:
        from torch.distributed.distributed_c10d import _get_default_store
        store = _get_default_store()

    def others_wait(tag):
        if store is None:
            return
        if rank == 0:
            store.set(tag, "1")
        else:
            store.wait([tag])

    multi = None
    do_multi = world > 1 and rank == 0 and lib.ahs_device_count() >= world
    if do_multi:
        multi = {"devices": world, "equal_to_single_device": True,
                 "what": "one batch dealt over all devices by ahs_phase_batch_multi inside rank 0 (strong scaling of one call; the other ranks wait off the GPU)"}
        multi["pinned_inputs"] = checked_multi_leg(e2e_ms)
    others_wait("ahs_multi_pinned_done")
    barrier()
    # ---- the same call with PAGEABLE input arrays, as a one-shot caller (the drop-in CLI) passes them
    api.unpin_batch(batch)
    api.phase_batch(batch, device=local, copy=False).release()
    pg_times = []
    for _ in range(args.steps):
        t0 = time.perf_counter(); r2 = api.phase_batch(batch, device=local, copy=False); pg_times.append(time.perf_counter() - t0)
        r2.release()
    e2e_pageable_ms = 1e3 * sum(pg_times) / len(pg_times)
    barrier()
    if do_multi:
        multi["pageable_inputs"] = checked_multi_leg(e2e_pageable_ms)
    others_wait("ahs_multi_pageable_done")
    barrier()

    cells, chains_ok = res.n_cells, res.n_chains_ok
    cells_local = cells
    per_rank = None
    if dist is not None:
        import torch
        # every rank's own numbers (the line's times are the max over ranks): shows whether a drop in efficiency is one slow rank or all of them
        mine = torch.tensor([ms_step, e2e_ms, float(cells), t["ms_cluster"], t["ms_project"], 1e3 * min(e2e_times), 1e3 * max(e2e_times), ahead_ms or 0.0],
                            device=f"cuda:{local}", dtype=torch.float64)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        cols = ["ms_per_step", "e2e_ms_per_step", "cells", "ms_cluster", "ms_project", "e2e_ms_min", "e2e_ms_max", "e2e_ms_upload_ahead_leg"]
        per_rank = {c: [round(float(a[i]), 3) for a in allr] for i, c in enumerate(cols)}
        if clocks is not None and len(getattr(sampler, "per_gpu", {}).get("sm_mhz", [])) >= world:
            per_rank["sm_mhz_median_by_gpu"] = sampler.per_gpu["sm_mhz"]; per_rank["power_w_median_by_gpu"] = sampler.per_gpu["power_w"]
        try:
            per_rank["cpus_rank0"] = sorted(os.sched_getaffinity(0))
        except (AttributeError, OSError):
            pass
        v = torch.tensor([ms_step, e2e_ms], device=f"cuda:{local}", dtype=torch.float64)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        ms_step, e2e_ms = float(v[0]), float(v[1])
        s = torch.tensor([cells, chains_ok], device=f"cuda:{local}", dtype=torch.int64)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        cells, chains_ok = int(s[0]), int(s[1])
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peak, peak_src = measured_peak()
    stages = {}
    for name, ms_key, bytes_key in (("project", "ms_project", "bytes_project"), ("score", "ms_score", "bytes_score"),
                                    ("consensus", "ms_consensus", "bytes_consensus")):
        ms = t[ms_key]; b = t[bytes_key]
        gbs = b / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        stages[name] = {"ms": ms, "algorithmic_bytes": b, "achieved_gbs": gbs, "frac": gbs / peak}
    for name, ms_key in (("rows", "ms_rows"), ("cluster_edit", "ms_cluster"), ("thread_dp", "ms_thread")):
        stages[name] = {"ms": t[ms_key], "bound": "latency / integer pipes (not an HBM-roofline stage)"}
    dominant = max(("project", "rows", "score", "cluster_edit", "consensus", "thread_dp"), key=lambda k: stages[k]["ms"])
    sc = stages["score"]
    traffic = None                     # dram bytes of the scoring kernels from the committed `ncu --set full` capture
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and args.workload == "cfg2" and args.scale == 1.0:
        try:
            traffic = json.load(open(tp)).get("score_dram_bytes_per_pass")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "score = k_score_chain launches (read-pair agreement scoring, K2; one pass = all size classes)",
                "achieved": sc["achieved_gbs"], "peak": peak, "unit": "GB/s", "frac": sc["frac"], "traffic": traffic,
                "peak_source": peak_src, "dominant_stage_by_time": dominant, "stages": stages}
    line = {"metric": METRIC, "value": cells / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8 codes / i32-i64 fixed point",
            "data": "synthetic", "config": dict(workload_desc(args.workload, args.scale, batch), parallelism=f"chains x{world} (no collective)"),
            "chains_per_s": chains_ok / (ms_step * 1e-3), "cells": cells, "pairs_per_gpu": res.n_pairs,
            "e2e": {"value": cells / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": batch.nbytes(), "d2h_bytes_per_step": int(d2h),
                    "ms_per_step": e2e_ms, "inputs": "page-locked host arrays (ahs_pin_host, outside the timed region)",
                    "pageable_inputs": {"value": cells_local / (e2e_pageable_ms * 1e-3), "ms_per_step": e2e_pageable_ms, "n_gpus": 1,
                                        "what": "rank 0's call with plain pageable numpy arrays, as a one-shot caller passes them"}},
            "gpu_launches": int(t["n_launches"]) * args.steps, "roofline": roofline, "clocks": clocks}
    if multi is not None:
        line["multi"] = multi
    if per_rank is not None:
        line["per_rank"] = per_rank
    if not args.no_cpu_baseline and world == 1:          # reported on rank 0 at N=1 only
        line["cpu_baseline"] = cpu_port_baseline(batch)
    if args.dump_outputs:
        dump_outputs(res, args.dump_outputs)
    _emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

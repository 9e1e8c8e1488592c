#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on its headline config (relpose_5pt essential, 10 000 2D-2D corrs, 30 % inliers,
max 100 000 iterations), one JSON line.

A step = one pass of the LO-RANSAC hot path over a batch of `--pairs` independent synthetic image pairs of that
config (own data seed each), per GPU.  Metric = RANSAC hypotheses/s (models passed to score_model) with
scored-correspondences/s alongside.
  value : whole job with the correspondences already resident in HBM (plb_resident_create handles)
  e2e   : the same batch through the reference-facing C-ABI call with HOST buffers: the host->device copy of the
          correspondences / sample tables and the device->host read of records, models and inlier masks are inside
          the timed region (counted from the copies the engine makes)
  --impl reference : the CPU restatement of the reference path (oracle/, the reference itself needs Eigen3, which
          this image lacks) on the host cores, one problem per thread, same config/metric; the reference's own sources
          built on mini-Eigen (oracle/_ref/libplref2.so) are timed beside it as `reference_sources` (informational).
Multi-GPU (torchrun): independent image pairs are sharded across ranks, no data-path collective; weak scaling.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from poselib_b200 import problem_generator as G  # noqa: E402

BYTES_PER_CORR_FP64 = 32  # the exact-mode kernel reads 4 fp64 per 2D-2D correspondence (DESIGN.md §kernels)


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"], "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


def usable_cores():
    """Host cores this process may actually use: affinity mask and cgroup CPU quota (the box reports 128 logical CPUs
    but the container may be limited to fewer)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def cpu_model():
    try:
        for l in open("/proc/cpuinfo"):
            if l.startswith("model name"):
                return l.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


_PIN = False  # set by main() of the GPU arm: host buffers of the timed calls are page-locked (the harness's e2e contract)


def pin(a):
    """float64 C-contiguous copy of `a` in page-locked host memory (the engine then DMAs straight from it)."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    if not _PIN:
        return a
    import torch
    return torch.from_numpy(a).pin_memory().numpy()  # the array keeps the pinned tensor alive


def make_batch(pairs, first_idx):
    probs = []
    for i in range(pairs):
        p = G.config_c2(first_idx + i)
        probs.append((pin(p["x1"] / G.FOCAL), pin(p["x2"] / G.FOCAL)))
    return probs


def totals(results):
    hyp = sum(r["counters"]["hypotheses"] for r in results)
    cor = sum(r["counters"]["scored_corrs"] for r in results)
    smp = sum(r["counters"]["samples"] for r in results)
    return hyp, cor, smp


def run_reference(args, rank, world):
    """CPU arm: oracle restatement, all host threads, one problem per thread (the reference itself is single-threaded)."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import plo_py as P
    threads = usable_cores()
    pairs = max(threads, min(args.pairs, 2 * threads))  # bounded sample of the same workload, >= one problem per core
    batch = make_batch(pairs, 0)
    opts = [P.RansacOpt(max_iterations=100000, min_iterations=1000, seed=0) for _ in range(pairs)]
    me = [1.0 / G.FOCAL] * pairs
    x1, x2 = [b[0] for b in batch], [b[1] for b in batch]
    for _ in range(args.warmup):
        P.ransac_relpose_batch_mt(x1[:threads], x2[:threads], opts[:threads], me[:threads], threads)
    t_tot, hyp, cor, smp = 0.0, 0, 0, 0
    for _ in range(args.steps):
        sec, _, stats, cnts = P.ransac_relpose_batch_mt(x1, x2, opts, me, threads)
        t_tot += sec
        hyp += sum(c["hypotheses"] for c in cnts)
        cor += sum(c["scored_corrs"] for c in cnts)
        smp += sum(c["samples"] for c in cnts)
    val = hyp / t_tot
    try:  # SURVEY §8d: the -march=native build of the same port beside the reference-flags build (built on this box)
        nsec, _, nstats, ncnts = P.ransac_relpose_batch_mt(x1, x2, opts, me, threads, native=True)
        same = sum(int(a["iterations"] == b["iterations"] and a["num_inliers"] == b["num_inliers"]) for a, b in zip(nstats, stats))
        native = {"value": sum(c["hypotheses"] for c in ncnts) / nsec, "unit": "hypotheses/s", "cores": threads,
                  "kind": "port", "flags": "g++ -O3 -march=native -ffp-contract=off",
                  "same_trajectory_as_reference_flags_build": f"{same}/{len(x1)}"}
    except Exception as e:
        native = {"unavailable": f"{type(e).__name__}: {e}"}
    try:
        ref_src = reference_sources_leg(P, x1, x2, opts, me, threads, stats, cnts)
    except Exception as e:  # informational leg only: never let it take the arm's line down
        ref_src = {"unavailable": f"{type(e).__name__}: {e}"}
    line = {
        "impl": "reference", "metric": "RANSAC hypotheses/sec (5pt E, 10k corrs)", "value": val, "unit": "hypotheses/s",
        "scored_corrs_per_s": cor / t_tot, "samples_per_s": smp / t_tot, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{pairs} x relpose_5pt C2 (10000 corrs, 30% inliers, max 100000 its), one problem per host thread",
                   "pairs_per_step": pairs},
        "cpu_baseline": {"value": val, "unit": "hypotheses/s", "cores": threads, "host_cpus": os.cpu_count(), "cpu_model": cpu_model(), "kind": "port",
                         "sample": f"{pairs} C2 problems per step x {args.steps} steps; restated PoseLib path (no Eigen), "
                                   "g++ -O3 -ffp-contract=off"},
        "e2e": {"value": val, "unit": "hypotheses/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    line["cpu_baseline_native"] = native
    if ref_src:
        line["reference_sources"] = ref_src
    print(json.dumps(line))


def reference_sources_leg(P, x1, x2, opts, me, threads, stats, cnts):
    """Informational: the reference's OWN sources (oracle/_ref/libplref2.so: robust/ransac.cc, estimators, solvers,
    scorers, bundle, compiled unmodified on mini-Eigen) on the same problems, one problem per thread.  That build pays for
    mini-Eigen's heap temporaries and bounds checks, so it is slower than the reference with real Eigen would be; the
    arm's `value` therefore stays the faster oracle port and this number is reported beside it, not instead of it."""
    if not P.ref2_available(build_if_possible=False):
        return None
    from concurrent.futures import ThreadPoolExecutor
    with P.reference_sources():
        P.ransac("relpose", x1[0], x2[0], opts[0], me[0])  # load + warm
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=threads) as ex:  # ctypes releases the GIL inside the call
            out = list(ex.map(lambda i: P.ransac("relpose", x1[i], x2[i], opts[i], me[i])["stats"], range(len(x1))))
        sec = time.perf_counter() - t0
    same = sum(int(o["iterations"] == s["iterations"] and o["num_inliers"] == s["num_inliers"]) for o, s in zip(out, stats))
    hyp = sum(c["hypotheses"] for c in cnts)  # same trajectory => same hypotheses; counted by the oracle run
    return {"value": hyp / sec, "unit": "hypotheses/s", "cores": threads, "kind": "reference",
            "problems": len(x1), "same_trajectory_as_port": f"{same}/{len(x1)}",
            "note": "PoseLib sources unmodified on mini-Eigen (no Eigen3 in this image); slower than a real-Eigen build"}


# ---- the other BASELINE.json configs, single calls, config 5 ----------------------------------------------------
def config_batches(cabi, rank, quick):
    """Batches of BASELINE configs 1, 3 and 4 for plb_ransac_batch (ransac_* level, calibrated points), own data per rank."""
    F = G.FOCAL
    n1, n3, n4d, n4s = (256, 4, 2, 2) if quick else (1024, 16, 8, 4)
    out = {}
    probs = []
    for i in range(n1):
        p = G.config_c1(rank * n1 + i)
        probs.append(dict(kind="pnp", a=pin(p["x"] / F), b=pin(p["X"]), ransac=cabi.RansacOpt(seed=i, **p["ransac"]), max_error=12.0 / F))
    out["c1"] = dict(problems=probs, n=200, bytes_per_corr=20, what=f"{n1} x p3p absolute pose C1 (200 corrs, 50% inliers, 1000 its)")
    probs = []
    for i in range(n3):
        p = G.config_c3(rank * n3 + i)
        probs.append(dict(kind="fundamental", a=pin(p["x1"] / F), b=pin(p["x2"] / F), ransac=cabi.RansacOpt(seed=i, **p["ransac"]),
                          max_error=1.0 / F, rfc=True))
    out["c3"] = dict(problems=probs, n=5000, bytes_per_corr=16,
                     what=f"{n3} x relpose_7pt fundamental C3 (5000 corrs, 20% inliers, PROSAC, real_focal_check, max 100000 its)")
    probs = []
    for d in range(n4d):  # the plane generator is slow on the host: n4d data sets x n4s RANSAC seeds
        p = G.config_c4(rank * n4d + d)
        a4, b4 = pin(p["x1"] / F), pin(p["x2"] / F)
        for sd in range(n4s):
            probs.append(dict(kind="homography", a=a4, b=b4, ransac=cabi.RansacOpt(seed=sd, **p["ransac"]),
                              max_error=1.0 / F))
    out["c4"] = dict(problems=probs, n=20000, bytes_per_corr=16,
                     what=f"{n4d * n4s} x homography_4pt C4 (20000 corrs, 60% inliers, LO refit TRUNCATED; {n4d} data sets x {n4s} seeds)")
    return out


def run_config(cabi, torch, flush, cfg, streams, steps):
    """Timed passes of one config batch through plb_ransac_batch (host buffers) + one single-group pass for the kernel
    shares (CUDA-event durations are not inflated by kernels of other groups when only one group is in flight)."""
    batch = cabi.Batch(cfg["problems"])
    batch.run(streams=streams)  # buffers
    t_tot, agg = 0.0, None
    for _ in range(steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        batch.run(streams=streams)
        torch.cuda.synchronize()
        t_tot += time.perf_counter() - t0
        c = batch.counter_sums()
        agg = c if agg is None else {k: agg[k] + c[k] for k in c}
    batch.run(streams=1)
    flush.zero_()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    batch.run(streams=1)
    torch.cuda.synchronize()
    t1 = time.perf_counter() - t0
    return t_tot, agg, t1, batch.counter_sums()


def single_calls(cabi, reps=7):
    """Latency of ONE plb_estimate_* call (pixels in, model + inlier mask out, final bundle included) on one problem of
    each BASELINE config 1-4: median of `reps` calls after two warm-up calls."""
    F = G.FOCAL
    cam = cabi.Camera("PINHOLE", (F, F, 0.0, 0.0))
    bo = cabi.BundleOpt()
    out = {}
    cases = []
    p = G.config_c1(0)
    cases.append(("c1", "pnp", p["x"], p["X"], p, dict(cam1=cam), 12.0))
    p = G.config_c2(0)
    cases.append(("c2", "relpose", p["x1"], p["x2"], p, dict(cam1=cam, cam2=cam), 1.0))
    p = G.config_c3(0)
    cases.append(("c3", "fundamental", p["x1"], p["x2"], p, dict(rfc=True), 1.0))
    p = G.config_c4(0)
    cases.append(("c4", "homography", p["x1"], p["x2"], p, dict(), 1.0))
    for name, kind, a, b, p, kw, me in cases:
        ro = cabi.RansacOpt(**p["ransac"])
        ts, last = [], None
        for i in range(reps + 2):
            t0 = time.perf_counter()
            last = cabi.estimate(kind, a, b, ro, bo, me, **kw)
            dt = time.perf_counter() - t0
            if i >= 2:
                ts.append(dt)
        ts.sort()
        c = last["counters"]
        out[name] = {"entry": "plb_estimate_" + {"pnp": "absolute_pose", "relpose": "relative_pose", "fundamental": "fundamental",
                                                  "homography": "homography"}[kind],
                     "ms": 1e3 * ts[len(ts) // 2], "ms_min": 1e3 * ts[0], "iterations": last["stats"]["iterations"],
                     "hypotheses": c["hypotheses"], "rounds": c["rounds"], "gpu_launches": c["gpu_launches"],
                     "h2d_bytes": c["h2d_bytes"], "d2h_bytes": c["d2h_bytes"]}
    return out


def c5_costs(count):
    from poselib_b200 import sharding
    return [sharding.expected_cost("pnp", 200, 1000) if i % 2 == 0 else sharding.expected_cost("relpose", 10000, 100000)
            for i in range(count)]


def c5_problems(cabi, indices):
    F = G.FOCAL
    probs = []
    for i in indices:
        i = int(i)
        if i % 2 == 0:
            p = G.abspose_problem(200, 0.5, 5, i)
            probs.append(dict(kind="pnp", a=pin(p["x"] / F), b=pin(p["X"]), ransac=cabi.RansacOpt(max_iterations=1000, min_iterations=1000),
                              max_error=12.0 / F))
        else:
            p = G.relpose_problem(10000, 0.3, 5, i)
            probs.append(dict(kind="relpose", a=pin(p["x1"] / F), b=pin(p["x2"] / F),
                              ransac=cabi.RansacOpt(max_iterations=100000, min_iterations=1000), max_error=1.0 / F))
    return probs


DUMP_BUDGET = 64 << 20  # bytes of .npy data that --dump-outputs may write in all


def dump_outputs(out_dir, passes):
    """What a caller of the timed path receives, per problem of the last timed step: model, inlier mask and RANSAC stats of
    every pass, as DIR/<pass>_<field>.npy (float64; the masks as float32 0/1).  When the masks of all problems would exceed
    DUMP_BUDGET, a fixed, seeded sample of the problems is written; <pass>_index.npy holds the problem indices written."""
    os.makedirs(out_dir, exist_ok=True)
    count = len(next(iter(passes.values())))
    per_problem = sum(4 * len(r[0]["inliers"]) + 8 * (len(r[0]["model"].ravel()) + len(r[0]["stats"]) + 1)
                      for r in passes.values())
    keep = min(count, (DUMP_BUDGET - (1 << 16)) // per_problem)  # 64 KiB left for the .npy headers
    index = np.arange(count) if keep == count else np.sort(np.random.default_rng(0).choice(count, keep, replace=False))
    for name, results in passes.items():
        rows = [results[i] for i in index]
        arrays = {"index": index.astype(np.float64),
                  "model": np.stack([np.asarray(r["model"], dtype=np.float64) for r in rows]),
                  "inliers": np.stack([np.asarray(r["inliers"], dtype=np.float32) for r in rows])}
        for key in rows[0]["stats"]:
            arrays["stats_" + key] = np.array([r["stats"][key] for r in rows], dtype=np.float64)
        for field, a in arrays.items():
            np.save(os.path.join(out_dir, f"{name}_{field}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--pairs", type=int, default=256, help="independent C2 image pairs per GPU per step")
    ap.add_argument("--streams", type=int, default=8, help="lock-step problem groups in flight per GPU")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="fast", choices=["exact", "fast"],
                    help="fast (the library default): fp32 SMEM screening of every model with rigorous error intervals + "
                         "fp64 confirmation of candidates (identical results)")
    ap.add_argument("--no-extras", action="store_true",
                    help="headline only: skip the configs 1/3/4 batches, the single calls and the config-5 strong-scaling pass")
    ap.add_argument("--c5", type=int, default=4096, help="problems of the config-5 batch (sharded over the ranks)")
    ap.add_argument("--quick", action="store_true", help="small extras (smoke test of the bench itself)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step of the headline (resident) and e2e passes as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    # ranks of one node share the host cores: tell the engine its share (helper threads for the sample tables)
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    os.environ.setdefault("PLB_HOST_THREADS", str(max(1, usable_cores() // max(1, local_world))))
    from poselib_b200 import cabi
    if not torch.cuda.is_available() or cabi.device_count() == 0:
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    cabi.set_device(local_rank)
    global _PIN
    _PIN = True
    cabi.set_mode(args.mode)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    pairs = args.pairs
    batch = make_batch(pairs, rank * pairs)  # every rank gets its own image pairs (weak scaling)
    n = len(batch[0][0])
    ropt = dict(max_iterations=100000, min_iterations=1000, seed=0)
    host_probs = [dict(kind="relpose", a=a, b=b, ransac=cabi.RansacOpt(**ropt), max_error=1.0 / G.FOCAL) for a, b in batch]
    handles = [cabi.resident_create("relpose", a, b) for a, b in batch]
    res_probs = [dict(kind="relpose", resident=h, n=n, ransac=cabi.RansacOpt(**ropt), max_error=1.0 / G.FOCAL)
                 for h in handles]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    from poselib_b200 import sharding
    my_idx = list(range(rank * pairs, (rank + 1) * pairs))

    # The batches are marshalled into the C-ABI's plb_problem arrays ONCE (cabi.Batch); a timed step is the C call itself
    # — plb_ransac_batch with its host->device copies, kernels, device->host results — not Python building structs.
    def timed(batch, steps, gather=False):
        t_tot, agg = 0.0, None
        for _ in range(steps):
            flush.zero_()  # L2 flush between timed iterations (untimed)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            batch.run(streams=args.streams)  # returns after its own stream syncs
            if gather and dist is not None:
                # the only inter-GPU traffic of the path: fixed-size result records gathered over NCCL (SURVEY §8e)
                sharding.gather_records_equal(batch.records(my_idx), dist)
            torch.cuda.synchronize()
            t_tot += time.perf_counter() - t0
            c = batch.counter_sums()
            agg = c if agg is None else {k: agg[k] + c[k] for k in c}
        return t_tot, agg, batch.results()

    res_probs, host_probs = cabi.Batch(res_probs), cabi.Batch(host_probs)
    for _ in range(args.warmup):
        res_probs.run(streams=args.streams)
        host_probs.run(streams=args.streams)
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    t_res, c_res, last_value = timed(res_probs, args.steps)
    barrier()
    t_e2e, c_e2e, last = timed(host_probs, args.steps, gather=True)
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"resident": last_value, "e2e": last})
    # roofline pass: the same workload with ONE lock-step group in flight, so that the CUDA-event duration of the scoring
    # kernel is not inflated by kernels of other groups sharing the GPU (still live, still on the engine's stream)
    streams_saved = args.streams
    args.streams = 1
    t_roof, c_roof, _ = timed(res_probs, max(3, args.steps // 2))
    args.streams = streams_saved
    barrier()
    # cross-check pass: the same resident batch in the OTHER precision mode (fp64 scoring of every model when the headline
    # ran with fp32 screening, and vice versa).  Reported beside the headline together with whether every result
    # (stats, model bits, inlier mask) is identical.  No collective inside the try block: a failure here must not be
    # able to desynchronise the ranks or lose the headline line.
    other_mode = "exact" if args.mode == "fast" else "fast"
    t_other, hyp_other, steps_other, same_other = float("nan"), 0.0, max(2, args.steps // 3), 0.0
    try:
        cabi.set_mode(other_mode)
        res_probs.run(streams=args.streams)  # buffers of the other mode
        t_other, c_other, last_other = timed(res_probs, steps_other)
        hyp_other = float(c_other["hypotheses"])
        same_other = float(all(a["stats"] == b["stats"] and np.array_equal(a["model"], b["model"]) and
                               np.array_equal(a["inliers"], b["inliers"]) for a, b in zip(last_value, last_other)))
    except Exception as e:  # noqa: BLE001
        sys.stderr.write(f"[bench] cross-check pass failed: {e}\n")
    finally:
        cabi.set_mode(args.mode)
    barrier()
    sampler.stop_flag = True

    def allmax(v):
        if dist is None:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(v):
        if dist is None:
            return v
        t = torch.tensor([float(v)], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- extras: BASELINE configs 1, 3, 4 (batched), single calls, config 5 (strong scaling over the ranks) -------------
    # Local work sits in try blocks; the collectives that aggregate it run unconditionally on every rank afterwards.
    extras = {}
    if not args.no_extras:
        peak_x, _ = load_peaks()
        try:
            batches = config_batches(cabi, rank, args.quick)
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"[bench] config batches failed: {e}\n")
            batches = {}
        cfg_out = {}
        for name in ("c1", "c3", "c4"):
            loc = dict(t=1e30, hyp=0.0, cor=0.0, t1=0.0, k=None, problems=0)
            try:
                cfg = batches[name]
                t_tot, agg, t1, k = run_config(cabi, torch, flush, cfg, args.streams, 2 if args.quick else 3)
                loc = dict(t=t_tot, hyp=float(agg["hypotheses"]), cor=float(agg["scored_corrs"]), t1=t1, k=k,
                           problems=len(cfg["problems"]))
            except Exception as e:  # noqa: BLE001
                sys.stderr.write(f"[bench] config {name} failed: {e}\n")
            T = allmax(loc["t"])
            H, Cr, NPb = allsum(loc["hyp"]), allsum(loc["cor"]), allsum(loc["problems"])
            if rank == 0 and loc["k"] is not None and T < 1e29:
                k, cfg, st = loc["k"], batches[name], (2 if args.quick else 3)
                score_s = k["gpu_seconds_score"]
                ach = k["models_evaluated"] * cfg["n"] * cfg["bytes_per_corr"] / score_s / 1e9 if score_s > 0 else 0.0
                cfg_out[name] = {
                    "workload": cfg["what"] + " per GPU per step", "problems_per_step": int(NPb), "value": H / T,
                    "unit": "hypotheses/s", "scored_corrs_per_s": Cr / T, "ms_per_step": 1e3 * T / st,
                    "kernels_single_group_pass": {
                        "wall_s": loc["t1"], "solve_s": k["gpu_seconds"] - k["gpu_seconds_score"] - k["gpu_seconds_select"],
                        "score_s": score_s, "select_confirm_s": k["gpu_seconds_select"], "lo_s": k["gpu_seconds_lo"],
                        "rounds": int(k["rounds"]), "launches": int(k["gpu_launches"])},
                    "roofline": {"bound": "hbm", "kernel": "k_screen (fp32 MSAC screening)", "achieved": ach, "peak": peak_x,
                                 "unit": "GB/s", "frac": ach / peak_x, "bytes_per_scored_corr": cfg["bytes_per_corr"]}}
        extras["configs"] = cfg_out
        if rank == 0:
            try:
                extras["single_call"] = single_calls(cabi, 3 if args.quick else 7)
            except Exception as e:  # noqa: BLE001
                extras["single_call"] = {"failed": str(e)}
        barrier()
        # config 5: `--c5` independent problems (even index: C1-type p3p, odd: C2-type 5pt), LPT-partitioned over the
        # ranks, results (records + inlier masks) gathered on every rank: STRONG scaling, total work fixed
        loc5 = dict(t=1e30, hyp=0.0, cor=0.0, n=0, ok=1.0)
        c5_count = 64 if args.quick else args.c5
        try:
            part = sharding.partition(c5_costs(c5_count), world)[rank]
            p5 = cabi.Batch(c5_problems(cabi, part))
            p5.run(streams=args.streams)
        except Exception as e:  # noqa: BLE001
            sys.stderr.write(f"[bench] config 5 setup failed: {e}\n")
            p5, part, loc5["ok"] = None, [], 0.0
        c5_steps = 2
        barrier()
        t5, hyp5, cor5, gathered = 0.0, 0.0, 0.0, 0
        for _ in range(c5_steps):
            flush.zero_()
            barrier()
            t0 = time.perf_counter()
            if p5 is not None:
                p5.run(streams=args.streams)
                cs5 = p5.counter_sums()
                hyp5 += cs5["hypotheses"]
                cor5 += cs5["scored_corrs"]
            if dist is not None:  # the only inter-GPU traffic: fixed-size records + bit-packed masks over NCCL
                rec = sharding.gather_records(p5.records([int(i) for i in part]) if p5 is not None else np.zeros((0, 14)), dist)
                gathered = len(rec)
                sharding.gather_masks([k[2] for k in p5.keep] if p5 is not None else [], [int(i) for i in part], dist)
            else:
                gathered = p5.count if p5 is not None else 0
            torch.cuda.synchronize()
            t5 += time.perf_counter() - t0
        T5 = allmax(t5 if loc5["ok"] else 1e30)
        H5, C5 = allsum(hyp5), allsum(cor5)
        if rank == 0 and T5 < 1e29:
            extras["c5"] = {"workload": f"{c5_count} independent problems (even: p3p C1-type, odd: 5pt C2-type), own data seeds, "
                                        f"LPT-sharded over {world} rank(s); records and inlier masks gathered",
                            "scaling": "strong", "problems": c5_count, "seconds_per_pass": T5 / c5_steps,
                            "problems_per_s": c5_count * c5_steps / T5, "value": H5 / T5, "unit": "hypotheses/s",
                            "scored_corrs_per_s": C5 / T5, "records_gathered": int(gathered)}
        barrier()

    T_res, T_e2e = allmax(t_res), allmax(t_e2e)
    T_other = allmax(t_other if t_other == t_other else 1e30)
    hyp_o = allsum(hyp_other)
    same_o = allsum(same_other)
    hyp, cor, smp = allsum(c_res["hypotheses"]), allsum(c_res["scored_corrs"]), allsum(c_res["samples"])
    hyp_e, cor_e = allsum(c_e2e["hypotheses"]), allsum(c_e2e["scored_corrs"])
    launches = allsum(c_res["gpu_launches"])
    if rank == 0:
        peak, peak_kind = load_peaks()
        # roofline of the scoring kernel (the streaming map-reduce of SURVEY §8d):
        #   fast mode : k_screen  — fp32 SoA, 16 B / scored correspondence, staged in shared memory by TMA
        #   exact mode: k_score_tiled — fp64 SoA, 32 B / scored correspondence
        # algorithmic bytes = models scored x N x bytes/corr ; duration = CUDA events around the scoring launches on
        # the engine's stream.  The 5-point solver kernels (latency/issue bound, no streaming) are timed beside it.
        bpc = 16 if args.mode == "fast" else BYTES_PER_CORR_FP64
        roof_steps = max(3, args.steps // 2)
        alg_bytes = c_roof["models_evaluated"] * n * bpc
        k_sec = c_roof["gpu_seconds_score"]
        k_sec_all = c_roof["gpu_seconds"]
        ach = alg_bytes / k_sec / 1e9 if k_sec > 0 else 0.0
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic_scoring_kernel.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(args.mode, {}).get("dram_bytes_per_launch")
        # The §8d yardstick is an HBM-read roofline, but the kernel does not stream from HBM: operands are staged once per
        # CTA into shared memory by TMA and reused by every model.  What actually binds it is the instruction issue rate:
        # thread-instructions per (model, correspondence) pair from the committed ncu capture x pairs/s vs the SM issue
        # peak at the measured clock.
        binding = None
        try:
            prof = json.load(open(os.path.join(ROOT, "profiles", "issue_model.json")))[args.mode]
            pairs_per_s = c_roof["models_evaluated"] * n / k_sec if k_sec > 0 else 0.0
            clk = (sampler.summary().get("sm_mhz") or 1965.0) * 1e6
            peak_issue = 148 * 4 * 32 * clk  # thread-instructions/s: 4 warp-instructions per clock per SM
            binding = {"resource": "instruction issue (fp32 FMA + compare/record per pair), not HBM",
                       "thread_instr_per_pair": prof["thread_instr_per_pair"], "source": prof["source"],
                       "pairs_per_s": pairs_per_s, "achieved_thread_instr_per_s": pairs_per_s * prof["thread_instr_per_pair"],
                       "peak_thread_instr_per_s": peak_issue,
                       "frac_of_issue_peak": pairs_per_s * prof["thread_instr_per_pair"] / peak_issue,
                       "whole_step_hbm_frac": (c_res["models_evaluated"] * n * bpc / T_res / 1e9) / peak}
        except Exception as e:  # noqa: BLE001
            binding = {"resource": "instruction issue, not HBM", "unavailable": str(e)}
        line = {
            "metric": "RANSAC hypotheses/sec (5pt E, 10k corrs)", "value": hyp / T_res, "unit": "hypotheses/s",
            "scored_corrs_per_s": cor / T_res, "samples_per_s": smp / T_res,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * T_res / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64" if args.mode == "exact" else "f64 (fp32 screening of all models, fp64 confirmation + solvers + LO)",
            "data": "synthetic",
            "config": {"workload": f"{pairs} x relpose_5pt C2 (10000 corrs, 30% inliers, max 100000 its) per GPU per step",
                       "pairs_per_step_per_gpu": pairs, "streams": args.streams, "mode": args.mode,
                       "l2": "flushed (256 MiB write) between timed steps", "timing": "host clock around synchronous "
                       "C-ABI calls, cuda synchronize both sides, max over ranks; kernel time by CUDA events"},
            "e2e": {"value": hyp_e / T_e2e, "unit": "hypotheses/s", "scored_corrs_per_s": cor_e / T_e2e,
                    "includes": "page-locked host buffers in (DMA straight from the caller's arrays), results out to host memory" + ("; NCCL all_gather of the result records" if world > 1 else ""),
                    "ms_per_step": 1e3 * T_e2e / args.steps,
                    "h2d_bytes_per_step": c_e2e["h2d_bytes"] // args.steps, "d2h_bytes_per_step": c_e2e["d2h_bytes"] // args.steps},
            "gpu_launches": int(launches),
            "other_mode": {"mode": other_mode, "value": (hyp_o / T_other) if T_other < 1e29 else None,
                           "unit": "hypotheses/s", "steps": steps_other,
                           "ms_per_step": (1e3 * T_other / steps_other) if T_other < 1e29 else None,
                           "results_identical_to_headline_mode": bool(same_o == world),
                           "note": "same resident batch; stats, model bits and inlier masks compared problem by problem"},
            "roofline": {"bound": "hbm", "binding": binding, "kernel": "k_screen<relpose> (fp32 MSAC screening, TMA-staged SMEM)" if args.mode == "fast"
                         else "k_score_tiled<relpose> (fp64 MSAC scoring)", "achieved": ach,
                         "peak": peak, "peak_kind": peak_kind, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                         "bytes_per_scored_corr": bpc,
                         "algorithmic_bytes_per_step": alg_bytes / roof_steps, "kernel_seconds_per_step": k_sec / roof_steps,
                         "solver_kernels_seconds_per_step": (k_sec_all - k_sec - c_roof["gpu_seconds_select"]) / roof_steps,
                         "select_confirm_seconds_per_step": c_roof["gpu_seconds_select"] / roof_steps,
                         "lo_seconds_per_step": c_roof["gpu_seconds_lo"] / roof_steps,
                         "kernel_share_of_step": k_sec / t_roof if t_roof > 0 else None,
                         "measured": f"{roof_steps} extra steps of the same workload with one lock-step group in flight "
                                     "(kernel durations by CUDA events on the engine's stream, no co-running kernels)",
                         "note": "correspondences are SMEM/L2-resident and reused across thousands of models: DRAM "
                                 "traffic << algorithmic bytes by design (SURVEY H7); frac is the SURVEY §8d figure and "
                                 "can exceed 1 for the fp32 screening kernel: its operand stream is served from shared "
                                 "memory after one TMA stage per CTA, the binding resource is fp32 issue (60 % of the "
                                 "slots, profiles/r01_v7_summary.md)"},
            "clocks": sampler.summary(),
        }
        line.update(extras)
        # CPU baseline on this box's host cores: 1 thread (the reference's execution model), bounded sample
        try:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import plo_py as P
            k = min(8, pairs)
            sec, _, _, cnts = P.ransac_relpose_batch_mt([b[0] for b in batch[:k]], [b[1] for b in batch[:k]],
                                                         [P.RansacOpt(**ropt) for _ in range(k)], [1.0 / G.FOCAL] * k, 1)
            line["cpu_baseline"] = {"value": sum(c["hypotheses"] for c in cnts) / sec, "unit": "hypotheses/s",
                                    "scored_corrs_per_s": sum(c["scored_corrs"] for c in cnts) / sec, "cores": 1,
                                    "kind": "port", "sample": f"first {k} problems of the step, 1 thread, restated "
                                    "PoseLib path (no Eigen), g++ -O3 -ffp-contract=off", "seconds": sec,
                                    "host_cpus": os.cpu_count(), "usable_cores": usable_cores(), "cpu_model": cpu_model()}
        except Exception as e:  # the baseline is a reported number, never part of the product path
            line["cpu_baseline"] = {"value": None, "unit": "hypotheses/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line))
    for h in handles:
        cabi.resident_free(h)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

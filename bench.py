#!/usr/bin/env python
"""bench.py — headline benchmark of the GP-surrogate + acquisition hot path.

metric (BASELINE.json): candidate posterior+EI evaluations / second at n = 8192 observations,
d = 20 (config C4 of SURVEY §8d: SE kernel, l = 1, sigma^2 = 1, noise 1e-2, 2,097,152 candidates
per GPU = 16 M over 8 GPUs).  A "step" is one BO iteration's worth of the hot path: rank 0 conditions
the surrogate on one more observation (copy-on-write snapshot + O(n^2) row append, n - 1 -> n), the posterior
(lower tiles of L and L^-1, X, alpha) is broadcast to the other ranks over NCCL / NVLink (abo_gp_sync), every
rank sweeps its candidate shard with the fused kernel (K* tiles -> L^-1 K* on the FP64 tensor pipe -> mean,
variance -> EI -> scores) and selects its stable top-100 on the device, and the per-rank lists are merged into
the global top-100 with abo_topk_allgather.  `iteration_ms` breaks the step down.

  value : candidates/s, whole job (all ranks), candidates already resident in HBM
  e2e   : the same through the host-buffer C-ABI call abo_acq_eval (pinned host candidates,
          H2D copy, sweep, D2H of the scores, top-k) — copies inside the timed region
  roofline : the dominant kernel (DMMA triangular product + sum of squares), algorithmic
          n^2 flop per candidate / its CUDA-event duration, against the measured FP64 GEMM peak
  cholesky : second BASELINE metric — blocked FP64 Cholesky TFLOP/s at n = 8192
  cpu_baseline : the CPU restatement (oracle, NumPy/SciPy on OpenBLAS, all host cores) on a
          bounded sample of the same workload (the Julia reference cannot run here: no Julia)

`--impl reference` times that CPU restatement as the reference arm.
`--dump-outputs DIR` writes the scores and the top-k of the last timed step as .npy files; the inputs are seeded, so
two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

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

N_OBS, DIM = 8192, 20
M_PER_GPU = 2_097_152
TOPK = 100
DUMP_BYTES = 60_000_000          # --dump-outputs stays under 64 MB in all, whatever the candidate count and world size
METRIC = "candidate posterior+EI evals/sec at n=8192,d=20"
UNIT = "candidates/s"


def flops_per_candidate(n, d):
    return float(n) * n + 3.0 * n * d + 4.0 * n          # SURVEY §8(d)


def fp64_peak():
    """FP64 roofline denominator.  MEASURED_PEAKS.json (driver-written) has no FP64 row, so the
    denominator is this repo's own measurement on the same pool: cuBLAS Dgemm NT 8192^3
    (tools/fp64_peaks.cu -> profiles/fp64_peaks_r01.json)."""
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        if "fp64_tflops" in mp:
            return float(mp["fp64_tflops"]), "MEASURED_PEAKS.json fp64_tflops"
    except Exception:
        pass
    try:
        pk = json.load(open(os.path.join(ROOT, "profiles", "fp64_peaks_r01.json")))
        return float(pk["cublas_dgemm_nt_tflops"]["8192"]), \
            "cuBLAS Dgemm NT 8192^3 measured on this pool (profiles/fp64_peaks_r01.json); MEASURED_PEAKS.json has no FP64 row"
    except Exception:
        return 37.0, "nominal B200 FP64 (no measurement file found)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.device)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def use_all_host_cores(limit=None):
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs are meant to use every host core (or `limit`).
    Returns the thread count the BLAS pools actually run with (threadpoolctl), not os.cpu_count()."""
    try:
        from threadpoolctl import threadpool_info, threadpool_limits
        threadpool_limits(limits=limit or (os.cpu_count() or 1))
        info = [i for i in threadpool_info() if i.get("user_api") == "blas"]
        return max([int(i.get("num_threads", 1)) for i in info] or [1]), \
            "; ".join(sorted({f"{i.get('internal_api')} {i.get('version')}" for i in info})) or "unknown"
    except Exception:
        return (limit or os.cpu_count() or 1), "threadpoolctl unavailable"


def cpu_restatement_throughput(sample_m, seed=42, n=N_OBS):
    """Oracle (CPU restatement of the reference path) on a bounded sample of the C4 workload:
    conditioning is untimed set-up, the timed part is posterior mean + variance + EI over
    `sample_m` candidates (best of 2 after one warm-up) with all host cores, and once more with ONE thread on
    a quarter of the sample (SURVEY 8d asks for both)."""
    from oracle import abo_oracle as orc
    threads, blas = use_all_host_cores()
    c = orc.make_config("C4", seed=seed, n=n, m=sample_m, d=DIM)
    t0 = time.perf_counter()
    post = orc.fit_standard(c["X"], c["y"], c["kind"], c["inv_ls"], c["scale"], c["noise"])
    t_fit = time.perf_counter() - t0
    best = float(c["y"].min())

    def one(Xc):
        mu, var = orc.posterior_mean_var(post, Xc, chunk=2048)
        ei = orc.expected_improvement(mu, var, 0.01, best)
        orc.sortperm_rev(ei, TOPK)
    times = []
    for it in range(3):
        t0 = time.perf_counter(); one(c["Xc"]); times.append(time.perf_counter() - t0)
    t = min(times[1:])
    use_all_host_cores(1)
    m1 = max(256, sample_m // 4)
    t0 = time.perf_counter(); one(c["Xc"][:m1]); t1 = time.perf_counter() - t0
    use_all_host_cores()
    return {"value": sample_m / t, "t_step": t, "t_fit": t_fit, "threads": threads, "blas": blas,
            "one_thread_value": m1 / t1, "one_thread_sample": m1}


def workload_config(n, d, m, world):
    """The `config` object of BOTH arms (the reference arm evaluates a bounded sample of the same workload)."""
    return {"workload": f"C4: StandardGP SE n={n} d={d} noise=1e-2; one BO iteration = observation n-1 -> n appended, posterior "
                        f"broadcast, EI(xi=0.01) over {m} candidates per GPU ({world * m} total), global stable top-{TOPK}; "
                        f"candidate set ({m * d * 8 / 1e6:.0f} MB per GPU) and the K* tiles exceed L2, no explicit flush",
            "n": n, "d": d, "candidates_per_gpu": m, "l2": "inputs larger than L2"}


def dump_outputs(out_dir, scores, top_idx, top_val, rank, world):
    """What the last timed step handed its caller, as .npy files for comparing two builds output for output: the
    global top-k (indices as float64, exact below 2^53) and this rank's candidate scores.  Scores that would exceed
    the size budget are replaced by a fixed, seeded sample, and the sampled candidate indices are written beside them."""
    os.makedirs(out_dir, exist_ok=True)
    tag = "" if world == 1 else f"_rank{rank}"
    if rank == 0:
        np.save(os.path.join(out_dir, "topk_index.npy"), np.asarray(top_idx, dtype=np.float64))
        np.save(os.path.join(out_dir, "topk_value.npy"), np.asarray(top_val, dtype=np.float64))
    cap = DUMP_BYTES // world // 16                 # float64 score + float64 index per sampled candidate
    if len(scores) > 2 * cap:
        idx = np.sort(np.random.default_rng(0).choice(len(scores), cap, replace=False))
        np.save(os.path.join(out_dir, f"scores_index{tag}.npy"), idx.astype(np.float64))
        scores = scores[idx]
    np.save(os.path.join(out_dir, f"scores{tag}.npy"), np.asarray(scores, dtype=np.float64))


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path.  The reference is Julia
    and cannot run in this image (no Julia toolchain, no network); the timed stand-in is the CPU
    restatement in oracle/ (NumPy/SciPy on OpenBLAS with all host cores), kind = "port"."""
    if rank != 0:
        return
    sample = args.cpu_sample
    from oracle import abo_oracle as orc
    cores, blas = use_all_host_cores()
    c = orc.make_config("C4", n=args.n, m=sample, d=DIM)
    post = orc.fit_standard(c["X"], c["y"], c["kind"], c["inv_ls"], c["scale"], c["noise"])
    best = float(c["y"].min())

    def step():
        mu, var = orc.posterior_mean_var(post, c["Xc"], chunk=2048)
        ei = orc.expected_improvement(mu, var, 0.01, best)
        orc.sortperm_rev(ei, TOPK)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    v = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.n, DIM, args.m, args.gpus),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "blas": blas,
                         "sample": f"each step a bounded sample of {sample} candidates of that workload (same n, d, kernel, "
                                   "EI + stable top-100), oracle/abo_oracle.py on NumPy/SciPy; the conditioning step is "
                                   "un-timed set-up; the Julia reference cannot run in this image"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cands", dest="m", type=int, default=M_PER_GPU, help="candidates per GPU per step")
    ap.add_argument("--n", type=int, default=N_OBS)
    ap.add_argument("--cpu-sample", type=int, default=8192)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cholesky", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the scores and the top-k of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import abo_b200 as abo
    from oracle import abo_oracle as orc            # data generators + cpu_baseline leg only

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    ctx = abo.default_context(local_rank)
    n, d, m = args.n, DIM, args.m

    # ---- conditioning set (seeded, identical on every rank).  Rank 0 holds the posterior on the first n - 1
    # observations; every step it conditions on the n-th one (copy-on-write snapshot + O(n^2) row append — the BO
    # loop's update(BO, x, y), src/bayesian_opt.jl:113-150, without the reference's O(n^3) re-fit) and the other ranks
    # receive the new posterior over NCCL.
    c = orc.make_config("C4", n=n, m=1, d=d)
    kern = c["scale"] * abo.with_lengthscale(abo.SqExponentialKernel(), 1.0 / c["inv_ls"])
    t0 = time.perf_counter()
    base = abo.update(abo.StandardGP(kern, c["noise"], ctx=ctx), c["X"][:-1], c["y"][:-1]) if rank == 0 else None
    t_fit = time.perf_counter() - t0
    if world > 1:
        abo.init_nccl_context(ctx)
    recv = abo.empty_posterior_like(abo.StandardGP(kern, c["noise"], ctx=ctx), d) if rank != 0 else None
    acq = abo.ExpectedImprovement(0.01, float(c["y"].min()))
    params = acq.params()
    x_new, y_new = c["X"][-1], c["y"][-1:]

    # ---- candidates: this rank's shard, device-resident for `value`, pinned host copy for e2e
    gen = torch.Generator(device="cuda")
    gen.manual_seed(1234 + rank)
    Xc_dev = torch.rand((m, d), dtype=torch.float64, device="cuda", generator=gen)
    scores_dev = torch.empty(m, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    lib_stream = torch.cuda.ExternalStream(ctx.stream())
    parts = {"append": 0.0, "sync": 0.0, "sweep": 0.0, "topk_allgather": 0.0}

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    local_top = [None]

    def step_dev(timed=False):
        """One BO iteration of the hot path; every call of the library is synchronous, so host timers bracket
        device work (the device-side total is taken with CUDA events around the K steps)."""
        t = [time.perf_counter()]
        if rank == 0:
            h = base.gpx.clone()                      # O(1) snapshot (Base.copy)
            h.append(x_new, y_new)                    # un-share + O(n^2) append: posterior on n observations
        else:
            h = recv.gpx
        t.append(time.perf_counter())
        if world > 1:
            h.sync(0)                                 # NCCL broadcast of the packed lower tiles of L, L^-1 + X, alpha
        t.append(time.perf_counter())
        ti, tv = h.acq_eval_dev(acq.acq_id, params, Xc_dev.data_ptr(), m, scores_dev.data_ptr(), k=TOPK)
        t.append(time.perf_counter())
        local_top[0] = (ti, tv)
        if world > 1:
            ti, tv = ctx.topk_allgather(TOPK, ti + rank * m, tv)      # global indices: rank r owns [r m, (r+1) m)
        t.append(time.perf_counter())
        if timed:
            for key, dt in zip(parts, np.diff(t)):
                parts[key] += dt
        if rank == 0:
            h.close()
        return ti, tv, h

    for _ in range(args.warmup):
        step_dev()
    launches0 = ctx.launch_count()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.perf_counter()
    e0.record(lib_stream)
    for _ in range(args.steps):
        top_idx, top_val, _ = step_dev(timed=True)
    e1.record(lib_stream)
    barrier()
    wall = time.perf_counter() - w0
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, scores_dev.cpu().numpy(), top_idx, top_val, rank, world)
    ms = max(e0.elapsed_time(e1), 0.0)
    launches = ctx.launch_count() - launches0
    # the posterior the sweeps ran on, kept for the e2e leg and the checks below
    if rank == 0:
        model_h = base.gpx.clone(); model_h.append(x_new, y_new)
    else:
        model_h = recv.gpx
    if world > 1:
        model_h.sync(0)
    # one extra, un-timed pass with CUDA-event brackets around the sweep kernel for the roofline of the dominant kernel
    ctx.profile(True)
    model_h.acq_eval_dev(acq.acq_id, params, Xc_dev.data_ptr(), m, scores_dev.data_ptr(), k=TOPK)
    prof_ms, prof_n = ctx.profile_read()
    ctx.profile(False)
    prof_steps = 1
    t = torch.tensor([ms, 1e3 * wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t[0].item())
    value = world * m * args.steps / (ms_max * 1e-3)
    h = model_h

    # ---- cross-rank check (N > 1, outside the timed region): rank 0 re-evaluates every shard by itself and must find
    #      the same global top-100 (indices AND values) as the sharded run
    xrank = None
    if world > 1:
        shard_tops = [None] * world
        dist.all_gather_object(shard_tops, (np.asarray(local_top[0][0]), np.asarray(local_top[0][1])))
        if rank == 0:
            from abo_b200.parallel import merge_topk
            idxs, vals = [], []
            for r in range(world):
                g2 = torch.Generator(device="cuda"); g2.manual_seed(1234 + r)
                Xr = torch.rand((m, d), dtype=torch.float64, device="cuda", generator=g2)
                ti_r, tv_r = h.acq_eval_dev(acq.acq_id, params, Xr.data_ptr(), m, 0, k=TOPK)
                idxs.append(ti_r + r * m); vals.append(tv_r)
                del Xr
            gi, gv = merge_topk(idxs, vals, TOPK)
            same_i = np.array_equal(gi, top_idx); same_v = np.array_equal(gv, top_val)
            shard_ok = [bool(np.array_equal(shard_tops[r][0] + r * m, idxs[r]) and np.array_equal(shard_tops[r][1], vals[r]))
                        for r in range(world)]
            xrank = {"global_top100_equals_single_gpu": bool(same_i and same_v), "per_shard_top100_equal": shard_ok,
                     "argmax_global_index": int(top_idx[0])}
            if not (same_i and same_v):
                nb = min(len(gi), len(top_idx))
                bad = [int(q) for q in np.flatnonzero((gi[:nb] != top_idx[:nb]) | (gv[:nb] != top_val[:nb]))[:5]]
                xrank["first_mismatches"] = [{"pos": q, "sharded": [int(top_idx[q]), float(top_val[q])], "single": [int(gi[q]), float(gv[q])],
                                              "owner_rank_sharded": int(top_idx[q] // m), "owner_rank_single": int(gi[q] // m)} for q in bad]
                xrank["lengths"] = [int(len(top_idx)), int(len(gi))]
        barrier()

    # ---- e2e: host buffers through the C-ABI call, copies inside the timed region
    Xc_host = torch.empty((m, d), dtype=torch.float64, pin_memory=True)
    Xc_host.copy_(Xc_dev)
    Xh = Xc_host.numpy()
    scores_host = torch.empty(m, dtype=torch.float64, pin_memory=True)
    import ctypes as C
    from abo_b200 import _lib
    ti = np.empty(TOPK, dtype=np.int64); tv = np.empty(TOPK)
    pp = _lib.f64(params)

    def step_e2e():
        # the call a user makes: host candidates in, scores + top-k out (H2D, sweep, D2H inside the call)
        _lib.check(_lib.lib().abo_acq_eval(h._h, acq.acq_id, _lib.ptr(pp), C.c_void_p(Xh.ctypes.data), m,
                                           C.c_void_p(scores_host.data_ptr()), TOPK, _lib.ptr(ti), _lib.ptr(tv)))
    step_e2e()
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(lib_stream)
    w0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    e3.record(lib_stream)
    barrier()
    wall_e2e = time.perf_counter() - w0
    ms_e2e = max(e2.elapsed_time(e3), 1e3 * wall_e2e)          # host-side top-k is part of the call
    t = torch.tensor([ms_e2e], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * m * args.steps / (float(t.item()) * 1e-3)
    same_top = bool(np.array_equal(ti + rank * m, top_idx)) if world == 1 else None

    # ---- roofline of the dominant kernel (rank 0's numbers)
    peak, peak_src = fp64_peak()
    Npad = (n + 127) // 128 * 128
    fused = prof_ms[0] < 0.05 * max(prof_ms[1], 1e-9)             # single-kernel path: the builder class is empty
    trmm_ms, trmm_n = prof_ms[1], max(prof_n[1], 1)
    cand_per_launch = m * prof_steps / trmm_n
    achieved = (float(n) * n * cand_per_launch) / (trmm_ms / trmm_n * 1e-3) / 1e12
    traffic, traffic_src = None, None
    try:
        summ = json.load(open(os.path.join(ROOT, "profiles", "ncu_sweep_fused_r02_summary.json")))
        if fused and n == summ["n"] and abs(cand_per_launch - summ["candidates_per_launch"]) < 1:
            traffic = summ["dram_bytes_read"] + summ["dram_bytes_write"]
            traffic_src = "static: dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture of this exact " \
                          "launch shape (profiles/ncu_sweep_fused_r02_summary.json); not re-measured in this run"
    except Exception:
        pass
    kname = ("sweep_fused_kernel (K* tile build + TMA/mbarrier/DMMA W = L^-1 K* + column sum of squares + mean + EI in ONE kernel)"
             if fused else "sweep_tma_kernel (TMA + mbarrier + DMMA: W = L^-1 K*, fused column sum of squares)")
    roofline = {"bound": "tensor", "kernel": kname,
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src,
                "peak_source": peak_src, "algorithmic_flop_per_candidate": float(n) * n,
                "candidates_per_launch": cand_per_launch, "avg_launch_ms": trmm_ms / trmm_n,
                "note": "achieved counts the n^2 flop per candidate of the variance contraction only, although the fused "
                        "kernel also evaluates the n kernel entries per candidate (3 n d flop + n exp on the same FP64 pipe)",
                "share_of_step": {"ks_build": prof_ms[0] / max(sum(prof_ms), 1e-9),
                                  "sweep_kernel": prof_ms[1] / max(sum(prof_ms), 1e-9),
                                  "acq_epilogue": prof_ms[2] / max(sum(prof_ms), 1e-9)},
                "whole_step_tflops": flops_per_candidate(n, d) * m * args.steps / (ms * 1e-3) / 1e12}

    # ---- Cholesky TFLOP/s (second BASELINE metric), rank 0 only: ours (abo_potrf_dev) next to the library
    #      (cuSOLVER Dpotrf through torch.linalg.cholesky_ex) on the same matrices, same events, same run
    chol = None
    if rank == 0 and not args.no_cholesky:
        try:
            torch.backends.cuda.preferred_linalg_library("cusolver")
        except Exception:
            pass

        def spd(nn, seed):
            Xs = torch.rand((nn, DIM), dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
            return torch.exp(-0.5 * torch.cdist(Xs, Xs) ** 2) + 1e-2 * torch.eye(nn, dtype=torch.float64, device="cuda")

        def time_ours(K0, nn, reps):
            A = torch.empty_like(K0); best = 1e30
            for it in range(reps + 1):
                A.copy_(K0); torch.cuda.synchronize()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record(lib_stream); ctx.potrf_dev(A.data_ptr(), nn, nn); s1.record(lib_stream); torch.cuda.synchronize()
                if it:
                    best = min(best, s0.elapsed_time(s1))
            return best, A

        def time_lib(K0, reps):
            best = 1e30; L = None
            for it in range(reps + 1):
                torch.cuda.synchronize()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record(); L, _ = torch.linalg.cholesky_ex(K0, check_errors=False); s1.record(); torch.cuda.synchronize()
                if it:
                    best = min(best, s0.elapsed_time(s1))
            return best, L
        sizes = []
        for nn in (2048, 4096, 5632, 8192):
            K0 = spd(nn, 100 + nn)
            t_ours, A = time_ours(K0, nn, 4)
            t_lib, L = time_lib(K0, 4)
            err = float((torch.tril(A) - L).abs().max())
            fl = nn ** 3 / 3.0 + nn ** 2 / 2.0
            sizes.append({"n": nn, "ours_ms": t_ours, "cusolver_ms": t_lib, "ours_tflops": fl / (t_ours * 1e-3) / 1e12,
                          "cusolver_tflops": fl / (t_lib * 1e-3) / 1e12, "ours_faster": bool(t_ours < t_lib),
                          "max_abs_diff_L": err})
            del K0, A, L
        main_sz = [z for z in sizes if z["n"] == 8192][0]
        chol = {"n": 8192, "ms": main_sz["ours_ms"], "tflops": main_sz["ours_tflops"], "frac_of_peak": main_sz["ours_tflops"] / peak,
                "vs_library": sizes, "library": "cuSOLVER Dpotrf via torch.linalg.cholesky_ex (preferred_linalg_library=cusolver)",
                "first_fit_s_incl_allocation": t_fit}
        # the whole conditioning step (K build + Cholesky + triangular inverse + alpha), warm, through the host API
        tw = []
        for _ in range(3):
            t1 = time.perf_counter()
            mfit = abo.update(abo.StandardGP(kern, c["noise"], ctx=ctx), c["X"], c["y"], allow_append=False)
            tw.append(time.perf_counter() - t1)
            del mfit
        chol["fit_ms_warm"] = 1e3 * min(tw)
        # a larger factorisation: the look-ahead schedule approaches the GEMM rate as the panel share shrinks
        n2 = 16384
        K2 = spd(n2, 7)
        best2, A2 = time_ours(K2, n2, 2)
        fl2 = n2 ** 3 / 3.0 + n2 ** 2 / 2.0
        chol["larger"] = {"n": n2, "ms": best2, "tflops": fl2 / (best2 * 1e-3) / 1e12,
                          "frac_of_peak": fl2 / (best2 * 1e-3) / 1e12 / peak}
        del K2, A2

    cpu = None
    if rank == 0 and args.gpus == 1 and not args.no_cpu_baseline:
        r = cpu_restatement_throughput(args.cpu_sample, n=n)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["threads"], "kind": "port", "blas": r["blas"],
               "host_cpu_count": os.cpu_count() or 1,
               "sample": f"{args.cpu_sample} candidates (posterior mean+var+EI+top-{TOPK}) at n={n}, d={d}; "
                         f"{r['t_step']:.2f} s per pass; oracle/abo_oracle.py on NumPy/SciPy (the Julia reference cannot run here)",
               "one_thread": {"value": r["one_thread_value"], "cores": 1, "sample": f"{r['one_thread_sample']} candidates"},
               "fit_s": r["t_fit"]}

    if rank == 0:
        steps = max(args.steps, 1)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": workload_config(n, d, m, world),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": m * d * 8, "d2h_bytes_per_step": m * 8 + TOPK * 16,
                    "what": "abo_acq_eval with pinned host candidates and host score / top-k buffers: H2D, sweep, device "
                            "top-k, D2H inside the timed call (the conditioning step is in `value`'s step, not here)",
                    "topk_matches_device_run": same_top},
            "gpu_launches": int(launches),
            "iteration_ms": {k: 1e3 * v / steps for k, v in parts.items()} | {
                "what": "rank 0's host timers around the synchronous library calls of one step, averaged over the timed steps",
                "posterior_broadcast_bytes": None if world == 1 else int(Npad // 128 * (Npad // 128 + 1) * 128 * 128 * 8),
                "posterior_broadcast_gb_per_s": None if world == 1 or parts["sync"] == 0 else
                Npad // 128 * (Npad // 128 + 1) * 128 * 128 * 8 / (parts["sync"] / steps) / 1e9},
            "cross_rank_check": xrank,
            "roofline": roofline,
            "cholesky": chol,
            "cpu_baseline": cpu,
        }
        print(json.dumps(line), flush=True)
    if rank == 0:
        model_h.close()
    del base, recv                                 # release the device state explicitly, not at interpreter exit
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Device-resident sweep throughput of the fused single-kernel path as a function of n:
EI + stable top-100 over m candidates already in HBM (abo_acq_eval_dev), CUDA events on the library's stream.
    python tools/sweep_scan.py [--n 64,128,...] [--d 20] [--m 2097152] [--kind 0] [--label fused]
(profiles/sweep_scan_r02.jsonl also records the three-kernel path at the same n for comparison.)  Prints one JSON line per n:
candidates/s, algorithmic TFLOP/s (n^2 and n^2 + 3nd + 4n per candidate), fraction of the measured FP64 peak,
and the candidate-stream GB/s (8(d+1) B per candidate) for the small-n, HBM-side view."""
import argparse, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import abo_b200 as abo
from oracle import abo_oracle as orc

ap = argparse.ArgumentParser()
ap.add_argument("--n", default="64,128,256,512,1024,2048")
ap.add_argument("--d", type=int, default=20)
ap.add_argument("--m", type=int, default=1 << 21)
ap.add_argument("--kind", type=int, default=0)
ap.add_argument("--label", default="fused")
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()
KN = {0: "SqExponentialKernel", 1: "Matern52Kernel", 2: "Matern72Kernel"}
try:
    PEAK = float(json.load(open(os.path.join(os.path.dirname(__file__), "..", "profiles", "fp64_peaks_r01.json")))["cublas_dgemm_nt_tflops"]["8192"])
except Exception:
    PEAK = 35.95
ctx = abo.default_context()
stream = torch.cuda.ExternalStream(ctx.stream())
for n in [int(v) for v in args.n.split(",")]:
    d, m = args.d, args.m
    rng = np.random.default_rng(n)
    X = rng.random((n, d)); y = np.sin(3 * X).sum(1) / d + 0.1 * rng.standard_normal(n); y = (y - y.mean()) / y.std(ddof=1)
    ell = 1.0 if d >= 12 else 0.5
    gp = abo.update(abo.StandardGP(1.0 * abo.with_lengthscale(abo.Kernel(KN[args.kind]), ell), 1e-2 if d >= 12 else 1e-4), X, y)
    acq = abo.ExpectedImprovement(0.01, float(y.min()))
    Xc = torch.rand((m, d), dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n))
    S = torch.empty(m, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    run = lambda: gp.gpx.acq_eval_dev(acq.acq_id, acq.params(), Xc.data_ptr(), m, S.data_ptr(), k=100)
    run(); run()
    best = 1e30
    for _ in range(args.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); e0.record(stream); run(); e1.record(stream); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    ctx.profile(True); run(); pms, pn = ctx.profile_read(); ctx.profile(False)
    t = best * 1e-3
    print(json.dumps({"label": args.label, "n": n, "d": d, "m": m, "kind": args.kind, "ms": best, "cand_per_s": m / t,
                      "tflops_n2": n * n * m / t / 1e12, "frac_peak_n2": n * n * m / t / 1e12 / PEAK,
                      "tflops_all": (n * n + 3 * n * d + 4 * n) * m / t / 1e12,
                      "cand_stream_gbs": 8 * (d + 1) * m / t / 1e9,
                      "kernel_ms": {"ks_build": pms[0], "contraction_or_fused": pms[1], "epilogue": pms[2]},
                      "launches_per_sweep": pn[1]}), flush=True)
    del gp, Xc, S

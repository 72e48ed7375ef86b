"""Max-value entropy search on the device: the sweep rate with the MES epilogue against EI, the cost of the y* draw, and
the per-iteration time of optimize_acquisition with MES and with EI.

Sweep: SE, d = 20, n in {64, 512, 2048, 8192} observations, 2 097 152 device-resident candidates (262 144 at n = 8192),
K in {16, 64} sampled minimum values.  abo_acq_eval_dev writes the scores to a device buffer; windows of at least
--window seconds of back-to-back calls are timed with CUDA events on the library's stream after a warm-up call, EI and
MES alternating in the same process, --reps windows each.  The candidates (8 m d bytes, up to 336 MB) do not fit the
126 MB L2.
y* draw: abo_gp_pathwise_sample_dev over the same candidates with K draws and 4096 features, argmins only (what
MaxValueEntropySearch.topk draws before its sweep); median of --reps calls.
optimize_acquisition: the reference's sizes, n = 60, d = 2, a 10 000-point grid, 100 starts and the batched analytic
refinement; host wall time per call (it ends in a device synchronise), median of --reps, MES (K = 16) and EI alternating.

    python tools/mes_probe.py --out profiles/mes_probe_r03.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import abo_b200 as abo  # noqa: E402

D = 20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def window(fn, stream, min_s):
    """Calls per second of fn over a window of at least min_s seconds (CUDA events on `stream`)."""
    fn()
    torch.cuda.synchronize()
    calls, ms = 0, 0.0
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    t0 = time.perf_counter()
    while True:
        fn()
        calls += 1
        if time.perf_counter() - t0 >= min_s:
            break
    b.record(stream); b.synchronize()
    ms = a.elapsed_time(b)
    return calls, ms


def model(rng, n):
    X = rng.random((n, D))
    y = np.sin(3 * X[:, 0]) + np.cos(2 * X[:, 1]) + 0.3 * X.sum(1) + 0.01 * rng.standard_normal(n)
    y = (y - y.mean()) / y.std()
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.SqExponentialKernel(), 1.5), 1e-3), X, y)
    return gp, float(y.min())


def sweep_part(args, stream, out):
    rng = np.random.default_rng(1)
    for n in args.ns:
        m = 262144 if n >= 8192 else 2097152
        gp, best = model(rng, n)
        h = gp.gpx
        xc = torch.rand((m, D), dtype=torch.float64, device="cuda")
        sc = torch.empty(m, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        ei = [0.0, best]
        row = {"n": n, "m": m, "d": D}
        for K in args.ks:
            _, yv = h.pathwise_sample_dev(xc.data_ptr(), m, K, 7, 4096)
            ys = np.minimum(yv, best)
            mes = np.concatenate([[float(K)], ys])
            # y* draw: argmins only
            h.pathwise_sample_dev(xc.data_ptr(), m, K, 7, 4096)
            torch.cuda.synchronize()
            tdraw = []
            for _ in range(args.reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(stream); h.pathwise_sample_dev(xc.data_ptr(), m, K, 7, 4096); b.record(stream); b.synchronize()
                tdraw.append(a.elapsed_time(b))
            rates = {"EI": [], "MES": []}
            for _ in range(args.reps):
                for name, aid, pr in (("EI", 0, ei), ("MES", 4, mes)):
                    calls, ms = window(lambda: h.acq_eval_dev(aid, pr, xc.data_ptr(), m, sc.data_ptr(), 0), stream, args.window)
                    rates[name].append(calls * m / (ms / 1e3))
            # the same bits as the sweep's own posterior: spot check of the scores against the read-back posterior
            h.acq_eval_dev(4, mes, xc.data_ptr(), m, sc.data_ptr(), 0)
            torch.cuda.synchronize()
            idx = np.arange(0, m, max(1, m // 4096))
            mu, var = h.posterior(xc[idx].cpu().numpy())
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import mes_reference as mref
            ref = mref.mes(mu, var, ys)
            rel = float(np.max(np.abs(sc[idx].cpu().numpy() - ref) / (np.abs(ref) + 1e-300)))
            e, s = np.array(rates["EI"]), np.array(rates["MES"])
            row[f"K{K}"] = {
                "ei_cands_per_s": rates["EI"], "mes_cands_per_s": rates["MES"],
                "ei_median": float(np.median(e)), "mes_median": float(np.median(s)),
                "mes_over_ei": float(np.median(s) / np.median(e)),
                "ei_spread": float((e.max() - e.min()) / np.median(e)),
                "ystar_draw_ms_median": float(np.median(tdraw)), "ystar_draw_ms": tdraw,
                "sweep_ms_ei": float(m / np.median(e) * 1e3), "sweep_ms_mes": float(m / np.median(s) * 1e3),
                "mes_vs_reference_max_rel": rel,
            }
            print(json.dumps({"n": n, "K": K, **{k: v for k, v in row[f"K{K}"].items() if not isinstance(v, list)}}), flush=True)
        out["sweep"].append(row)
        del xc, sc
        h.ctx.trim()


def bo_part(args, out):
    rng = np.random.default_rng(2)
    X = rng.random((60, 2)) * 12 - 6
    f = lambda x: (x[:, 0] ** 2 + x[:, 1] - 11) ** 2 + (x[:, 0] + x[:, 1] ** 2 - 7) ** 2
    y = f(X); y = (y - y.mean()) / y.std()
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.SqExponentialKernel(), 2.0), 1e-6), X, y)
    dom = abo.ContinuousDomain([-6.0, -6.0], [6.0, 6.0])
    acqs = {"EI": abo.ExpectedImprovement(0.0, float(y.min())), "MES": abo.MaxValueEntropySearch(3, float(y.min()), 16)}
    ts = {"EI": [], "MES": []}
    for name, a in acqs.items():
        abo.optimize_acquisition(a, gp, dom, n_grid=10_000, n_local=100, rng=np.random.default_rng(0))
    for r in range(args.reps):
        for name, a in acqs.items():
            t0 = time.perf_counter()
            abo.optimize_acquisition(a, gp, dom, n_grid=10_000, n_local=100, rng=np.random.default_rng(r))
            ts[name].append((time.perf_counter() - t0) * 1e3)
    out["optimize_acquisition"] = {"n": 60, "d": 2, "n_grid": 10000, "n_local": 100, "K": 16,
                                   "ei_ms": ts["EI"], "mes_ms": ts["MES"],
                                   "ei_ms_median": float(np.median(ts["EI"])), "mes_ms_median": float(np.median(ts["MES"]))}
    print(json.dumps({k: v for k, v in out["optimize_acquisition"].items() if not isinstance(v, list)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--ns", type=int, nargs="+", default=[64, 512, 2048, 8192])
    ap.add_argument("--ks", type=int, nargs="+", default=[16, 64])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--window", type=float, default=0.5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("mes_probe needs a GPU")
    ctx = abo.default_context()
    stream = torch.cuda.ExternalStream(ctx.stream())
    out = {"card": card(), "sweep": [], "window_s": args.window, "reps": args.reps}
    sweep_part(args, stream, out)
    bo_part(args, out)
    out["card_after"] = card()
    s = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(s + "\n")
    print("mes_probe done")


if __name__ == "__main__":
    main()

"""Monte-Carlo batch expected improvement on the device (abo_acq_qei): the cost of scoring a grid cut into batches, of a
value-and-gradient call, and of optimize_acquisition with batches, each next to a reference point.

Grid: SE, d = 20, n in {512, 2048, 8192} observations, a 10 000-point grid cut into 10 000 // q batches, q in {2, 4, 8},
S in {128, 512} samples.  Value-only abo_acq_qei against abo_acq_eval's EI sweep of the same 10 000 points.  Host wall time
per call (every call ends in a device synchronise), median of --reps after a warm-up call.
Gradient: 100 batches, value and gradient in one call.
Torch: the same math written in torch on the GPU (K* from torch ops, solve_triangular with the library's own factor,
batched cholesky, the same normals, autograd for the gradient), timed in the same process with the order alternated, and
its values compared with the library's.
optimize_acquisition: the reference's sizes, n = 60, d = 2, a 10 000-point grid, 100 starts, qExpectedImprovement with
q = 4 (S = 512) next to EI (q = 1).

    python tools/qei_probe.py --out profiles/qei_probe_r03.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import abo_b200 as abo  # noqa: E402
import qei_reference as qref  # noqa: E402

D = 20
M = 10_000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def model(rng, n):
    X = rng.random((n, D))
    y = np.sin(3 * X[:, 0]) + np.cos(2 * X[:, 1]) + 0.3 * X.sum(1) + 0.01 * rng.standard_normal(n)
    y = (y - y.mean()) / y.std()
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.SqExponentialKernel(), 1.5), 1e-3), X, y)
    return gp, X, float(y.min())


def torch_qei(h, X, Xb, params, S, seed, tau, grad=False):
    """The same estimate in torch on the GPU from the library's factor L and alpha (SE kernel, isotropic)."""
    dev = "cuda"
    L = torch.as_tensor(h.factor(0), device=dev)
    alpha = torch.as_tensor(h.alpha(), device=dev)
    Xt = torch.as_tensor(X, device=dev)
    B, q, d = Xb.shape
    xb = torch.tensor(Xb, device=dev, requires_grad=grad)
    s = 1.0 / 1.5

    def run():
        P = xb.reshape(B * q, d)
        Ks = torch.exp(-0.5 * torch.cdist(Xt * s, P * s, compute_mode="donot_use_mm_for_euclid_dist") ** 2)   # (n, B q)
        mu = (Ks.T @ alpha).reshape(B, q)
        V = torch.linalg.solve_triangular(L, Ks, upper=False).T.reshape(B, q, -1)       # (B, q, n)
        Pb = xb * s
        prior = torch.exp(-0.5 * ((Pb[:, :, None, :] - Pb[:, None, :, :]) ** 2).sum(-1))
        eye = torch.eye(q, dtype=torch.float64, device=dev)
        Sig = prior - V @ V.transpose(1, 2) + (1e-18 + tau) * eye
        Lc = torch.linalg.cholesky(Sig)
        F = mu[:, None, :] + torch.einsum("bjk,sk->bsj", Lc, Z)
        val = torch.clamp((params[1] - params[0]) - F.min(dim=2).values, min=0.0).mean(dim=1)
        if grad:
            return val.detach(), torch.autograd.grad(val.sum(), xb)[0]
        return val.detach(), None

    Z = torch.as_tensor(qref.normals(seed, S, q), device=dev)
    return run


def grid_part(args, out):
    rng = np.random.default_rng(1)
    for n in args.ns:
        gp, X, best = model(rng, n)
        h = gp.gpx
        grid = rng.random((M, D))
        pr = [0.0, best]
        t_ei = [timed(lambda: h.acq_eval(0, pr, grid))[0] for _ in range(args.reps + 1)][1:]
        for q in args.qs:
            Xb = grid[:(M // q) * q].reshape(M // q, q, D)
            for S in args.ss:
                h.acq_qei(pr, q, Xb, S, 3)
                tq, tt = [], []
                run = torch_qei(h, X, Xb, pr, S, 3, 1e-10 * 1.0)
                run()
                for r in range(args.reps):                                          # alternated order
                    pair = [("lib", lambda: h.acq_qei(pr, q, Xb, S, 3)), ("torch", run)]
                    for name, fn in (pair if r % 2 == 0 else pair[::-1]):
                        ms, res = timed(fn)
                        (tq if name == "lib" else tt).append(ms)
                v, _, tau = h.acq_qei(pr, q, Xb, S, 3)
                vt = run()[0].cpu().numpy()
                row = {"n": n, "d": D, "grid": M, "q": q, "S": S, "batches": M // q,
                       "qei_ms": tq, "qei_ms_median": float(np.median(tq)),
                       "ei_sweep_ms": t_ei, "ei_sweep_ms_median": float(np.median(t_ei)),
                       "qei_over_ei": float(np.median(tq) / np.median(t_ei)),
                       "torch_ms": tt, "torch_ms_median": float(np.median(tt)),
                       "torch_over_lib": float(np.median(tt) / np.median(tq)),
                       "tau_all_first_rung": bool(np.all(tau == 1e-10)),
                       "max_abs_diff_vs_torch": float(np.max(np.abs(v - vt))), "max_value": float(np.max(v))}
                print(json.dumps({k: x for k, x in row.items() if not isinstance(x, list)}), flush=True)
                out["grid"].append(row)
                del run
                torch.cuda.empty_cache()
        # value and gradient, 100 batches, with an incumbent most of them can improve on
        for q in args.qs:
            Xb = grid[:100 * q].reshape(100, q, D)
            S = 512
            pr = [0.0, float(np.quantile(abo.posterior_mean(gp, Xb.reshape(-1, D)), 0.3))]
            h.acq_qei(pr, q, Xb, S, 3, want_grad=True)
            run = torch_qei(h, X, Xb, pr, S, 3, 1e-10, grad=True)
            run()
            tq, tt = [], []
            for r in range(args.reps):
                pair = [("lib", lambda: h.acq_qei(pr, q, Xb, S, 3, want_grad=True)), ("torch", run)]
                for name, fn in (pair if r % 2 == 0 else pair[::-1]):
                    ms, _ = timed(fn)
                    (tq if name == "lib" else tt).append(ms)
            v, g, _ = h.acq_qei(pr, q, Xb, S, 3, want_grad=True)
            vt, gt = run()
            row = {"n": n, "q": q, "S": S, "batches": 100, "qei_grad_ms": tq, "qei_grad_ms_median": float(np.median(tq)),
                   "torch_autograd_ms": tt, "torch_autograd_ms_median": float(np.median(tt)),
                   "max_abs_diff_value": float(np.max(np.abs(v - vt.cpu().numpy()))),
                   "max_abs_diff_grad": float(np.max(np.abs(g - gt.cpu().numpy()))), "max_abs_grad": float(np.max(np.abs(g)))}
            print(json.dumps({k: x for k, x in row.items() if not isinstance(x, list)}), flush=True)
            out["grad"].append(row)
        h.ctx.trim()


def bo_part(args, out):
    rng = np.random.default_rng(2)
    X = rng.random((60, 2)) * 12 - 6
    f = lambda x: (x[:, 0] ** 2 + x[:, 1] - 11) ** 2 + (x[:, 0] + x[:, 1] ** 2 - 7) ** 2
    y = f(X); y = (y - y.mean()) / y.std()
    gp = abo.update(abo.StandardGP(abo.with_lengthscale(abo.SqExponentialKernel(), 2.0), 1e-6), X, y)
    dom = abo.ContinuousDomain([-6.0, -6.0], [6.0, 6.0])
    acqs = {"EI": abo.ExpectedImprovement(0.0, float(y.min())), "qEI4": abo.qExpectedImprovement(0.0, float(y.min()), 4)}
    ts = {k: [] for k in acqs}
    for a in acqs.values():
        abo.optimize_acquisition(a, gp, dom, n_grid=10_000, n_local=100, rng=np.random.default_rng(0))
    for r in range(args.reps):
        for name, a in (list(acqs.items()) if r % 2 == 0 else list(acqs.items())[::-1]):
            t0 = time.perf_counter()
            abo.optimize_acquisition(a, gp, dom, n_grid=10_000, n_local=100, rng=np.random.default_rng(r))
            ts[name].append((time.perf_counter() - t0) * 1e3)
    out["optimize_acquisition"] = {"n": 60, "d": 2, "n_grid": 10000, "n_local": 100, "q": 4, "S": 512,
                                   "ei_ms": ts["EI"], "qei_ms": ts["qEI4"],
                                   "ei_ms_median": float(np.median(ts["EI"])), "qei_ms_median": float(np.median(ts["qEI4"]))}
    print(json.dumps({k: v for k, v in out["optimize_acquisition"].items() if not isinstance(v, list)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--ns", type=int, nargs="+", default=[512, 2048, 8192])
    ap.add_argument("--qs", type=int, nargs="+", default=[2, 4, 8])
    ap.add_argument("--ss", type=int, nargs="+", default=[128, 512])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("qei_probe needs a GPU")
    out = {"card": card(), "grid": [], "grad": [], "reps": args.reps}
    grid_part(args, out)
    bo_part(args, out)
    out["card_after"] = card()
    s = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(s + "\n")
    print("qei_probe done")


if __name__ == "__main__":
    main()

"""Joint posterior sampling (abo_gp_posterior_sample) against the same math composed from torch / cuBLAS / cuSOLVER.

Shape: n = 8192 observations, d = 20, SE kernel; m in {2048, 4096, 8192, 16384} candidates, S in {1, 256, 4096} draws.
Both sides are timed with CUDA events on the library's stream after one warm-up call per shape (median of --reps), and
both stop at the per-draw argmins: no draw is copied to the host in the timed calls.  The algorithmic flop count is
    N^2 M (W = L^-1 K*) + N M^2 (G = W^T W, lower half) + M^3 / 3 (Cholesky) + M^2 S (L_Sigma Z),
reported as TFLOP/s and against the 35.95 TFLOP/s measured Dgemm rate of DESIGN.md section 3.  For every m the draws of
both sides at S = 256 are computed from the same normals (the library's Philox stream, restated in NumPy) and compared
within max(1e-9, 16 eps cond2(Sigma + tau I)) sigma_f max|Z|, cond2 by power / inverse-power iteration on the device.

    python tools/sample_probe.py --out profiles/sample_probe_r03.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import abo_b200 as abo  # noqa: E402
import sample_reference as ref  # noqa: E402

DGEMM_TFLOPS = 35.95
N, D, INV_LS, SCALE, NOISE, JITTER = 8192, 20, 1.0 / 1.5, 1.0, 1e-3, 1e-10


def flops(n, m, s):
    return n * n * m + n * m * m + m ** 3 / 3 + m * m * s


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, stream, reps):
    fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream); fn(); b.record(stream); b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def se_kernel(A, B):
    d2 = torch.cdist(A * INV_LS, B * INV_LS, compute_mode="donot_use_mm_for_euclid_dist") ** 2
    return SCALE * torch.exp(-0.5 * d2)


class TorchSampler:
    """The posterior of the same data and the per-call math: K*, W = L^-1 K*, Sigma = K** - W^T W + (1e-18 + tau) I,
    chol(Sigma), mu + L_Sigma Z, argmin."""

    def __init__(self, X, y):
        self.X = torch.tensor(X, device="cuda")
        K = se_kernel(self.X, self.X) + NOISE * torch.eye(len(X), device="cuda", dtype=torch.float64)
        self.L = torch.linalg.cholesky(K)
        self.alpha = torch.cholesky_solve(torch.tensor(y, device="cuda")[:, None], self.L)[:, 0]

    def factor(self, Xc, tau):
        Ks = se_kernel(self.X, Xc)
        W = torch.linalg.solve_triangular(self.L, Ks, upper=False)
        sig = se_kernel(Xc, Xc) - W.T @ W
        sig.diagonal().add_(1e-18 + tau)
        return Ks.T @ self.alpha, torch.linalg.cholesky(sig)

    def sample(self, Xc, Z, tau):
        mu, Ls = self.factor(Xc, tau)
        F = mu[None, :] + Z @ Ls.T
        return F, torch.argmin(F, dim=1)


def cond2(Ls, iters=30):
    """2-norm condition number of Ls Ls^T by power and inverse-power iteration."""
    g = torch.Generator(device="cuda").manual_seed(0)
    v = torch.randn(Ls.shape[0], 1, device="cuda", dtype=torch.float64, generator=g); w = v.clone()
    lmax = lmin_inv = 1.0
    for _ in range(iters):
        t = Ls @ (Ls.T @ v); lmax = float(t.norm()); v = t / lmax
        t = torch.cholesky_solve(w, Ls); lmin_inv = float(t.norm()); w = t / lmin_inv
    return lmax * lmin_inv


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--m", type=int, nargs="*", default=[2048, 4096, 8192, 16384])
    ap.add_argument("--s", type=int, nargs="*", default=[1, 256, 4096])
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("sample_probe needs a CUDA device")
    rng = np.random.default_rng(0)
    X = rng.random((N, D)); y = np.sin(3 * X[:, 0]) + np.cos(2 * X[:, 1]) + 0.1 * X.sum(1)
    ctx = abo.default_context()
    gp = abo.update(abo.StandardGP(SCALE * abo.with_lengthscale(abo.SqExponentialKernel(), 1.0 / INV_LS), NOISE), X, y)
    h = gp.gpx
    stream = torch.cuda.ExternalStream(ctx.stream())
    ts = TorchSampler(X, y)
    out = {"card": card(), "shape": {"n": N, "d": D, "kernel": "SE", "inv_ls": INV_LS, "noise": NOISE, "jitter": JITTER},
           "dgemm_tflops": DGEMM_TFLOPS, "runs": [], "parity": []}
    for m in a.m:
        Xc = rng.random((m, D)); Xt = torch.tensor(Xc, device="cuda")
        # parity at S = 256 with the library's own normals
        F, _, _, tau = h.posterior_sample(Xc, 256, 7, JITTER)
        Z = torch.tensor(ref.normals(7, 256, m), device="cuda")
        with torch.cuda.stream(stream):
            Ft, _ = ts.sample(Xt, Z, tau)
            _, Ls = ts.factor(Xt, tau)
            c2 = cond2(Ls)
        tol = max(1e-9, 16 * np.finfo(float).eps * c2) * np.sqrt(SCALE) * float(Z.abs().max())
        err = float((torch.tensor(F, device="cuda") - Ft).abs().max())
        out["parity"].append({"m": m, "S": 256, "tau": tau, "cond2": c2, "max_abs_diff": err, "tol": tol, "ok": bool(err <= tol)})
        del Ls, Ft
        for S in a.s:
            lib_ms = timed(lambda: h.posterior_sample(Xc, S, 11, JITTER, want_samples=False), stream, a.reps)
            Zs = torch.randn(S, m, device="cuda", dtype=torch.float64)
            with torch.cuda.stream(stream):
                torch_ms = timed(lambda: ts.sample(Xt, Zs, tau)[1].cpu(), stream, a.reps)
            fl = flops(N, m, S)
            r = {"m": m, "S": S, "flop": fl, "lib_ms": lib_ms, "lib_tflops": fl / lib_ms * 1e-9,
                 "lib_share_of_dgemm": fl / lib_ms * 1e-9 / DGEMM_TFLOPS, "torch_ms": torch_ms,
                 "torch_tflops": fl / torch_ms * 1e-9, "speedup_vs_torch": torch_ms / lib_ms}
            out["runs"].append(r)
            print(json.dumps(r), flush=True)
            del Zs
        torch.cuda.empty_cache()
    print(json.dumps(out["parity"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

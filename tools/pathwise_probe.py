"""Pathwise posterior draws (abo_gp_pathwise_sample_dev) on large candidate sets, with the exact joint sampler and the same
pathwise math composed from torch at the exact sampler's largest set.

Shape: n = 8192 observations, d = 20, SE and Matern-5/2, L = 4096 random Fourier features; m in {16384, 262144, 2097152}
device-resident candidates, S in {16, 128} draws.  Each call is timed with CUDA events on the library's stream after one
warm-up call per shape (median of --reps) and ends at the per-draw argmins: the timed calls write no draw.  The flop count
is the algorithm's, from the shapes (N = n, padded sizes not counted):
    2 S L N (R = Theta' Phi(X)^T) + 2 N^2 S (L^-1 R and L^-T Y, triangular halves) + 2 m (N + L) S (the draws)
    + m N (3 d + 20) (K* rows, the kernel counted as 20 flops) + m L (2 d + 20) (features, the cosine counted as 20).
At m = 16384 the same run times abo_gp_posterior_sample with the same S, and the pathwise math written in torch
(cdist kernel, torch.cos, matmuls, cholesky_solve on the factor of the fit, which is not timed), on the library's own
feature and draw streams; the two pathwise results are compared.

    python tools/pathwise_probe.py --out profiles/pathwise_probe_r03.json
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
import pathwise_reference as pref  # noqa: E402

N, D, L, INV_LS, SCALE, NOISE = 8192, 20, 4096, 1.0 / 1.5, 1.0, 1e-3
KINDS = {"SE": (0, "SqExponentialKernel"), "Matern52": (1, "Matern52Kernel")}


def flops(m, S, n=N, d=D, nf=L):
    return 2 * S * nf * n + 2 * n * n * S + 2 * m * (n + nf) * S + m * n * (3 * d + 20) + m * nf * (2 * d + 20)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, stream, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream); fn(); b.record(stream); b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def kern(kind, A, B):
    r2 = torch.cdist(A * INV_LS, B * INV_LS, compute_mode="donot_use_mm_for_euclid_dist") ** 2
    if kind == 0:
        return SCALE * torch.exp(-0.5 * r2)
    r = torch.sqrt(r2)
    return SCALE * (1 + 5 ** 0.5 * r + 5 * r2 / 3) * torch.exp(-(5 ** 0.5) * r)


class TorchPathwise:
    """The same pathwise draws from torch: mean_c + K* (alpha - V) + Phi* Theta'^T, V = (K + noise I)^-1 R."""

    def __init__(self, kind, X, y, Om, b, Theta):
        self.kind = kind
        self.X = torch.tensor(X, device="cuda")
        K = kern(kind, self.X, self.X) + NOISE * torch.eye(len(X), device="cuda", dtype=torch.float64)
        self.Lc = torch.linalg.cholesky(K)
        self.alpha = torch.cholesky_solve(torch.tensor(y, device="cuda")[:, None], self.Lc)[:, 0]
        self.Om, self.b = torch.tensor(Om, device="cuda"), torch.tensor(b, device="cuda")
        self.Theta = torch.tensor(Theta, device="cuda")

    def sample(self, Xc, S):
        th = (2.0 * SCALE / L) ** 0.5 * self.Theta[:S, :L]
        eps = NOISE ** 0.5 * self.Theta[:S, L:]
        R = torch.cos((self.X * INV_LS) @ self.Om.T + self.b) @ th.T + eps.T
        V = torch.cholesky_solve(R, self.Lc)
        F = kern(self.kind, Xc, self.X) @ (self.alpha[:, None] - V) + torch.cos((Xc * INV_LS) @ self.Om.T + self.b) @ th.T
        F = F.T
        return F, torch.argmin(F, dim=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--m", type=int, nargs="*", default=[16384, 262144, 2097152])
    ap.add_argument("--s", type=int, nargs="*", default=[16, 128])
    ap.add_argument("--kernels", nargs="*", default=list(KINDS))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pathwise_probe needs a CUDA device")
    rng = np.random.default_rng(0)
    X = rng.random((N, D)); y = np.sin(3 * X[:, 0]) + np.cos(2 * X[:, 1]) + 0.1 * X.sum(1)
    ctx = abo.default_context()
    stream = torch.cuda.ExternalStream(ctx.stream())
    out = {"card": card(), "shape": {"n": N, "d": D, "L": L, "inv_ls": INV_LS, "noise": NOISE},
           "timing": "CUDA events on the library's stream, median of %d calls after one warm-up; argmins only" % a.reps,
           "runs": [], "m16384": []}
    seed = 11
    for kname in a.kernels:
        kind, cname = KINDS[kname]
        gp = abo.update(abo.StandardGP(SCALE * abo.with_lengthscale(abo.Kernel(cname), 1.0 / INV_LS), NOISE), X, y)
        h = gp.gpx
        for m in a.m:
            Xt = torch.tensor(rng.random((m, D)), device="cuda")
            for S in a.s:
                ms = timed(lambda: h.pathwise_sample_dev(Xt.data_ptr(), m, S, seed, L), stream, a.reps)
                fl = flops(m, S)
                r = {"kernel": kname, "m": m, "S": S, "flop": fl, "ms": ms, "tflops": fl / ms * 1e-9,
                     "candidates_per_s": m / ms * 1e3}
                out["runs"].append(r)
                print(json.dumps(r), flush=True)
            if m == 16384:
                Om, b = pref.features(seed, L, D, kind)
                Theta = pref.draw_normals(seed, max(a.s), L + N)
                tp = TorchPathwise(kind, X, y, Om, b, Theta)
                Xc = Xt.cpu().numpy()
                for S in a.s:
                    exact_ms = timed(lambda: h.posterior_sample(Xc, S, seed, 1e-10, want_samples=False), stream, a.reps)
                    with torch.cuda.stream(stream):
                        torch_ms = timed(lambda: tp.sample(Xt, S)[1].cpu(), stream, a.reps)
                        Ft, _ = tp.sample(Xt, S)
                    F, _, _ = h.pathwise_sample(Xc, S, seed, L)
                    lib_ms = next(r["ms"] for r in out["runs"] if r["kernel"] == kname and r["m"] == m and r["S"] == S)
                    q = {"kernel": kname, "m": m, "S": S, "pathwise_ms": lib_ms, "exact_posterior_sample_ms": exact_ms,
                         "torch_pathwise_ms": torch_ms, "speedup_vs_exact": exact_ms / lib_ms,
                         "speedup_vs_torch": torch_ms / lib_ms,
                         "max_abs_diff_vs_torch": float((torch.tensor(F, device="cuda") - Ft).abs().max())}
                    out["m16384"].append(q)
                    print(json.dumps(q), flush=True)
                del tp
            del Xt
            torch.cuda.empty_cache()
        del gp, h
        ctx.trim()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

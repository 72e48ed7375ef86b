"""Torch FP64 CPU restatement of Monte-Carlo batch expected improvement (abo_acq_qei, include/abo.h), the reference of the
qEI tests.  The oracle's fit supplies the Cholesky factor U and alpha as constants; K*, the prior block of each batch and
the Monte-Carlo estimate are written in torch so that autograd gives the exact reference gradient:

    mu = mean_c + K*^T alpha,   Sigma = k(x_i, x_j) - V^T V + 1e-18 I,   V = U^-T K*,
    L = chol(Sigma + tau I),    f_s = mu + L z_s,   qEI = mean_s max((best_y - xi) - min_j f_{s,j}, 0),

z_s the normals [0, q) of the Philox stream with key (seed, 2^62 + s) and tau the first rung jitter sigma^2 10^k,
k = 0 .. 6, that factors.  Test infrastructure only, like oracle/."""
import numpy as np
import torch

import sample_reference as sref

KEY_OFFSET = 2 ** 62


def normals(seed, S, q):
    """(S, q): row s = the normals [0, q) of the stream with key (seed, 2^62 + s)."""
    return np.stack([sref.philox_normals(seed, KEY_OFFSET + s, q) for s in range(S)])


def _phi(kind, u):
    if kind == 0:
        return torch.exp(-u / 2), None
    r = torch.sqrt(u)
    if kind in (1, 3, 5):
        z = torch.exp(-np.sqrt(5.0) * r)
        return (1 + np.sqrt(5.0) * r + 5 * u / 3) * z, (-5.0 / 6.0) * (1 + np.sqrt(5.0) * r) * z
    z = torch.exp(-np.sqrt(7.0) * r)
    return ((1 + np.sqrt(7.0) * r + 14 * u / 5 + 7 * np.sqrt(7.0) * r * u / 15) * z,
            (-7.0 / 10.0) * (1 + np.sqrt(7.0) * r + 7 * u / 3) * z)


def _dphi(kind, u):
    if kind == 0:
        return -torch.exp(-u / 2) / 2
    return _phi(kind, u)[1]


def _kstar(post, Xb):
    """K* of the value output at the B q points of Xb (B, q, d): (B, N, q), training outputs out-major as the oracle's U."""
    sv = torch.as_tensor(np.broadcast_to(np.asarray(post.inv_ls, dtype=np.float64), (post.X.shape[1],)).copy())
    Xs = torch.as_tensor(post.X) * sv                                   # (n, d)
    Ys = Xb * sv                                                        # (B, q, d)
    D = Xs[None, :, None, :] - Ys[:, None, :, :]                        # (B, n, q, d): s (x_i - x_c)
    u = (D * D).sum(-1)
    blocks = [post.scale * _phi(post.kind, u)[0]]
    if post.p > 1:                                                      # d/dx_a rows of a GradientGP: 2 s_a sigma^2 phi' D_a
        dp = _dphi(post.kind, u)
        for a in range(post.X.shape[1]):
            blocks.append(2 * sv[a] * post.scale * dp * D[..., a])
    return torch.cat(blocks, dim=1)


def _sigma_mu(post, Xb):
    B, q, d = Xb.shape
    Ks = _kstar(post, Xb)
    alpha = torch.as_tensor(post.alpha)
    mu = float(post.mean_c[0]) + torch.einsum("bnq,n->bq", Ks, alpha)
    Ut = torch.as_tensor(post.U.T.copy())
    N = Ks.shape[1]
    V = torch.linalg.solve_triangular(Ut, Ks.permute(1, 0, 2).reshape(N, B * q), upper=False)
    V = V.reshape(N, B, q).permute(1, 0, 2)                            # (B, N, q)
    sv = torch.as_tensor(np.broadcast_to(np.asarray(post.inv_ls, dtype=np.float64), (d,)).copy())
    Ys = Xb * sv
    D = Ys[:, :, None, :] - Ys[:, None, :, :]
    u = (D * D).sum(-1)
    eye = torch.eye(q, dtype=torch.float64).expand(B, q, q)
    u = torch.where(eye > 0, torch.ones_like(u), u)                     # no sqrt(0) on the diagonal (its gradient is NaN)
    prior = torch.where(eye > 0, torch.full_like(u, post.scale), post.scale * _phi(post.kind, u)[0])
    Sig = prior - V.transpose(1, 2) @ V + 1e-18 * eye
    return Sig, mu


def ladder(Sig, jitter, scale):
    """tau per batch: the first jitter * scale * 10^k, k = 0 .. 6, whose Cholesky succeeds; NaN if none."""
    Sig = Sig.detach()
    B, q, _ = Sig.shape
    tau = np.full(B, np.nan)
    for k in range(7):
        t = jitter * scale * 10.0 ** k
        _, info = torch.linalg.cholesky_ex(Sig + t * torch.eye(q, dtype=torch.float64))
        ok = (info.numpy() == 0) & np.isnan(tau)
        tau[ok] = t
    return tau


def qei(post, Xb, xi, best_y, S, seed, jitter=1e-10, want_grad=True, tau=None):
    """(values (B,), grad (B, q, d) or None, tau (B,), the per-sample improvements (B, S)).  `tau` fixes the jitter per
    batch (the device's, for parity); by default the ladder picks it."""
    X = torch.tensor(np.asarray(Xb, dtype=np.float64), requires_grad=want_grad)
    B, q, d = X.shape
    Sig, mu = _sigma_mu(post, X)
    if tau is None:
        tau = ladder(Sig, jitter, post.scale)
    tau = np.asarray(tau, dtype=np.float64)
    L = torch.linalg.cholesky(Sig + torch.as_tensor(tau)[:, None, None] * torch.eye(q, dtype=torch.float64))
    Z = torch.as_tensor(normals(seed, S, q))                            # (S, q)
    F = mu[:, None, :] + torch.einsum("bjk,sk->bsj", L, Z)              # (B, S, q)
    imp = torch.clamp((best_y - xi) - F.min(dim=2).values, min=0.0)     # (B, S)
    val = imp.mean(dim=1)
    grad = None
    if want_grad:
        grad = torch.autograd.grad(val.sum(), X)[0].numpy()
    return val.detach().numpy(), grad, tau, imp.detach().numpy()

"""NumPy reference of abo_gp_pathwise_sample (include/abo.h): the feature and draw streams it consumes and the pathwise
posterior draws built from them with the oracle's posterior.  Test infrastructure only, like oracle/."""
import numpy as np
import scipy.linalg as sla

from oracle import abo_oracle as orc
import sample_reference as sref

DRAW_KEY = 1 << 63
KDF = {0: 0, 1: 5, 3: 5, 5: 5, 2: 7, 4: 7, 6: 7}      # Student-t degrees of freedom 2 nu per kernel id (0: SE, Gaussian)


def u01(w):
    return ((np.asarray(w, dtype=np.uint64) >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53


def features(seed, L, d, kind):
    """(Om (L, d), b (L,)): feature l's frequency in the library's scaled coordinates, z_l t_l (omega_l = s (.) Om[l]),
    and its phase b_l, from the stream with key (seed, 2^64 - 1 - l)."""
    kdf = KDF[kind]
    nz = d + kdf
    nblk = (nz + 3) // 4
    Om, b = np.empty((L, d)), np.empty(L)
    for l in range(L):
        key = (1 << 64) - 1 - l
        z = sref.philox_normals(seed, key, 4 * nblk)
        Om[l] = z[:d] * (np.sqrt(kdf / np.sum(z[d:nz] ** 2)) if kdf else 1.0)
        b[l] = 2.0 * np.pi * u01(sref.philox_words(seed, key, nblk + 1)[nblk, 0])
    return Om, b


def draw_normals(seed, S, count):
    """(S, count): normals [0, count) of draw s, key (seed, 2^63 + s)."""
    return np.stack([sref.philox_normals(seed, DRAW_KEY + s, count) for s in range(S)])


def inv_ls_vector(post):
    return np.broadcast_to(np.asarray(post.inv_ls, dtype=np.float64), (post.X.shape[1],))


def phi_value(Xc, sv, Om, b):
    """cos(omega_l . x + b_l), (m, L)."""
    return np.cos((np.atleast_2d(Xc) * sv) @ Om.T + b)


def phi_train(post, Om, b):
    """Feature rows of the training outputs in the oracle's out-major order (value rows, then d/dx_a for a GradientGP)."""
    sv = inv_ls_vector(post)
    ph = (post.X * sv) @ Om.T + b
    rows = [np.cos(ph)]
    for a in range(post.p - 1):
        rows.append(-(sv[a] * Om[:, a])[None, :] * np.sin(ph))
    return np.vstack(rows)


def pathwise_sample(post, Xc, S, seed, L):
    """(draws (S, m), Theta (S, L + N) the draw normals): mean + k*^T (-v_s) + phi(x) theta'_s with
    v_s = (K + noise I)^-1 (phi(X) theta'_s + eps_s)."""
    Xc = np.atleast_2d(np.asarray(Xc, dtype=np.float64))
    n, d = post.X.shape
    p, N = post.p, post.X.shape[0] * post.p
    Om, b = features(seed, L, d, post.kind)
    Theta = draw_normals(seed, S, L + N)
    th = np.sqrt(2.0 * post.scale / L) * Theta[:, :L]
    eps = np.sqrt(post.noise) * Theta[:, L:]                     # point-major i p + a
    eps = eps.reshape(S, n, p).transpose(0, 2, 1).reshape(S, N)  # -> out-major a n + i
    R = phi_train(post, Om, b) @ th.T + eps.T
    v = sla.cho_solve((post.U, False), R, check_finite=False)
    mean, _ = orc.posterior_mean_var(post, Xc)
    Ks = orc._kstar(post, Xc, [0])
    F = mean[None, :] - (Ks.T @ v).T + th @ phi_value(Xc, inv_ls_vector(post), Om, b).T
    return F, Theta

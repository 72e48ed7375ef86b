"""NumPy reference of abo_gp_posterior_sample (include/abo.h): the Philox4x64-10 normals it draws and the joint
posterior draws built from the oracle's posterior mean and covariance.  Test infrastructure only, like oracle/."""
import numpy as np
import scipy.linalg as sla

from oracle import abo_oracle as orc

PHILOX_M = (0xD2E7470EE14C6C93, 0xCA5A826395121157)
PHILOX_W = (0x9E3779B97F4A7C15, 0xBB67AE8584CAA73B)
MASK64 = (1 << 64) - 1


def philox4x64_10(ctr, key):
    """Pure-Python Philox4x64-10 (Salmon et al., SC'11): ten rounds, the key bumped by the Weyl constants in between."""
    c = [int(v) for v in ctr]
    k0, k1 = int(key[0]), int(key[1])
    for _ in range(10):
        p0, p1 = PHILOX_M[0] * c[0], PHILOX_M[1] * c[2]
        c = [(p1 >> 64) ^ c[1] ^ k0, p1 & MASK64, (p0 >> 64) ^ c[3] ^ k1, p0 & MASK64]
        k0, k1 = (k0 + PHILOX_W[0]) & MASK64, (k1 + PHILOX_W[1]) & MASK64
    return c


def philox_words(seed, s, nblk):
    """Blocks j = 0 .. nblk-1 of draw s: NumPy's Philox with key (seed, s); it increments the counter before each block,
    so block j is the counter (j + 1, 0, 0, 0)."""
    return np.random.Philox(key=np.array([seed, s], dtype=np.uint64)).random_raw(4 * nblk).reshape(nblk, 4)


def philox_normals(seed, s, m):
    """The m standard normals of draw s: u = ((w >> 11) + 0.5) 2^-53 per word, two Box-Muller pairs per block."""
    w = philox_words(seed, s, (m + 3) // 4)
    u = ((w >> np.uint64(11)).astype(np.float64) + 0.5) * 2.0 ** -53
    r0, r2 = np.sqrt(-2.0 * np.log(u[:, 0])), np.sqrt(-2.0 * np.log(u[:, 2]))
    z = np.stack([r0 * np.cos(2 * np.pi * u[:, 1]), r0 * np.sin(2 * np.pi * u[:, 1]),
                  r2 * np.cos(2 * np.pi * u[:, 3]), r2 * np.sin(2 * np.pi * u[:, 3])], axis=1).reshape(-1)
    return z[:m]


def normals(seed, S, m):
    return np.stack([philox_normals(seed, s, m) for s in range(S)]) if S > 0 else np.empty((0, m))


def posterior_sample(post, Xc, S, seed, tau):
    """(draws (S, m), Sigma + tau I, Z): row s = mean + cholesky(posterior_cov + tau I) z_s, value output."""
    Xc = np.atleast_2d(np.asarray(Xc, dtype=np.float64))
    m = Xc.shape[0]
    mean, _ = orc.posterior_mean_var(post, Xc)
    sig = orc.posterior_cov(post, Xc, outputs=[0]) + tau * np.eye(m)
    L = sla.cholesky(sig, lower=True, check_finite=False)
    Z = normals(seed, S, m)
    return mean[None, :] + Z @ L.T, sig, Z

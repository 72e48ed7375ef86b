"""NumPy / SciPy float64 restatement of max-value entropy search (include/abo.h, ABO_ACQ_MES), the reference of the MES
tests.  Minimising: for K sampled minimum values y*_k,

    MES(x) = (1/K) sum_k h(gamma_k),  gamma_k = (mu - y*_k) / sigma,  h(g) = g r(g) / 2 - log Phi(g),  r = phi / Phi,

and 0 where var <= 1e-12.  The branches are those of the device code (csrc/kernels.cuh, mes_h / mes_hprime): erfc for
g >= 0, erfcx for g < 0, and for h' at g <= -4 the continued fraction of the Mills ratio, where the direct form cancels."""
import numpy as np
from scipy.special import erfc, erfcx

_S2 = 0.70710678118654752440
_SQRT_2_OVER_PI = 0.79788456080286535588
_INV_SQRT_2PI = 0.39894228040143267794
MES_TAIL = -4.0
MES_CF_DEPTH = 32


def _normpdf(g):
    return np.exp(-(g * g) / 2) * _INV_SQRT_2PI


def h(g):
    """h(g) = g r(g) / 2 - log Phi(g), elementwise."""
    g = np.asarray(g, dtype=np.float64)
    out = np.empty_like(g)
    pos = g >= 0
    gp = g[pos]
    e = erfc(gp * _S2)
    r = _normpdf(gp) / (1.0 - e / 2)
    out[pos] = gp * r / 2 - np.log1p(-e / 2)
    gn = g[~pos]
    t = -gn * _S2
    ex = erfcx(t)
    r = _SQRT_2_OVER_PI / ex
    out[~pos] = gn * r / 2 - (np.log(ex / 2) - t * t)
    return out


def hprime(g):
    """dh/dg = -(r/2)(1 + g (g + r)), elementwise."""
    g = np.asarray(g, dtype=np.float64)
    out = np.empty_like(g)
    mid = g > MES_TAIL
    gm = g[mid]
    r = np.where(gm >= 0, _normpdf(gm) / (1.0 - erfc(gm * _S2) / 2), _SQRT_2_OVER_PI / erfcx(-np.minimum(gm, 0.0) * _S2))
    out[mid] = -(r / 2) * (1.0 + gm * (gm + r))
    u = -g[~mid]
    rho = np.zeros_like(u); rho2 = np.zeros_like(u)
    for k in range(MES_CF_DEPTH, 0, -1):
        rho = k / (u + rho)
        if k == 2:
            rho2 = rho
    out[~mid] = -(rho * rho2) * (u + rho) / 2
    return out


def _gammas(mu, var, ystar):
    mu = np.asarray(mu, dtype=np.float64); var = np.asarray(var, dtype=np.float64)
    ys = np.asarray(ystar, dtype=np.float64).reshape(-1)
    live = var > 1e-12
    sig = np.sqrt(np.where(live, var, 1.0))
    return mu, var, ys, live, sig


def mes(mu, var, ystar):
    """MES scores for posterior means / variances mu, var (any shape) and the y* values; the sum runs over k in
    ascending order and is then divided by K."""
    mu, var, ys, live, sig = _gammas(mu, var, ystar)
    acc = np.zeros_like(mu)
    for y in ys:
        acc = acc + h((mu - y) / sig)
    return np.where(live, acc / len(ys), 0.0)


def mes_dmu_dvar(mu, var, ystar):
    """(d MES / d mu, d MES / d var); both 0 where var <= 1e-12."""
    mu, var, ys, live, sig = _gammas(mu, var, ystar)
    sd = np.zeros_like(mu); sdg = np.zeros_like(mu)
    for y in ys:
        g = (mu - y) / sig
        hp = hprime(g)
        sd = sd + hp
        sdg = sdg + hp * g
    K = len(ys)
    return np.where(live, (sd / K) / sig, 0.0), np.where(live, -(sdg / K) / (2 * np.where(live, var, 1.0)), 0.0)

"""ctypes binding of libabo_cuda.so (include/abo.h).  This is the analogue of the `ccall`
stubs a Julia maintainer would add (INTEGRATION.md).  There is no CPU fallback: if the shared
library or a CUDA device is missing every call raises."""
from __future__ import annotations

import ctypes as C
import itertools
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libabo_cuda.so")

ABO_OK, ABO_ERR_INVALID, ABO_ERR_DIM, ABO_ERR_NOT_POSDEF, ABO_ERR_CUDA, ABO_ERR_NOT_FITTED, ABO_ERR_NCCL, ABO_ERR_ALLOC = range(8)

# every symbol include/abo.h declares (tests check the library exports all of them)
SYMBOLS = [
    "abo_version", "abo_last_error", "abo_ctx_create", "abo_ctx_destroy", "abo_ctx_device", "abo_ctx_stream",
    "abo_ctx_launch_count", "abo_ctx_profile", "abo_ctx_profile_read", "abo_debug_potf2_clocks", "abo_gp_create", "abo_gp_destroy", "abo_gp_set_params", "abo_gp_fit", "abo_gp_append",
    "abo_gp_clone", "abo_gp_n", "abo_gp_alpha", "abo_gp_factor", "abo_gp_posterior", "abo_gp_posterior_cov", "abo_acq_eval", "abo_acq_eval_dev", "abo_acq_eval_grad",
    "abo_nlml_batch", "abo_potrf_dev", "abo_fill_distance", "abo_nccl_unique_id", "abo_ctx_init_rank", "abo_gp_sync",
    "abo_topk_allgather", "abo_allgather_f64", "abo_ctx_ranks", "abo_ctx_trim", "abo_acq_eval_multi", "abo_standardize", "abo_gp_set_params_ard", "abo_nlml_batch_ard",
    "abo_gp_posterior_sample", "abo_gp_pathwise_sample", "abo_gp_pathwise_sample_dev", "abo_acq_qei",
]


class PosDefException(Exception):
    """LinearAlgebra.PosDefException(info): what `update` throws when the Cholesky fails
    (src/bayesian_opt.jl:126-141 catches it)."""

    def __init__(self, info, msg=""):
        super().__init__(msg or f"matrix is not positive definite; Cholesky factorization failed at pivot {info}")
        self.info = int(info)


class DimensionMismatch(ValueError):
    pass


class AboCudaError(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AboCudaError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no CPU fallback.")
        L = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        vp, i32, i64, u64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_double
        pd = C.POINTER(C.c_double)
        L.abo_version.restype = i32
        L.abo_last_error.restype = C.c_char_p
        sigs = {
            "abo_ctx_create": [i32, C.POINTER(vp)],
            "abo_ctx_destroy": [vp],
            "abo_ctx_trim": [vp],
            "abo_ctx_device": [vp, C.POINTER(i32)],
            "abo_ctx_stream": [vp, C.POINTER(vp)],
            "abo_ctx_launch_count": [vp, C.POINTER(i64)],
            "abo_ctx_profile": [vp, i32],
            "abo_ctx_profile_read": [vp, vp, vp],
            "abo_debug_potf2_clocks": [vp, vp],
            "abo_gp_create": [vp, i32, i32, i32, C.POINTER(vp)],
            "abo_gp_destroy": [vp],
            "abo_gp_set_params": [vp, dbl, dbl, dbl, vp],
            "abo_gp_set_params_ard": [vp, vp, dbl, dbl, vp],
            "abo_gp_fit": [vp, vp, vp, i64, C.POINTER(i64)],
            "abo_gp_append": [vp, vp, vp, C.POINTER(i64)],
            "abo_gp_clone": [vp, C.POINTER(vp)],
            "abo_gp_n": [vp, C.POINTER(i64)],
            "abo_gp_alpha": [vp, vp],
            "abo_gp_factor": [vp, i32, vp],
            "abo_gp_posterior": [vp, vp, i64, i32, vp, vp],
            "abo_gp_posterior_cov": [vp, vp, i64, i32, vp],
            "abo_gp_posterior_sample": [vp, vp, i64, i64, u64, dbl, vp, vp, vp, C.POINTER(C.c_double)],
            "abo_gp_pathwise_sample": [vp, vp, i64, i64, i64, u64, vp, vp, vp],
            "abo_gp_pathwise_sample_dev": [vp, vp, i64, i64, i64, u64, vp, vp, vp],
            "abo_acq_eval": [vp, i32, vp, vp, i64, vp, i64, vp, vp],
            "abo_acq_eval_dev": [vp, i32, vp, vp, i64, vp, i64, vp, vp],
            "abo_acq_eval_multi": [vp, i32, vp, vp, vp, vp, i64, vp, i64, vp, vp],
            "abo_acq_eval_grad": [vp, i32, vp, vp, i64, vp, vp, vp, vp],
            "abo_acq_qei": [vp, vp, i32, vp, i64, i64, u64, dbl, vp, vp, vp],
            "abo_nlml_batch": [vp, vp, vp, i64, vp, i64, vp, vp, vp],
            "abo_nlml_batch_ard": [vp, vp, vp, i64, vp, i64, vp, vp, vp],
            "abo_potrf_dev": [vp, vp, i64, i64, C.POINTER(i64)],
            "abo_fill_distance": [vp, vp, i64, i32, vp, i64, C.POINTER(C.c_double)],
            "abo_standardize": [vp, vp, i64, i32, i32, vp, vp, vp, C.POINTER(C.c_double)],
            "abo_nccl_unique_id": [vp],
            "abo_ctx_init_rank": [vp, i32, i32, vp],
            "abo_gp_sync": [vp, i32],
            "abo_topk_allgather": [vp, i64, i64, vp, vp, C.POINTER(i64)],
            "abo_allgather_f64": [vp, vp, i64, vp],
            "abo_ctx_ranks": [vp, C.POINTER(i32), C.POINTER(i32)],
        }
        for name, args in sigs.items():
            f = getattr(L, name)
            f.argtypes = args
            f.restype = i32
        _lib = L
    return _lib


def check(rc, info=None):
    if rc == ABO_OK:
        return
    msg = lib().abo_last_error().decode("utf-8", "replace")
    if rc == ABO_ERR_NOT_POSDEF:
        raise PosDefException(info if info is not None else -1, msg)
    if rc == ABO_ERR_DIM:
        raise DimensionMismatch(msg)
    if rc == ABO_ERR_INVALID:
        raise ValueError(msg)
    raise AboCudaError(f"libabo_cuda status {rc}: {msg}")


def f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


class Context:
    """abo_ctx: one CUDA device, its stream and workspace."""

    def __init__(self, device: int = 0):
        h = C.c_void_p()
        check(lib().abo_ctx_create(int(device), C.byref(h)))
        self._h = h
        self.device = int(device)

    @property
    def handle(self):
        return self._h

    def stream(self) -> int:
        s = C.c_void_p()
        check(lib().abo_ctx_stream(self._h, C.byref(s)))
        return s.value or 0

    def launch_count(self) -> int:
        n = C.c_int64()
        check(lib().abo_ctx_launch_count(self._h, C.byref(n)))
        return n.value

    def profile(self, enable: bool):
        check(lib().abo_ctx_profile(self._h, 1 if enable else 0))

    def profile_read(self):
        ms = (C.c_double * 3)(); n = (C.c_int64 * 3)()
        check(lib().abo_ctx_profile_read(self._h, ms, n))
        return list(ms), list(n)

    def fill_distance(self, X, S) -> float:
        X = f64(X); S = f64(S)
        out = C.c_double(0.0)
        check(lib().abo_fill_distance(self._h, ptr(X), X.shape[0], X.shape[1], ptr(S), S.shape[0], C.byref(out)))
        return out.value

    def standardize(self, y_flat, n: int, p: int, choice: str):
        """get_mean_std + std_y on the device; returns (mu[p], sd[p], y_std (out-major), min of the standardised values)."""
        code = {"mean_scale": 0, "scale_only": 1, "mean_only": 2}[choice]
        y = f64(np.ravel(y_flat))
        if y.size != n * p:
            raise DimensionMismatch("ys length does not match n * p")
        mu = np.empty(p); sd = np.empty(p); ys = np.empty(n * p); best = C.c_double(0.0)
        check(lib().abo_standardize(self._h, ptr(y), n, p, code, ptr(mu), ptr(sd), ptr(ys), C.byref(best)))
        return mu, sd, ys, best.value

    def potf2_clocks(self):
        out = (C.c_int64 * 16)()
        check(lib().abo_debug_potf2_clocks(self._h, out))
        return list(out)

    def potrf_dev(self, dptr: int, n: int, ld: int) -> int:
        info = C.c_int64(0)
        rc = lib().abo_potrf_dev(self._h, C.c_void_p(dptr), n, ld, C.byref(info))
        check(rc, info.value)
        return info.value

    def init_rank(self, rank: int, nranks: int, unique_id: bytes):
        buf = (C.c_uint8 * 128).from_buffer_copy(unique_id)
        check(lib().abo_ctx_init_rank(self._h, rank, nranks, buf))

    def trim(self):
        """Release the pooled posterior buffer sets and workspaces the context keeps between calls."""
        check(lib().abo_ctx_trim(self._h))

    def ranks(self):
        """(rank, nranks) of the context's NCCL communicator; (0, 1) without one."""
        r = C.c_int32(0); n = C.c_int32(1)
        check(lib().abo_ctx_ranks(self._h, C.byref(r), C.byref(n)))
        return r.value, n.value

    def topk_allgather(self, k, idx, val):
        """NCCL all-gather + merge of per-rank (global index, value) top-k lists."""
        ti = np.zeros(k, dtype=np.int64); tv = np.zeros(k)
        cnt = min(len(idx), k)
        ti[:cnt] = idx[:cnt]; tv[:cnt] = val[:cnt]
        out = C.c_int64(0)
        check(lib().abo_topk_allgather(self._h, k, cnt, ptr(ti), ptr(tv), C.byref(out)))
        return ti[:out.value], tv[:out.value]

    def allgather_f64(self, send, nranks: int):
        """NCCL all-gather of equally sized float64 blocks; returns an (nranks, len(send)) array."""
        send = f64(np.ravel(send))
        if self.ranks()[1] != nranks:
            raise AboCudaError(f"allgather_f64 over {nranks} ranks, but the context's NCCL communicator spans "
                               f"{self.ranks()[1]} (call init_nccl_context first)")
        recv = np.empty((nranks, send.size))
        check(lib().abo_allgather_f64(self._h, ptr(send), send.size, ptr(recv)))
        return recv

    def close(self):
        if self._h is not None and self._h.value:
            lib().abo_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def nccl_unique_id() -> bytes:
    buf = (C.c_uint8 * 128)()
    check(lib().abo_nccl_unique_id(buf))
    return bytes(buf)


_default_ctx = {}

# posterior tokens: a handle takes a fresh one whenever its posterior may change (create, set_params, fit, append, the
# receiving side of sync), so a token names one posterior state for the life of the process (ids of dead handles are
# reused, tokens are not)
_TOKENS = itertools.count(1)


def default_context(device: int | None = None) -> Context:
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if "ABO_DEVICE" not in os.environ else int(os.environ["ABO_DEVICE"])
    if device not in _default_ctx or _default_ctx[device]._h is None:      # never created, or closed by the caller
        _default_ctx[device] = Context(device)
    return _default_ctx[device]


class GpHandle:
    """abo_gp: a surrogate resident in HBM."""

    def __init__(self, ctx: Context, kernel_id: int, d: int, p: int, _h=None):
        self.ctx, self.kernel_id, self.d, self.p = ctx, kernel_id, d, p
        if _h is None:
            h = C.c_void_p()
            check(lib().abo_gp_create(ctx.handle, kernel_id, d, p, C.byref(h)))
            _h = h
        self._h = _h
        self.token = next(_TOKENS)

    def set_params(self, inv_ls, scale, noise, mean_c=None):
        self.token = next(_TOKENS)
        mc = None if mean_c is None else f64(np.atleast_1d(mean_c))
        if mc is not None and mc.size != self.p:
            raise DimensionMismatch("mean_c must have p entries")
        if np.ndim(inv_ls) > 0:                               # ARD: one inverse length scale per dimension
            sv = f64(np.ravel(inv_ls))
            if sv.size != self.d:
                raise DimensionMismatch(f"ARD kernel has {sv.size} length scales, the data have dimension {self.d}")
            check(lib().abo_gp_set_params_ard(self._h, ptr(sv), float(scale), float(noise), ptr(mc)))
        else:
            check(lib().abo_gp_set_params(self._h, float(inv_ls), float(scale), float(noise), ptr(mc)))

    def fit(self, X, y_flat):
        X = f64(X); y = f64(y_flat)
        n = X.shape[0]
        if X.ndim != 2 or X.shape[1] != self.d:
            raise DimensionMismatch(f"xs must be n x {self.d}")
        if y.size != n * self.p:
            raise DimensionMismatch("ys length does not match xs")
        info = C.c_int64(0)
        self.token = next(_TOKENS)
        rc = lib().abo_gp_fit(self._h, ptr(X), ptr(y), n, C.byref(info))
        check(rc, info.value)

    def append(self, x, y):
        x = f64(np.ravel(x)); y = f64(np.ravel(y))
        if x.size != self.d or y.size != self.p:
            raise DimensionMismatch("appended observation has the wrong dimension")
        info = C.c_int64(0)
        self.token = next(_TOKENS)
        rc = lib().abo_gp_append(self._h, ptr(x), ptr(y), C.byref(info))
        check(rc, info.value)

    def clone(self) -> "GpHandle":
        h = C.c_void_p()
        check(lib().abo_gp_clone(self._h, C.byref(h)))
        return GpHandle(self.ctx, self.kernel_id, self.d, self.p, _h=h)

    def n(self) -> int:
        n = C.c_int64()
        check(lib().abo_gp_n(self._h, C.byref(n)))
        return n.value

    def alpha(self):
        out = np.empty(self.n() * self.p)
        check(lib().abo_gp_alpha(self._h, ptr(out)))
        return out

    def factor(self, which=0):
        N = self.n() * self.p
        out = np.empty((N, N))
        check(lib().abo_gp_factor(self._h, which, ptr(out)))
        return np.tril(out)

    def posterior(self, Xc, outputs=1, want_mean=True, want_var=True):
        Xc = f64(Xc)
        if Xc.ndim != 2 or Xc.shape[1] != self.d:
            raise DimensionMismatch(f"query points must be m x {self.d}")
        m = Xc.shape[0]
        mean = np.empty(m * outputs) if want_mean else None
        var = np.empty(m * outputs) if want_var else None
        check(lib().abo_gp_posterior(self._h, ptr(Xc), m, outputs, ptr(mean), ptr(var)))
        return mean, var

    def posterior_cov(self, Xc, outputs=1):
        Xc = f64(Xc)
        if Xc.ndim != 2 or Xc.shape[1] != self.d:
            raise DimensionMismatch(f"query points must be m x {self.d}")
        M = Xc.shape[0] * outputs
        cov = np.empty((M, M))
        check(lib().abo_gp_posterior_cov(self._h, ptr(Xc), Xc.shape[0], outputs, ptr(cov)))
        return cov

    def posterior_sample(self, Xc, num_samples, seed, jitter=1e-10, want_samples=True):
        """Joint draws of the value output over Xc: (samples (S, m) or None, argmin indices (S,), argmin values (S,),
        the jitter tau actually added to the covariance)."""
        Xc = f64(Xc)
        if Xc.ndim != 2 or Xc.shape[1] != self.d:
            raise DimensionMismatch(f"query points must be m x {self.d}")
        m, S, seed = Xc.shape[0], int(num_samples), int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must be in [0, 2^64)")
        samples = np.empty((max(S, 0), m)) if want_samples else None
        ai = np.empty(max(S, 1), dtype=np.int64); av = np.empty(max(S, 1)); tau = C.c_double(0.0)
        check(lib().abo_gp_posterior_sample(self._h, ptr(Xc), m, S, seed, float(jitter),
                                            ptr(samples), ptr(ai), ptr(av), C.byref(tau)))
        return samples, ai[:max(S, 0)], av[:max(S, 0)], tau.value

    def pathwise_sample(self, Xc, num_samples, seed, num_features=4096, want_samples=True):
        """Pathwise posterior draws of the value output over Xc (random-Fourier-feature prior, Matheron's rule):
        (samples (S, m) or None, argmin indices (S,), argmin values (S,))."""
        Xc = f64(Xc)
        if Xc.ndim != 2 or Xc.shape[1] != self.d:
            raise DimensionMismatch(f"query points must be m x {self.d}")
        m, S, seed = Xc.shape[0], int(num_samples), int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must be in [0, 2^64)")
        samples = np.empty((max(S, 0), m)) if want_samples else None
        ai = np.empty(max(S, 1), dtype=np.int64); av = np.empty(max(S, 1))
        check(lib().abo_gp_pathwise_sample(self._h, ptr(Xc), m, S, int(num_features), seed, ptr(samples), ptr(ai), ptr(av)))
        return samples, ai[:max(S, 0)], av[:max(S, 0)]

    def pathwise_sample_dev(self, d_xc: int, m: int, num_samples, seed, num_features=4096, d_samples: int = 0):
        """As pathwise_sample for m device-resident candidates; the S x m draws go to d_samples when it is not 0.
        Returns (argmin indices (S,), argmin values (S,))."""
        S, seed = int(num_samples), int(seed)
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must be in [0, 2^64)")
        ai = np.empty(max(S, 1), dtype=np.int64); av = np.empty(max(S, 1))
        check(lib().abo_gp_pathwise_sample_dev(self._h, C.c_void_p(d_xc), int(m), S, int(num_features), seed,
                                               C.c_void_p(d_samples) if d_samples else None, ptr(ai), ptr(av)))
        return ai[:max(S, 0)], av[:max(S, 0)]

    def acq_eval(self, acq_id, params, Xc, k=0, want_scores=True):
        Xc = f64(Xc)
        if Xc.ndim != 2 or Xc.shape[1] != self.d:
            raise DimensionMismatch(f"query points must be m x {self.d}")
        m = Xc.shape[0]
        params = f64(params)
        scores = np.empty(m) if want_scores else None
        k = min(int(k), m)
        ti = np.empty(max(k, 1), dtype=np.int64); tv = np.empty(max(k, 1))
        check(lib().abo_acq_eval(self._h, acq_id, ptr(params), ptr(Xc), m, ptr(scores), k, ptr(ti), ptr(tv)))
        return scores, ti[:k], tv[:k]

    def acq_eval_multi(self, acq_ids, weights, params, Xc, k=0, want_scores=True):
        """Weighted sum of acquisition members (EI / PI / UCB / GradientNormUCB = 3) from one posterior pass."""
        Xc = f64(Xc)
        if Xc.ndim != 2 or Xc.shape[1] != self.d:
            raise DimensionMismatch(f"query points must be m x {self.d}")
        m = Xc.shape[0]
        ids = np.ascontiguousarray(acq_ids, dtype=np.int32); w = f64(weights)
        pr = np.zeros((len(ids), 2)); 
        for q, row in enumerate(params):
            pr[q, :len(row)] = row
        scores = np.empty(m) if want_scores else None
        k = min(int(k), m)
        ti = np.empty(max(k, 1), dtype=np.int64); tv = np.empty(max(k, 1))
        check(lib().abo_acq_eval_multi(self._h, len(ids), ptr(ids), ptr(w), ptr(pr), ptr(Xc), m, ptr(scores), k, ptr(ti), ptr(tv)))
        return scores, ti[:k], tv[:k]

    def acq_eval_grad(self, acq_id, params, Xc):
        """scores (m) and d score / d x (m x d) for a batch of points."""
        Xc = f64(Xc)
        if Xc.ndim != 2 or Xc.shape[1] != self.d:
            raise DimensionMismatch(f"query points must be m x {self.d}")
        m = Xc.shape[0]
        params = f64(params)
        scores = np.empty(m); grad = np.empty((m, self.d))
        check(lib().abo_acq_eval_grad(self._h, acq_id, ptr(params), ptr(Xc), m, ptr(scores), ptr(grad), None, None))
        return scores, grad

    def acq_qei(self, params, q, Xb, S, seed, jitter=1e-10, want_grad=False):
        """Monte-Carlo batch expected improvement of B batches of q points, Xb of shape (B, q, d), params = (xi, best_y):
        (values (B,), d values / d Xb (B, q, d) or None, the jitter tau of each batch (B,))."""
        q, S, seed = int(q), int(S), int(seed)
        Xb = f64(Xb)
        if Xb.ndim != 3 or Xb.shape[1] != q or Xb.shape[2] != self.d:
            raise DimensionMismatch(f"batches must be B x {q} x {self.d}")
        if not 0 <= seed < 2 ** 64:
            raise ValueError("seed must be in [0, 2^64)")
        B = Xb.shape[0]
        params = f64(params)
        values = np.empty(max(B, 1)); tau = np.empty(max(B, 1))
        grad = np.empty((max(B, 1), q, self.d)) if want_grad else None
        check(lib().abo_acq_qei(self._h, ptr(params), q, ptr(Xb), B, S, seed, float(jitter), ptr(values), ptr(grad), ptr(tau)))
        return values[:B], (grad[:B] if want_grad else None), tau[:B]

    def acq_eval_dev(self, acq_id, params, d_xc: int, m: int, d_scores: int = 0, k=0):
        params = f64(params)
        k = min(int(k), m)
        ti = np.empty(max(k, 1), dtype=np.int64); tv = np.empty(max(k, 1))
        check(lib().abo_acq_eval_dev(self._h, acq_id, ptr(params), C.c_void_p(d_xc), m,
                                     C.c_void_p(d_scores) if d_scores else None, k, ptr(ti), ptr(tv)))
        return ti[:k], tv[:k]

    def nlml_batch(self, X, y_flat, logparams, want_grad=True, ard=False):
        """ard=False: rows {log l, log sig2}; ard=True: rows {log l_1 .. log l_d, log sig2}."""
        X = f64(X); y = f64(y_flat); lp = f64(np.atleast_2d(logparams))
        n = X.shape[0]; R = lp.shape[0]
        npar = self.d + 1 if ard else 2
        if lp.shape[1] != npar:
            raise DimensionMismatch(f"parameter vectors must have {npar} entries")
        if y.size != n * self.p:
            raise DimensionMismatch("ys length does not match xs")
        val = np.empty(R); grad = np.empty((R, npar)) if want_grad else None
        info = np.zeros(R, dtype=np.int32)
        fn = lib().abo_nlml_batch_ard if ard else lib().abo_nlml_batch
        check(fn(self._h, ptr(X), ptr(y), n, ptr(lp), R, ptr(val), ptr(grad), ptr(info)))
        return val, grad, info

    def sync(self, root=0):
        self.token = next(_TOKENS)
        check(lib().abo_gp_sync(self._h, root))

    def close(self):
        if self._h is not None and self._h.value:
            lib().abo_gp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

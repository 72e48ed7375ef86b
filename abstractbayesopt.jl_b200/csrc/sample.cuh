// sample.cuh — device kernels of the joint posterior sampler (abo_gp_posterior_sample):
//     f_s = mu + chol(Sigma + tau I) z_s,    s = 0 .. S-1,
// the standard normals z from a counter-based Philox4x64-10 stream that is pinned to NumPy's `Philox` bit generator, and
// a per-draw epilogue that adds the mean and finds the minimising candidate.  The O(m^3) / O(m^2 S) products run on the
// persistent TMA GEMM (gemm_tma.cuh) and the look-ahead Cholesky; see the driver in abo_api.cu.
// Also the feature generator, feature builder and coefficient transpose of the pathwise sampler (abo_gp_pathwise_sample).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "kernels.cuh"

namespace abo {

// Philox4x64-10 (Salmon et al., SC'11; Random123's philox4x64 with its default round count)
__device__ __forceinline__ void philox4x64_10(uint64_t c[4], uint64_t k0, uint64_t k1) {
    constexpr uint64_t M0 = 0xD2E7470EE14C6C93ull, M1 = 0xCA5A826395121157ull;
    constexpr uint64_t W0 = 0x9E3779B97F4A7C15ull, W1 = 0xBB67AE8584CAA73Bull;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t hi0 = __umul64hi(M0, c[0]), lo0 = M0 * c[0];
        const uint64_t hi1 = __umul64hi(M1, c[2]), lo1 = M1 * c[2];
        const uint64_t o0 = hi1 ^ c[1] ^ k0, o2 = hi0 ^ c[3] ^ k1;
        c[0] = o0; c[1] = lo1; c[2] = o2; c[3] = lo0;
        k0 += W0; k1 += W1;
    }
}

// uniform in (0, 1): the top 53 bits, centred in their interval (never 0, so the logarithm below is finite)
__device__ __forceinline__ double philox_u01(uint64_t w) { return ((double)(w >> 11) + 0.5) * 0x1.0p-53; }

// Normals 4j .. 4j+3 of the stream with key (k0, k1): Philox block j, counter (j + 1, 0, 0, 0) -- the words
// np.random.Philox(key=[k0, k1]).random_raw() returns at positions 4j .. 4j+3, since NumPy increments the counter before
// each block -- turned into (r0 cos 2 pi u1, r0 sin 2 pi u1, r2 cos 2 pi u3, r2 sin 2 pi u3), r = sqrt(-2 ln u).
__device__ __forceinline__ void philox_normal4(uint64_t k0, uint64_t k1, uint64_t j, double z[4]) {
    uint64_t c[4] = {j + 1, 0, 0, 0};
    philox4x64_10(c, k0, k1);
    double sn, cs;
    const double r0 = sqrt(-2.0 * log(philox_u01(c[0])));
    sincospi(2.0 * philox_u01(c[1]), &sn, &cs);
    z[0] = r0 * cs; z[1] = r0 * sn;
    const double r2 = sqrt(-2.0 * log(philox_u01(c[2])));
    sincospi(2.0 * philox_u01(c[3]), &sn, &cs);
    z[2] = r2 * cs; z[3] = r2 * sn;
}

// Z [Spad][ld], columns [0, width): Z[s][i] = scale * normal (idx_off + i) of the stream with key (seed, key_off + s), for
// draw s < S and i < m, zero elsewhere.  Z[s][i] depends on (seed, key_off + s, idx_off + i) only.  One thread per four
// columns; width and ld are multiples of 4.  The joint sampler uses key_off = idx_off = 0 and scale = 1.
__global__ void philox_normal_kernel(uint64_t seed, uint64_t key_off, int64_t idx_off, double scale, int64_t S, int64_t m,
                                     int64_t Spad, int64_t width, int64_t ld, double* __restrict__ Z) {
    const int64_t nblk = width / 4;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= Spad * nblk) return;
    const int64_t s = t / nblk, j = t % nblk;
    double z[4] = {0.0, 0.0, 0.0, 0.0};
    if (s < S && 4 * j < m) {
        const uint64_t key = key_off + (uint64_t)s;
        const int64_t q0 = idx_off + 4 * j, b0 = q0 / 4, sh = q0 % 4;
        double a[4];
        philox_normal4(seed, key, (uint64_t)b0, a);
        if (sh == 0) {
#pragma unroll
            for (int q = 0; q < 4; ++q) z[q] = a[q];
        } else {                                      // the four normals straddle two blocks
            double b[4];
            philox_normal4(seed, key, (uint64_t)b0 + 1, b);
#pragma unroll
            for (int q = 0; q < 4; ++q) z[q] = (q + sh < 4) ? a[q + sh] : b[q + sh - 4];
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) z[q] = (4 * j + q < m) ? z[q] * scale : 0.0;
    }
    double2* dst = reinterpret_cast<double2*>(Z + s * ld + 4 * j);
    dst[0] = make_double2(z[0], z[1]);
    dst[1] = make_double2(z[2], z[3]);
}

// potrf_lookahead leaves the strictly-upper 32-blocks of each diagonal tile as the trailing updates wrote them (the
// diagonal-block kernel writes back the columns of the lower part only); L_Sigma Z^T reads the diagonal tiles whole, so
// their strict upper part is zeroed first.  grid (T), one CTA per diagonal tile.
__global__ void zero_diag_upper_kernel(double* __restrict__ A, int64_t ld) {
    double* t = A + (int64_t)blockIdx.x * 128 * (ld + 1);
    for (int e = threadIdx.x; e < 128 * 128; e += blockDim.x) {
        const int r = e >> 7, c = e & 127;
        if (c > r) t[(int64_t)r * ld + c] = 0.0;
    }
}

// Julia findmin order as one unsigned key, smallest first: NaN before everything, then isless (-0.0 < 0.0)
__device__ __forceinline__ uint64_t findmin_key(double v) {
    if (v != v) return 0ull;
    const uint64_t u = (uint64_t)__double_as_longlong(v);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

// One CTA per draw s: F[s][i] += mu[i] (or + mu_c when mu is null) in place for i < m (the draw, sample-major), and the
// draw's minimiser in that order, ties to the smallest index, written to idx[s] / val[s] as off + i.  With carry, the
// chunk's minimiser replaces the (idx[s], val[s]) of the earlier chunks only when it is strictly smaller in that order: the
// earlier chunks hold the smaller indices.  The reduction tree is fixed, so the result is too.
constexpr int SF_THREADS = 256;
__global__ void __launch_bounds__(SF_THREADS) sample_finish_kernel(double* __restrict__ F, int64_t ld, const double* __restrict__ mu,
                                                                   double mu_c, int64_t m, int64_t off, int carry,
                                                                   long long* __restrict__ idx, double* __restrict__ val) {
    __shared__ uint64_t sk[SF_THREADS];
    __shared__ long long si[SF_THREADS];
    double* row = F + (int64_t)blockIdx.x * ld;
    uint64_t bk = ~0ull;
    long long bi = -1;
    for (int64_t i = threadIdx.x; i < m; i += SF_THREADS) {
        const double v = mu ? row[i] + mu[i] : row[i] + mu_c;
        row[i] = v;
        const uint64_t k = findmin_key(v);
        if (bi < 0 || k < bk) { bk = k; bi = i; }       // indices ascend per thread: strict < keeps the first
    }
    sk[threadIdx.x] = bk; si[threadIdx.x] = bi;
    __syncthreads();
    for (int w = SF_THREADS / 2; w > 0; w >>= 1) {
        if (threadIdx.x < w) {
            const uint64_t k2 = sk[threadIdx.x + w];
            const long long i2 = si[threadIdx.x + w];
            if (i2 >= 0 && (si[threadIdx.x] < 0 || k2 < sk[threadIdx.x] || (k2 == sk[threadIdx.x] && i2 < si[threadIdx.x]))) {
                sk[threadIdx.x] = k2; si[threadIdx.x] = i2;
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double v = row[si[0]];
        if (!carry || findmin_key(v) < findmin_key(val[blockIdx.x])) {
            idx[blockIdx.x] = off + si[0];
            val[blockIdx.x] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------
// pathwise posterior draws (abo_gp_pathwise_sample): random-Fourier-feature prior draws conditioned by Matheron's rule,
//     f_s(x) = mean_c + k(x, X) (alpha - v_s) + phi(x) . theta'_s,      v_s = (K + noise I)^-1 (phi(X) theta'_s + eps_s).
// The library stores coordinates scaled, s (.) x, so the device keeps each frequency in those coordinates:
// Om[l][k] = z_lk t_l, and omega_l . x = Om_l . (s (.) x).  A derivative output d/dx_k carries the factor s_k Om[l][k].
// ------------------------------------------------------------------------------------------

// Feature l < L: the stream with key (seed, 2^64 - 1 - l).  Normals [0, d) are z_l, normals [d, d + kdf) are g_l, and the
// phase is b_l = 2 pi u01(word 0 of the first block after them).  t_l = 1 (SE, kdf = 0) or sqrt(kdf / |g_l|^2) (Matern,
// a Student-t frequency with kdf = 2 nu degrees of freedom).  Features l in [L, Lpad) have Om = 0 and b = 0; their weights
// theta' are 0.  One thread per feature.  Om [Lpad][d], b [Lpad].
__global__ void rff_params_kernel(uint64_t seed, int d, int kdf, int64_t L, int64_t Lpad, double* __restrict__ Om,
                                  double* __restrict__ b) {
    const int64_t l = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (l >= Lpad) return;
    double* om = Om + l * d;
    if (l >= L) {
        for (int k = 0; k < d; ++k) om[k] = 0.0;
        b[l] = 0.0;
        return;
    }
    const uint64_t key = ~0ull - (uint64_t)l;
    const int nz = d + kdf, nblk = (nz + 3) / 4;
    double g2 = 0.0;
    for (int j = 0; j < nblk; ++j) {
        double z[4];
        philox_normal4(seed, key, (uint64_t)j, z);
        for (int q = 0; q < 4; ++q) {
            const int i = 4 * j + q;
            if (i < d) om[i] = z[q];
            else if (i < nz) g2 = fma(z[q], z[q], g2);
        }
    }
    if (kdf > 0) {
        const double t = sqrt((double)kdf / g2);
        for (int k = 0; k < d; ++k) om[k] *= t;
    }
    uint64_t c[4] = {(uint64_t)nblk + 1, 0, 0, 0};
    philox4x64_10(c, seed, key);
    b[l] = 2.0 * CUDART_PI * philox_u01(c[0]);
}

// Feature rows of `count` points: Phi[r][l] for l < Lpad, k-contiguous (ld = Lpad), for the GEMM operands.
//   Point i's scaled coordinates are xs_k = X[i xi + k xk] * (scale_in ? s_k : 1): raw candidates (xi = d, xk = 1,
//   scale_in) or the library's XsT (xi = 1, xk = ldx).  ph = (sum_k Om[l][k] xs_k, in k order) + b_l.
//   p = 1: row i = cos(ph).  p = d + 1 (training side of a GradientGP): rows i p + a in the library's point-major order,
//   a = 0 cos(ph), a >= 1 -s_{a-1} Om[l][a-1] sin(ph).  Rows of points i >= count, up to rows_out, are zero.
// Every element is evaluated alone in a fixed order, so a point's features do not depend on the set it is in.
// grid (Lpad / 128, ceil(rows_out / p / RFF_PB)), 128 threads = 128 features; the points of a CTA are staged in shared memory.
constexpr int RFF_PB = 16, RFF_MAXD = 64;
__global__ void __launch_bounds__(128) rff_build_kernel(KSpec spec, const double* __restrict__ Om, const double* __restrict__ b,
                                                        int64_t Lpad, const double* __restrict__ X, int64_t xi, int64_t xk,
                                                        int scale_in, int64_t count, int p, int64_t rows_out,
                                                        double* __restrict__ Phi) {
    __shared__ double xs[RFF_PB][RFF_MAXD];
    const int d = spec.d;
    const int64_t l = blockIdx.x * 128LL + threadIdx.x;
    const int64_t i0 = (int64_t)blockIdx.y * RFF_PB;
    for (int e = threadIdx.x; e < RFF_PB * d; e += 128) {
        const int c = e / d, k = e - c * d;
        const int64_t i = i0 + c;
        xs[c][k] = (i < count) ? (scale_in ? spec.sk(k) * X[i * xi + k * xk] : X[i * xi + k * xk]) : 0.0;
    }
    __syncthreads();
    const double* om = Om + l * d;
    const double bl = b[l];
    for (int c = 0; c < RFF_PB; ++c) {
        const int64_t i = i0 + c;
        if (i * p >= rows_out) break;
        double* dst = Phi + i * p * Lpad + l;
        if (i >= count) {
            for (int a = 0; a < p; ++a) if (i * p + a < rows_out) dst[a * Lpad] = 0.0;
            continue;
        }
        double ph = 0.0;
        for (int k = 0; k < d; ++k) ph = fma(om[k], xs[c][k], ph);
        ph += bl;
        double sn, cs;
        sincos(ph, &sn, &cs);
        dst[0] = cs;
        for (int a = 1; a < p; ++a) dst[a * Lpad] = -(spec.sk(a - 1) * om[a - 1]) * sn;
    }
}

// Bc [Spad][ldb], columns [0, Npad): Bc[s][k] = (k < N ? alpha[k] : 0) - V[k][s], V [Npad][Spad] (the transpose, through a
// 32 x 32 shared tile).  grid (Npad / 32, Spad / 32), block (32, 8).
__global__ void pathwise_coef_kernel(const double* __restrict__ alpha, int64_t N, const double* __restrict__ V, int64_t Npad,
                                     int64_t Spad, double* __restrict__ Bc, int64_t ldb) {
    __shared__ double t[32][33];
    const int64_t k0 = blockIdx.x * 32LL, s0 = blockIdx.y * 32LL;
    for (int r = threadIdx.y; r < 32; r += 8) t[r][threadIdx.x] = V[(k0 + r) * Spad + s0 + threadIdx.x];
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += 8) {
        const int64_t k = k0 + threadIdx.x;
        Bc[(s0 + r) * ldb + k] = (k < N ? alpha[k] : 0.0) - t[threadIdx.x][r];
    }
}

}  // namespace abo

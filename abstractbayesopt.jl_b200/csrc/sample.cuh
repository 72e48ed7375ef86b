// sample.cuh — device kernels of the joint posterior sampler (abo_gp_posterior_sample):
//     f_s = mu + chol(Sigma + tau I) z_s,    s = 0 .. S-1,
// the standard normals z from a counter-based Philox4x64-10 stream that is pinned to NumPy's `Philox` bit generator, and
// a per-draw epilogue that adds the mean and finds the minimising candidate.  The O(m^3) / O(m^2 S) products run on the
// persistent TMA GEMM (gemm_tma.cuh) and the look-ahead Cholesky; see the driver in abo_api.cu.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

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

// Z^T [Spad][ld]: Z[s][i] for draw s < S and candidate i < m, zero elsewhere.  Block j of draw s is Philox with
// key (seed, s) and counter (j + 1, 0, 0, 0) -- the words np.random.Philox(key=[seed, s]).random_raw() returns at
// positions 4j .. 4j+3, since NumPy increments the counter before each block.  Its four words give candidates 4j .. 4j+3
// by two Box-Muller pairs: (r0 cos 2 pi u1, r0 sin 2 pi u1, r2 cos 2 pi u3, r2 sin 2 pi u3), r = sqrt(-2 ln u).
// Z[s][i] depends on (seed, s, i) only.  One thread per block of four; ld is a multiple of 4.
__global__ void philox_normal_kernel(uint64_t seed, int64_t S, int64_t m, int64_t Spad, int64_t ld, double* __restrict__ Z) {
    const int64_t nblk = ld / 4;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= Spad * nblk) return;
    const int64_t s = t / nblk, j = t % nblk;
    double z[4] = {0.0, 0.0, 0.0, 0.0};
    if (s < S && 4 * j < m) {
        uint64_t c[4] = {(uint64_t)j + 1, 0, 0, 0};
        philox4x64_10(c, seed, (uint64_t)s);
        double sn, cs;
        const double r0 = sqrt(-2.0 * log(philox_u01(c[0])));
        sincospi(2.0 * philox_u01(c[1]), &sn, &cs);
        z[0] = r0 * cs; z[1] = r0 * sn;
        const double r2 = sqrt(-2.0 * log(philox_u01(c[2])));
        sincospi(2.0 * philox_u01(c[3]), &sn, &cs);
        z[2] = r2 * cs; z[3] = r2 * sn;
#pragma unroll
        for (int q = 0; q < 4; ++q) if (4 * j + q >= m) z[q] = 0.0;
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

// One CTA per draw s: F[s][i] += mu[i] in place for i < m (the draw, sample-major), and the draw's minimiser in that
// order, ties to the smallest index, written to idx[s] / val[s].  The reduction tree is fixed, so the result is too.
constexpr int SF_THREADS = 256;
__global__ void __launch_bounds__(SF_THREADS) sample_finish_kernel(double* __restrict__ F, int64_t ld, const double* __restrict__ mu,
                                                                   int64_t m, long long* __restrict__ idx, double* __restrict__ val) {
    __shared__ uint64_t sk[SF_THREADS];
    __shared__ long long si[SF_THREADS];
    double* row = F + (int64_t)blockIdx.x * ld;
    uint64_t bk = ~0ull;
    long long bi = -1;
    for (int64_t i = threadIdx.x; i < m; i += SF_THREADS) {
        const double v = row[i] + mu[i];
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
        idx[blockIdx.x] = si[0];
        val[blockIdx.x] = row[si[0]];
    }
}

}  // namespace abo

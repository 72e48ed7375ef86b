// gemm_dmma.cuh — FP64 tensor-core (DMMA.8x8x4) GEMMs staged by cp.async:
//   gemm_dmma_kernel                       MN-contiguous operands: Z = L^-T W of the acquisition gradient
//                                          (abo_acq_eval_grad), G = W^T W of the posterior covariance;
//   gemm_small_kernel, gemm_k128_kernel    K-contiguous operands: the panel TRSM / SYRK of the look-ahead Cholesky.
// (The candidate sweep, the trailing updates, the batched Cholesky, the triangular inverse and K^-1 = L^-T L^-1 run
// on the TMA/mbarrier pipeline of tma_pipe.cuh (gemm_tma.cuh, sweep_fused.cuh), which shares the shared-memory tile
// layout and the DMMA inner loop.)
//
// tcgen05 has no f64 kind, so on sm_100a FP64 tensor work is the warp-level
// mma.sync.m8n8k4.f64 (SASS DMMA.8x8x4; the m16n8k{4,8,16} PTX shapes lower to the same SASS
// instruction).  Measured issue peak on this pool: 36.9 TFLOP/s (profiles/fp64_peaks_r01.json).
//
// gemm_dmma_kernel: CTA tile 128 x 128, K step 16, 256 threads = 8 warps (4 along M x 2 along N), warp
// tile 32 x 64 = 4 x 8 DMMA tiles (64 accumulator doubles / thread), 4-stage cp.async pipeline.
// Shared-memory tiles are laid out so that every fragment load is conflict-free:
//   K-contiguous operand (element (r,k) at r*ld + k in HBM)  -> smem [k/4][r][k%4]
//        a fragment (8 rows x 4 k) is one 256-byte contiguous run
//   MN-contiguous operand (element (r,k) at k*ld + r in HBM) -> smem [k][132]
//        ld = 132 = 4 (mod 16) spreads the four k-rows of a fragment over distinct banks
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace abo {

constexpr int BM = 128, BN = 128, BK = 16, STAGES = 4, GEMM_THREADS = 256;
constexpr int TILE_DOUBLES = 16 * 132;   // per operand per stage: [k][132]
constexpr int GEMM_SMEM_BYTES = STAGES * 2 * TILE_DOUBLES * (int)sizeof(double);

enum GemmFlags {
    KLO_M = 1,        // k starts at the tile's first row      (A^T-type lower operands)
    KLO_N = 2,        // k starts at the tile's first column   (B lower triangular, k >= n)
    KHI_M = 4,        // k stops after the tile's last row     (A lower triangular, k <= m)
    LOWER_ONLY = 8,   // skip tiles strictly above the diagonal
    SKIP_FIRST = 16   // leave out the first 128 x 128 tile of C (updated elsewhere)
};

struct GemmParams {
    const double* A; const double* B; double* C;
    int64_t lda, ldb, ldc;
    int64_t strideA, strideB, strideC;   // per blockIdx.z
    int M, N, K;                         // multiples of 128 / 128 / 16
    double alpha, beta;
    int flags;
    int lower_shift;                     // LOWER_ONLY keeps tiles with n0 <= m0 + lower_shift (C starts lower_shift rows below the diagonal)
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// programmatic dependent launch (PDL): let the next kernel of the stream get resident early, and
// wait for the previous kernel's results before touching global memory.  Both are no-ops for a
// kernel launched without the programmatic-serialization attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }

__device__ __forceinline__ void dmma8x8x4(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// one 128 x 16 tile of an MN-contiguous operand -> smem, 4 x 16-byte cp.async per thread
__device__ __forceinline__ void load_tile(double* s, const double* g, int64_t ld, int r0, int k0, int tid) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        int c = tid + GEMM_THREADS * q;
        int krow = c >> 6, ch = c & 63;                      // 64 chunks per k-row
        const double* src = g + (int64_t)(k0 + krow) * ld + r0 + 2 * ch;
        double* dst = s + krow * 132 + 2 * ch;
        cp_async16(dst, src);
    }
}

__device__ __forceinline__ double frag(const double* s, int kk, int r, int lane) {
    // element (row = r + lane/4, k = 4*kk + lane%4)
    return s[(kk * 4 + (lane & 3)) * 132 + r + (lane >> 2)];
}

// C = alpha * A^T B + beta * C  with A[k][m] at A + k lda + m and B[k][n] at B + k ldb + n
__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_dmma_kernel(GemmParams p) {
    extern __shared__ __align__(16) double smem[];
    double* sA = smem;
    double* sB = smem + STAGES * TILE_DOUBLES;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp & 3) * 32, wn = (warp >> 2) * 64;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    if ((p.flags & LOWER_ONLY) && n0 > m0) return;

    const double* A = p.A + (int64_t)blockIdx.z * p.strideA;
    const double* B = p.B + (int64_t)blockIdx.z * p.strideB;

    int klo = 0, khi = p.K;
    if (p.flags & KLO_M) klo = m0;
    if ((p.flags & KLO_N) && n0 > klo) klo = n0;
    if ((p.flags & KHI_M) && m0 + BM < khi) khi = m0 + BM;
    const int nk = (khi > klo) ? (khi - klo) / BK : 0;

    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < nk) {
            load_tile(sA + s * TILE_DOUBLES, A, p.lda, m0, klo + s * BK, tid);
            load_tile(sB + s * TILE_DOUBLES, B, p.ldb, n0, klo + s * BK, tid);
        }
        cp_async_commit();
    }

    for (int kt = 0; kt < nk; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {
            int nxt = kt + STAGES - 1;
            if (nxt < nk) {
                int s = nxt % STAGES;
                load_tile(sA + s * TILE_DOUBLES, A, p.lda, m0, klo + nxt * BK, tid);
                load_tile(sB + s * TILE_DOUBLES, B, p.ldb, n0, klo + nxt * BK, tid);
            }
            cp_async_commit();
        }
        const double* a_s = sA + (kt % STAGES) * TILE_DOUBLES;
        const double* b_s = sB + (kt % STAGES) * TILE_DOUBLES;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            double a[4], b[8];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = frag(a_s, kk, wm + i * 8, lane);
#pragma unroll
            for (int j = 0; j < 8; ++j) b[j] = frag(b_s, kk, wn + j * 8, lane);
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
    cp_async_wait<0>();

    double* C = p.C + (int64_t)blockIdx.z * p.strideC;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int row = m0 + wm + i * 8 + (lane >> 2);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int col = n0 + wn + j * 8 + 2 * (lane & 3);
            double2* dst = reinterpret_cast<double2*>(C + (int64_t)row * p.ldc + col);
            double2 v;
            v.x = p.alpha * acc[i][j][0];
            v.y = p.alpha * acc[i][j][1];
            if (p.beta != 0.0) {
                double2 o = *dst;
                v.x += p.beta * o.x;
                v.y += p.beta * o.y;
            }
            *dst = v;
        }
    }
}

// ------------------------------------------------------------------------------------------
// BMT x 128 tile variants (BMT = 64 or 32; K-contiguous operands, store epilogue) for the
// latency-critical panel operations of the Cholesky (TRSM-as-GEMM and the in-block SYRK,
// K = 128): 2x / 4x as many CTAs, half / quarter of the time per tile.
// 8 warps as (BMT/32) along M x (256/BMT) along N, warp tile 32 x (BMT/2).
// ------------------------------------------------------------------------------------------
template <int BMT, int NW>
struct GemmS {
    static constexpr int THREADS = NW * 32;
    static constexpr int WM = BMT / 32, WN = NW / WM, WNC = 128 / WN, NT = WNC / 8;
    static constexpr int A_DOUBLES = 4 * BMT * 4, B_DOUBLES = 4 * 128 * 4;
    static constexpr int SMEM_BYTES = STAGES * (A_DOUBLES + B_DOUBLES) * (int)sizeof(double);
};

// NW = 4 warps keeps a 32-row CTA at 128 threads / <= 16K registers / 80 KB shared memory, small
// enough to be co-resident with a trailing-update CTA of the look-ahead stream on the same SM.
template <int BMT, int NW>
__global__ void __launch_bounds__(NW * 32, NW == 4 ? 4 : 2) gemm_small_kernel(GemmParams p) {
    using S = GemmS<BMT, NW>;
    extern __shared__ __align__(16) double smem[];
    double* sA = smem;
    double* sB = smem + STAGES * S::A_DOUBLES;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = (warp % S::WM) * 32, wn = (warp / S::WM) * S::WNC;
    const int m0 = blockIdx.y * BMT, n0 = blockIdx.x * BN;
    pdl_launch_dependents();
    if ((p.flags & LOWER_ONLY) && n0 > m0 + p.lower_shift) return;
    if ((p.flags & SKIP_FIRST) && m0 < 128 && n0 == 0) return;
    const double* A = p.A + (int64_t)blockIdx.z * p.strideA;
    const double* B = p.B + (int64_t)blockIdx.z * p.strideB;
    const int nk = p.K / BK;
    pdl_wait();

    double acc[4][S::NT][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < S::NT; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

    auto load_stage = [&](int s, int kt) {
        const int k0 = kt * BK;
#pragma unroll
        for (int q = 0; q < BMT * 8 / S::THREADS; ++q) {   // A: BMT rows x 8 chunks of 16 B
            int c = tid + S::THREADS * q, row = c >> 3, ch = c & 7;
            cp_async16(sA + s * S::A_DOUBLES + (((ch >> 1) * BMT + row) << 2) + ((ch & 1) << 1),
                       A + (int64_t)(m0 + row) * p.lda + k0 + 2 * ch);
        }
#pragma unroll
        for (int q = 0; q < 1024 / S::THREADS; ++q) {      // B: 128 rows x 8 chunks
            int c = tid + S::THREADS * q, row = c >> 3, ch = c & 7;
            cp_async16(sB + s * S::B_DOUBLES + (((ch >> 1) * 128 + row) << 2) + ((ch & 1) << 1),
                       B + (int64_t)(n0 + row) * p.ldb + k0 + 2 * ch);
        }
    };
#pragma unroll
    for (int s = 0; s < STAGES - 1; ++s) {
        if (s < nk) load_stage(s, s);
        cp_async_commit();
    }
    for (int kt = 0; kt < nk; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {
            int nxt = kt + STAGES - 1;
            if (nxt < nk) load_stage(nxt % STAGES, nxt);
            cp_async_commit();
        }
        const double* a_s = sA + (kt % STAGES) * S::A_DOUBLES;
        const double* b_s = sB + (kt % STAGES) * S::B_DOUBLES;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            double a[4], b[S::NT];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = a_s[((kk * BMT + wm + i * 8 + (lane >> 2)) << 2) + (lane & 3)];
#pragma unroll
            for (int j = 0; j < S::NT; ++j) b[j] = b_s[((kk * 128 + wn + j * 8 + (lane >> 2)) << 2) + (lane & 3)];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < S::NT; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
    cp_async_wait<0>();
    double* C = p.C + (int64_t)blockIdx.z * p.strideC;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int row = m0 + wm + i * 8 + (lane >> 2);
#pragma unroll
        for (int j = 0; j < S::NT; ++j) {
            int col = n0 + wn + j * 8 + 2 * (lane & 3);
            double2* dst = reinterpret_cast<double2*>(C + (int64_t)row * p.ldc + col);
            double2 v;
            v.x = p.alpha * acc[i][j][0];
            v.y = p.alpha * acc[i][j][1];
            if (p.beta != 0.0) {
                double2 o = *dst;
                v.x += p.beta * o.x;
                v.y += p.beta * o.y;
            }
            *dst = v;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Latency kernels for the two GEMMs on the critical chain of the Cholesky (next diagonal tile: TRSM-as-GEMM and
// its SYRK, M = N = K = 128): small TM x TN output tiles -> 8 / 16 CTAs of 4 warps, the whole k-range staged by
// ONE cp.async group, no pipeline to fill or drain.  K-contiguous operands, store epilogue.
//   <16, 128>: a CTA owns whole rows, so C may alias A (the in-place TRSM)      <32, 32>: the SYRK of the tile
// ------------------------------------------------------------------------------------------
template <int TM, int TN>
struct GemmK128 {
    static constexpr int WM = TM / 16, WN = 4 / WM, WNC = TN / WN, NT = WNC / 8;
    static constexpr int SMEM_BYTES = 32 * (TM + TN) * 4 * (int)sizeof(double);
};
template <int TM, int TN>
__global__ void __launch_bounds__(128) gemm_k128_kernel(GemmParams p) {
    using S = GemmK128<TM, TN>;
    extern __shared__ __align__(16) double smem[];
    double* sA = smem;
    double* sB = smem + 32 * TM * 4;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
    pdl_launch_dependents();
    pdl_wait();
    const int wm = (warp % S::WM) * 16, wn = (warp / S::WM) * S::WNC;
    double acc[2][S::NT][2];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < S::NT; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
    for (int k0 = 0; k0 < p.K; k0 += 128) {            // K = 128 on the inner chain, up to the outer block width at its end
        if (k0) __syncthreads();
#pragma unroll
        for (int q = 0; q < TM * 64 / 128; ++q) {      // TM rows x 64 chunks of 16 B
            const int c = tid + 128 * q, row = c >> 6, ch = c & 63;
            cp_async16(sA + ((((ch >> 1) * TM + row) << 2) + ((ch & 1) << 1)), p.A + (int64_t)(m0 + row) * p.lda + k0 + 2 * ch);
        }
#pragma unroll 8
        for (int q = 0; q < TN * 64 / 128; ++q) {
            const int c = tid + 128 * q, row = c >> 6, ch = c & 63;
            cp_async16(sB + ((((ch >> 1) * TN + row) << 2) + ((ch & 1) << 1)), p.B + (int64_t)(n0 + row) * p.ldb + k0 + 2 * ch);
        }
        cp_async_commit();
        cp_async_wait<0>();
        __syncthreads();
#pragma unroll 4
        for (int kk = 0; kk < 32; ++kk) {
            double a[2], b[S::NT];
#pragma unroll
            for (int i = 0; i < 2; ++i) a[i] = sA[((kk * TM + wm + i * 8 + (lane >> 2)) << 2) + (lane & 3)];
#pragma unroll
            for (int j = 0; j < S::NT; ++j) b[j] = sB[((kk * TN + wn + j * 8 + (lane >> 2)) << 2) + (lane & 3)];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int j = 0; j < S::NT; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < S::NT; ++j) {
            double2* dst = reinterpret_cast<double2*>(p.C + (int64_t)(m0 + wm + i * 8 + (lane >> 2)) * p.ldc + n0 + wn + j * 8 + 2 * (lane & 3));
            double2 v;
            v.x = p.alpha * acc[i][j][0];
            v.y = p.alpha * acc[i][j][1];
            if (p.beta != 0.0) { const double2 o = *dst; v.x += p.beta * o.x; v.y += p.beta * o.y; }
            *dst = v;
        }
}

inline cudaError_t launch_gemm(const GemmParams& p, int batch, cudaStream_t st) {
    if (p.M <= 0 || p.N <= 0 || batch <= 0) return cudaSuccess;
    dim3 grid(p.N / BN, p.M / BM, batch);
    gemm_dmma_kernel<<<grid, GEMM_THREADS, GEMM_SMEM_BYTES, st>>>(p);
    return cudaGetLastError();
}

}  // namespace abo

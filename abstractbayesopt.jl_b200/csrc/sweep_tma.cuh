// sweep_tma.cuh — the hot kernel of the candidate sweep, second generation:
//     partial[ib][c] = sum over the 128 rows of tile ib of ( L^-1[ib rows, 0:k_hi] * K*[c, 0:k_hi]^T )^2
// i.e. the posterior-variance contraction  ||L^-1 k*||^2  (StandardGP.jl:377-379 via AbstractGPs
// diag_Xt_invA_X) as a triangular FP64 tensor-core product with a fused sum-of-squares epilogue.
//
// Persistent, warp-specialised:
//   * one CTA per SM, static serpentine tile schedule, heaviest (largest ib) tiles first;
//   * warp 8 = TMA producer: cp.async.bulk.tensor.2d boxes of 4 (k) x 128 (rows) doubles land in
//     shared memory as [k/4][row][4] — every DMMA fragment (8 rows x 4 k) is then one 256-byte
//     contiguous, bank-conflict-free run; completion is signalled on an mbarrier ring
//     (full/empty, NSTAGE stages of 32 KB), so the producer runs ahead across tile boundaries;
//   * warps 0..7 = DMMA consumers (4 along M x 2 along N, warp tile 32 x 64), fragments
//     double-buffered in registers, no block-wide barrier inside the k loop.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

#include "gemm_dmma.cuh"

namespace abo {

constexpr int SW_STAGES = 5;
constexpr int SW_CONSUMERS = 256;
constexpr int SW_THREADS = SW_CONSUMERS + 32;
constexpr int SW_OPER_DOUBLES = 4 * 128 * 4;                       // one operand, one stage: 16 KB
constexpr int SW_STAGE_BYTES = 2 * SW_OPER_DOUBLES * 8;            // 32 KB
constexpr int SW_SMEM_BYTES = SW_STAGES * SW_STAGE_BYTES + 4 * 128 * 8 + 2 * SW_STAGES * 8 + 128;

struct SweepParams {
    int T;              // row tiles of L^-1 (Npad / 128)
    int ncb;            // candidate tiles in this launch
    double* sumsq;      // [T][sumsq_ld]
    int64_t sumsq_ld;
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::
            "r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}

// tile t of the launch (heaviest first): ib = T-1 - t / ncb, cb = t % ncb
// CTA b processes rounds r = 0,1,...: t = r*G + (r odd ? G-1-b : b)   (serpentine: balances the
// triangular work to within one round's spread without any dynamic scheduling)
__device__ __forceinline__ int sweep_tile(int r, int b, int G) { return r * G + ((r & 1) ? (G - 1 - b) : b); }

__global__ void __launch_bounds__(SW_THREADS, 1)
sweep_tma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, SweepParams p) {
    extern __shared__ __align__(128) unsigned char sw_smem[];
    double* stage_base = reinterpret_cast<double*>(sw_smem);
    double* red = reinterpret_cast<double*>(sw_smem + SW_STAGES * SW_STAGE_BYTES);          // [4][128]
    uint64_t* full = reinterpret_cast<uint64_t*>(sw_smem + SW_STAGES * SW_STAGE_BYTES + 4 * 128 * 8);
    uint64_t* empty = full + SW_STAGES;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = gridDim.x, b = blockIdx.x;
    const int ntiles = p.T * p.ncb;

    if (tid == 0) {
        for (int s = 0; s < SW_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    if (warp == 8) {
        // ------------------------------ TMA producer ------------------------------
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int r = 0;; ++r) {
                const int t = sweep_tile(r, b, G);
                if (t >= ntiles) { if (r * G >= ntiles) break; else continue; }
                const int ib = p.T - 1 - t / p.ncb, cb = t % p.ncb;
                const int m0 = ib * 128, n0 = cb * 128;
                const int nk = (ib + 1) * 8;
                for (int kt = 0; kt < nk; ++kt) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    mbar_expect_tx(&full[stage], SW_STAGE_BYTES);
                    double* sa = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES);
                    double* sb = sa + SW_OPER_DOUBLES;
                    const int k0 = kt * 16;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        tma_load_2d(sa + q * 512, &tmA, k0 + 4 * q, m0, &full[stage]);
                        tma_load_2d(sb + q * 512, &tmB, k0 + 4 * q, n0, &full[stage]);
                    }
                    if (++stage == SW_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
        return;
    }

    // ------------------------------ DMMA consumers ------------------------------
    const int wm = (warp & 3) * 32, wn = (warp >> 2) * 64;
    const int fr = lane >> 2, fk = lane & 3;
    int stage = 0;
    uint32_t phase = 0;
    for (int r = 0;; ++r) {
        const int t = sweep_tile(r, b, G);
        if (t >= ntiles) { if (r * G >= ntiles) break; else continue; }
        const int ib = p.T - 1 - t / p.ncb, cb = t % p.ncb;
        const int nk = (ib + 1) * 8;

        double acc[4][8][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

        for (int kt = 0; kt < nk; ++kt) {
            mbar_wait(&full[stage], phase);
            const double* a_s = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES) + ((wm + fr) << 2) + fk;
            const double* b_s = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES) + SW_OPER_DOUBLES + ((wn + fr) << 2) + fk;
            double a[2][4], bb[2][8];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[0][i] = a_s[i * 32];
#pragma unroll
            for (int j = 0; j < 8; ++j) bb[0][j] = b_s[j * 32];
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                const int cur = kk & 1, nxt = cur ^ 1;
                if (kk < 3) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) a[nxt][i] = a_s[(kk + 1) * 512 + i * 32];
#pragma unroll
                    for (int j = 0; j < 8; ++j) bb[nxt][j] = b_s[(kk + 1) * 512 + j * 32];
                }
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 8; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[cur][i], bb[cur][j]);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == SW_STAGES) { stage = 0; phase ^= 1; }
        }

        // ---- epilogue: column sums of squares over the tile's 128 rows
#pragma unroll
        for (int j = 0; j < 8; ++j) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                double s = 0.0;
#pragma unroll
                for (int i = 0; i < 4; ++i) s = fma(acc[i][j][e], acc[i][j][e], s);
                s += __shfl_xor_sync(0xffffffffu, s, 4);
                s += __shfl_xor_sync(0xffffffffu, s, 8);
                s += __shfl_xor_sync(0xffffffffu, s, 16);
                if (fr == 0) red[(warp & 3) * 128 + wn + j * 8 + 2 * fk + e] = s;
            }
        }
        asm volatile("bar.sync 1, 256;\n" ::: "memory");       // consumer warps only
        if (tid < 128) {
            const double s = ((red[tid] + red[128 + tid]) + red[256 + tid]) + red[384 + tid];
            p.sumsq[(int64_t)ib * p.sumsq_ld + cb * 128 + tid] = s;
        }
        asm volatile("bar.sync 1, 256;\n" ::: "memory");
    }
}


// ------------------------------------------------------------------------------------------
// Trailing update of the blocked Cholesky with the same TMA / mbarrier / DMMA pipeline:
//     C[i-tile, j-tile] -= L[i rows, kcol0 : kcol0 + 16*nk] * L[j rows, same columns]^T
// for the lower tiles (j <= i) of a rectangular range of tiles.  One tile per CTA (not
// persistent) so that the higher-priority panel stream of the look-ahead schedule can slip its
// small kernels in between tiles.  A and B are both K-contiguous row panels of the SAME
// row-major matrix, hence one tensor map.
// ------------------------------------------------------------------------------------------
// same ring depth as the sweep kernel
constexpr int SY_STAGES = 5;
constexpr int SY_SMEM_BYTES = SY_STAGES * SW_STAGE_BYTES + 4 * 128 * 8 + 2 * SY_STAGES * 8 + 128;

struct SyrkParams {
    double* C;          // base of the matrix (row-major, ld)
    int64_t ld;
    int row_t0, col_t0; // first row tile / column tile of this launch's grid
    int kcol0;          // first column of the panel block
    int nk;             // k16 steps (panel width / 16)
    int skip_first;     // leave out tile (row_t0, col_t0): it was updated by the latency kernel on the critical chain
};

__global__ void __launch_bounds__(SW_THREADS, 1)
syrk_tma_kernel(const __grid_constant__ CUtensorMap tmL, SyrkParams p) {
    extern __shared__ __align__(128) unsigned char sw_smem[];
    double* stage_base = reinterpret_cast<double*>(sw_smem);
    uint64_t* full = reinterpret_cast<uint64_t*>(sw_smem + SY_STAGES * SW_STAGE_BYTES + 4 * 128 * 8);
    uint64_t* empty = full + SY_STAGES;
    const int it = p.row_t0 + blockIdx.y, jt = p.col_t0 + blockIdx.x;
    pdl_launch_dependents();
    if (jt > it || (p.skip_first && blockIdx.x == 0 && blockIdx.y == 0)) return;
    pdl_wait();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int m0 = it * 128, n0 = jt * 128;

    if (tid == 0) {
        for (int s = 0; s < SY_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();

    if (warp == 8) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int kt = 0; kt < p.nk; ++kt) {
                mbar_wait(&empty[stage], phase ^ 1);
                mbar_expect_tx(&full[stage], SW_STAGE_BYTES);
                double* sa = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES);
                double* sb = sa + SW_OPER_DOUBLES;
                const int k0 = p.kcol0 + kt * 16;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    tma_load_2d(sa + q * 512, &tmL, k0 + 4 * q, m0, &full[stage]);
                    tma_load_2d(sb + q * 512, &tmL, k0 + 4 * q, n0, &full[stage]);
                }
                if (++stage == SY_STAGES) { stage = 0; phase ^= 1; }
            }
        }
        return;
    }

    const int wm = (warp & 3) * 32, wn = (warp >> 2) * 64;
    const int fr = lane >> 2, fk = lane & 3;
    int stage = 0;
    uint32_t phase = 0;
    double acc[4][8][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }

    for (int kt = 0; kt < p.nk; ++kt) {
        mbar_wait(&full[stage], phase);
        const double* a_s = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES) + ((wm + fr) << 2) + fk;
        const double* b_s = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES) + SW_OPER_DOUBLES + ((wn + fr) << 2) + fk;
        double a[2][4], bb[2][8];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[0][i] = a_s[i * 32];
#pragma unroll
        for (int j = 0; j < 8; ++j) bb[0][j] = b_s[j * 32];
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const int cur = kk & 1, nxt = cur ^ 1;
            if (kk < 3) {
#pragma unroll
                for (int i = 0; i < 4; ++i) a[nxt][i] = a_s[(kk + 1) * 512 + i * 32];
#pragma unroll
                for (int j = 0; j < 8; ++j) bb[nxt][j] = b_s[(kk + 1) * 512 + j * 32];
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[cur][i], bb[cur][j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[stage]);
        if (++stage == SY_STAGES) { stage = 0; phase ^= 1; }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int row = m0 + wm + i * 8 + fr;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int col = n0 + wn + j * 8 + 2 * fk;
            double2* dst = reinterpret_cast<double2*>(p.C + (int64_t)row * p.ld + col);
            double2 o = *dst;
            o.x -= acc[i][j][0];
            o.y -= acc[i][j][1];
            *dst = o;
        }
    }
}


}  // namespace abo

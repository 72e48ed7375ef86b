// gemm_tma.cuh — persistent, batched FP64 tensor-core GEMM for K-CONTIGUOUS operands, fed by TMA:
//     C[m][n] (+)= alpha * sum_{k in [klo, khi)} A[m][k] * B[n][k]          (both operands row-major with k contiguous)
// with an optional TRANSPOSED second store CT[n][m] = alpha * (...) — which is what lets every O(n^3) step of the conditioning
// and of the batched marginal likelihood keep its operands k-contiguous (the triangular inverse carries X and X^T, the product
// of the inverse factors reads X^T twice), so that all of them run on the TMA + mbarrier + DMMA pipeline of tma_pipe.cuh
// instead of the cp.async kernels whose MN-contiguous shared-memory layout costs bank conflicts (ncu, round 1: 84.7 % DMMA).
// The EPI_COLSUMSQ instance is the contraction of the candidate sweep when it is not fused (GradientGP outputs, n > FS_MAX_NPAD):
//     C[mt][n] = sum over the 128 rows m of row tile mt of ( sum_k A[m][k] B[n][k] )^2
// with A = L^-1 and B = K*, i.e. the posterior-variance term ||L^-1 k*||^2 (StandardGP.jl:377-379 via AbstractGPs
// diag_Xt_invA_X) per row tile, summed over the row tiles by acq_epilogue_kernel.
//
// One CTA per SM, static serpentine schedule over (batch item, tile) work items ordered heaviest first; the producer warp runs
// ahead across item boundaries (no pipeline fill / drain per tile — the short k-loops of the batched n ~ 1000 matrices are
// exactly where that matters); k-ranges that are structurally zero are skipped (flags as in gemm_dmma.cuh).
//
// Also here: syrk_tma_kernel, the trailing update of the blocked Cholesky on the same pipeline.
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

#include "gemm_dmma.cuh"
#include "tma_pipe.cuh"

namespace abo {

struct TmaGemmParams {
    int Mt, Nt, batch, total;                       // tiles per item, items, work items in this launch
    int K;                                          // full k extent (multiple of 16)
    int flags;                                      // KLO_M | KLO_N | KHI_M | LOWER_ONLY
    // tile origins in the 2-D tensor maps (k coordinate, row coordinate), per batch item z:
    int a_row0, a_rstep, a_col0, a_cstep;           // A rows  a_row0 + z a_rstep + m0,  k columns a_col0 + z a_cstep + k
    int b_row0, b_rstep, b_col0, b_cstep;
    double* C;  int64_t ldc,  c_off0,  c_zstep;     // C  element (m, n): C [c_off0  + z c_zstep  + m ldc  + n]   (nullable)
    double* CT; int64_t ldct, ct_off0, ct_zstep;    // CT element (n, m): CT[ct_off0 + z ct_zstep + n ldct + m]   (nullable, beta = 0)
    double alpha, beta;                             // EPI_COLSUMSQ: C[mt ldc + n] = column sums of squares of tile (mt, nt);
                                                    // batch 1, c_off0 / CT / alpha / beta unused
};

enum { EPI_STORE = 0, EPI_COLSUMSQ = 1 };

struct TgTile { int z, m0, n0, klo, nk; };
__device__ __forceinline__ TgTile tg_decode(const TmaGemmParams& p, int t) {
    TgTile w;
    w.z = t % p.batch;
    const int tl = t / p.batch;
    int mt, nt;
    if (p.flags & LOWER_ONLY) {                     // lower tiles nt <= min(mt, Nt - 1) of an Mt x Nt grid (Nt <= Mt): the triangle of
                                                    // the first Nt tile rows, then full rows of Nt tiles (a trapezoid when Nt < Mt)
        const int tri = p.Nt * (p.Nt + 1) / 2;
        if (tl < tri) {
            mt = (int)((sqrt(8.0 * tl + 1.0) - 1.0) * 0.5);
            while ((mt + 1) * (mt + 2) / 2 <= tl) ++mt;
            while (mt * (mt + 1) / 2 > tl) --mt;
            nt = tl - mt * (mt + 1) / 2;
        } else { mt = p.Nt + (tl - tri) / p.Nt; nt = (tl - tri) % p.Nt; }
    } else if (p.flags & KLO_N) { nt = tl / p.Mt; mt = tl % p.Mt; }
    else if (p.flags & KHI_M) { mt = p.Mt - 1 - tl / p.Nt; nt = tl % p.Nt; }
    else { mt = tl / p.Nt; nt = tl % p.Nt; }
    w.m0 = mt * 128; w.n0 = nt * 128;
    int klo = 0, khi = p.K;
    if (p.flags & KLO_M) klo = w.m0;
    if ((p.flags & KLO_N) && w.n0 > klo) klo = w.n0;
    if ((p.flags & KHI_M) && w.m0 + 128 < khi) khi = w.m0 + 128;
    w.klo = klo;
    w.nk = (khi > klo) ? (khi - klo) / 16 : 0;
    return w;
}

// shared memory: the stage ring, the [4][128] column-sum buffer of EPI_COLSUMSQ, the barriers
template <int EPI> __host__ __device__ constexpr int tg_red_bytes() { return EPI == EPI_COLSUMSQ ? 4 * 128 * 8 : 0; }
template <int EPI> constexpr int tg_smem_bytes() { return SW_STAGES * SW_STAGE_BYTES + tg_red_bytes<EPI>() + 2 * SW_STAGES * 8 + 128; }

template <int EPI>
__global__ void __launch_bounds__(SW_THREADS, 1)
gemm_tma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TmaGemmParams p) {
    extern __shared__ __align__(128) unsigned char tg_smem[];
    double* stage_base = reinterpret_cast<double*>(tg_smem);
    double* red = reinterpret_cast<double*>(tg_smem + SW_STAGES * SW_STAGE_BYTES);
    uint64_t* full = reinterpret_cast<uint64_t*>(tg_smem + SW_STAGES * SW_STAGE_BYTES + tg_red_bytes<EPI>());
    uint64_t* empty = full + SW_STAGES;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = gridDim.x, b = blockIdx.x;
    if (tid == 0) {
        for (int s = 0; s < SW_STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 8); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();
    // work item r of this CTA: serpentine over the launch's item list
    auto item_of = [&](int r) { return r * G + ((r & 1) ? (G - 1 - b) : b); };

    if (warp == 8) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int r = 0;; ++r) {
                const int t = item_of(r);
                if (t >= p.total) { if (r * G >= p.total) break; else continue; }
                const TgTile w = tg_decode(p, t);
                const int arow = p.a_row0 + w.z * p.a_rstep + w.m0, acol = p.a_col0 + w.z * p.a_cstep + w.klo;
                const int brow = p.b_row0 + w.z * p.b_rstep + w.n0, bcol = p.b_col0 + w.z * p.b_cstep + w.klo;
                for (int kt = 0; kt < w.nk; ++kt) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    tma_stage_load(stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES), &full[stage], &tmA, acol + kt * 16, arow,
                                   &tmB, bcol + kt * 16, brow);
                    if (++stage == SW_STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
        return;
    }

    const int wm = (warp & 3) * 32, wn = (warp >> 2) * 64;
    const int fr = lane >> 2, fk = lane & 3;
    int stage = 0;
    uint32_t phase = 0;
    for (int r = 0;; ++r) {
        const int t = item_of(r);
        if (t >= p.total) { if (r * G >= p.total) break; else continue; }
        const TgTile w = tg_decode(p, t);
        double acc[4][8][2];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) { acc[i][j][0] = 0.0; acc[i][j][1] = 0.0; }
        for (int kt = 0; kt < w.nk; ++kt) {
            mbar_wait(&full[stage], phase);
            const double* st = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES);
            dmma_stage<0, 4, 32>(st + ((wm + fr) << 2) + fk, st + SW_OPER_DOUBLES + ((wn + fr) << 2) + fk, acc);
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == SW_STAGES) { stage = 0; phase ^= 1; }
        }
        // ---- epilogue
        if (EPI == EPI_COLSUMSQ) {
            // column sums of squares over the tile's 128 rows: the warp's 32 rows in registers and shuffles, then the four row
            // warps in a fixed order
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
                p.C[(int64_t)(w.m0 / 128) * p.ldc + w.n0 + tid] = s;
            }
            asm volatile("bar.sync 1, 256;\n" ::: "memory");
            continue;
        }
        if (p.C) {
            double* C = p.C + p.c_off0 + (int64_t)w.z * p.c_zstep;
            if (p.beta != 0.0) {
                // read-modify-write: the eight loads of a fragment row go out together (one global-memory latency per row group
                // instead of one per element: with stores in between the compiler must keep the loads in program order)
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int row = w.m0 + wm + i * 8 + fr;
                    double2* dst = reinterpret_cast<double2*>(C + (int64_t)row * p.ldc + w.n0 + wn + 2 * fk);
                    double2 o[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) o[j] = dst[j * 4];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        o[j].x = fma(p.beta, o[j].x, p.alpha * acc[i][j][0]);
                        o[j].y = fma(p.beta, o[j].y, p.alpha * acc[i][j][1]);
                        dst[j * 4] = o[j];
                    }
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int row = w.m0 + wm + i * 8 + fr;
                    double2* dst = reinterpret_cast<double2*>(C + (int64_t)row * p.ldc + w.n0 + wn + 2 * fk);
#pragma unroll
                    for (int j = 0; j < 8; ++j) dst[j * 4] = make_double2(p.alpha * acc[i][j][0], p.alpha * acc[i][j][1]);
                }
            }
        }
        if (p.CT) {
            // transposed copy: a lane owns (row fr, columns 2 fk, 2 fk + 1) of an 8 x 8 fragment -> two 8-byte stores into two
            // rows of CT; the eight lanes of equal fk write 64 contiguous bytes (rows fr = 0..7 of the source)
            double* CT = p.CT + p.ct_off0 + (int64_t)w.z * p.ct_zstep;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int row = w.m0 + wm + i * 8 + fr;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int col = w.n0 + wn + j * 8 + 2 * fk;
                    CT[(int64_t)col * p.ldct + row] = p.alpha * acc[i][j][0];
                    CT[(int64_t)(col + 1) * p.ldct + row] = p.alpha * acc[i][j][1];
                }
            }
        }
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
// same ring depth as gemm_tma_kernel
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
                const int k0 = p.kcol0 + kt * 16;
                tma_stage_load(stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES), &full[stage], &tmL, k0, m0, &tmL, k0, n0);
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
        const double* st = stage_base + (size_t)stage * (2 * SW_OPER_DOUBLES);
        dmma_stage<0, 4, 32>(st + ((wm + fr) << 2) + fk, st + SW_OPER_DOUBLES + ((wn + fr) << 2) + fk, acc);
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

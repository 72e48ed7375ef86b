// tma_pipe.cuh — the TMA / mbarrier / DMMA pipeline shared by the FP64 tensor kernels (gemm_tma_kernel, syrk_tma_kernel,
// sweep_fused_kernel):
//   * one producer warp (warp 8) issues cp.async.bulk.tensor.2d boxes of 4 (k) x 128 (rows) doubles, which land in shared
//     memory as [k/4][row][4] — every DMMA fragment (8 rows x 4 k) is then one 256-byte contiguous, bank-conflict-free run;
//     completion is signalled on a ring of full / empty mbarriers (stages of 32 KB: a 128 x 16 slab of each operand), so the
//     producer runs ahead of the consumers;
//   * eight DMMA consumer warps (warps 0..7) each contract a stage into a 32 x 64 accumulator tile with fragments
//     double-buffered in registers, and release the stage with one arrive per warp (empty barriers count 8); no block-wide
//     barrier inside the k loop.
// The ring loop itself (wait full -> dmma_stage -> __syncwarp -> arrive empty -> advance) is written out in each kernel.
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

// Producer: fill stage `st` (A slab, then B slab) with k columns [ka, ka + 16) of A rows [arow, arow + 128) and k columns
// [kb, kb + 16) of B rows [brow, brow + 128); `full` completes when all SW_STAGE_BYTES have landed.
__device__ __forceinline__ void tma_stage_load(double* st, uint64_t* full, const CUtensorMap* tmA, int ka, int arow,
                                               const CUtensorMap* tmB, int kb, int brow) {
    mbar_expect_tx(full, SW_STAGE_BYTES);
    double* sb = st + SW_OPER_DOUBLES;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        tma_load_2d(st + q * 512, tmA, ka + 4 * q, arow, full);
        tma_load_2d(sb + q * 512, tmB, kb + 4 * q, brow, full);
    }
}

// Consumer: one k16 stage, acc[i][j] += A fragment i x B fragment j^T for the row fragments ILO <= i < IHI.  a_s / b_s point
// at this lane's first A / B element of the stage; A fragment i sits ASTRIDE doubles after fragment i - 1 (32: the warp's rows
// are contiguous, 128: fragments interleaved across the four row warps), B fragment j at 32 j.  The range is compile-time so
// that every partial range is straight-line code (a run-time predicate inside the unrolled loops cost as much as the DMMAs
// it skipped).
template <int ILO, int IHI, int ASTRIDE>
__device__ __forceinline__ void dmma_stage(const double* __restrict__ a_s, const double* __restrict__ b_s, double (&acc)[4][8][2]) {
    double a[2][4], bb[2][8];
#pragma unroll
    for (int i = ILO; i < IHI; ++i) a[0][i] = a_s[i * ASTRIDE];
#pragma unroll
    for (int j = 0; j < 8; ++j) bb[0][j] = b_s[j * 32];
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
        const int cur = kk & 1, nxt = cur ^ 1;
        if (kk < 3) {
#pragma unroll
            for (int i = ILO; i < IHI; ++i) a[nxt][i] = a_s[(kk + 1) * 512 + i * ASTRIDE];
#pragma unroll
            for (int j = 0; j < 8; ++j) bb[nxt][j] = b_s[(kk + 1) * 512 + j * 32];
        }
#pragma unroll
        for (int i = ILO; i < IHI; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) dmma8x8x4(acc[i][j][0], acc[i][j][1], a[cur][i], bb[cur][j]);
    }
}

}  // namespace abo

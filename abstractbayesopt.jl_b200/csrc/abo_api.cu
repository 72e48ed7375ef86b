// abo_api.cu — C ABI of libabo_cuda.so (include/abo.h): handles, host drivers of the blocked
// Cholesky / triangular inverse / candidate sweep, top-k selection, joint and pathwise posterior sampling.  No CPU fallback anywhere:
// every entry point needs a live CUDA device.
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <limits>
#include <new>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/abo.h"
#include "gemm_dmma.cuh"
#include "kernels.cuh"
#include "sweep_fused.cuh"
#include "gemm_tma.cuh"
#include "sample.cuh"
#include "qei.cuh"
#include "abo_internal.h"

using namespace abo;

// ------------------------------------------------------------------------------------------
// error plumbing
// ------------------------------------------------------------------------------------------
static thread_local std::string g_err;

int abo_fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

extern "C" const char* abo_last_error(void) { return g_err.c_str(); }
extern "C" int32_t abo_version(void) { return 100; }

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
static int configure_kernels() {
    CU(cudaFuncSetAttribute(gemm_dmma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
    CU(cudaFuncSetAttribute(gemm_small_kernel<32, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmS<32, 8>::SMEM_BYTES));
    CU(cudaFuncSetAttribute(gemm_small_kernel<64, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmS<64, 8>::SMEM_BYTES));
    CU(cudaFuncSetAttribute(gemm_k128_kernel<16, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmK128<16, 128>::SMEM_BYTES));
    CU(cudaFuncSetAttribute(gemm_k128_kernel<32, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmK128<32, 32>::SMEM_BYTES));
    CU(cudaFuncSetAttribute(fill_distance_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 256 * 96 * 8));
    CU(cudaFuncSetAttribute(potf2_ws_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PW_SMEM_BYTES));
    CU(cudaFuncSetAttribute(syrk_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SY_SMEM_BYTES));
    CU(cudaFuncSetAttribute(gemm_tma_kernel<EPI_STORE>, cudaFuncAttributeMaxDynamicSharedMemorySize, tg_smem_bytes<EPI_STORE>()));
    CU(cudaFuncSetAttribute(gemm_tma_kernel<EPI_COLSUMSQ>, cudaFuncAttributeMaxDynamicSharedMemorySize, tg_smem_bytes<EPI_COLSUMSQ>()));
#define ABO_FS_CFG(DT) CU(cudaFuncSetAttribute(sweep_fused_kernel<DT>, cudaFuncAttributeMaxDynamicSharedMemorySize, fused_smem_bytes<DT>())); \
    CU(cudaFuncSetAttribute(sweep_fused_kernel<DT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, fused_smem_bytes<DT>()))
    ABO_FS_CFG(4); ABO_FS_CFG(8); ABO_FS_CFG(12); ABO_FS_CFG(16); ABO_FS_CFG(20); ABO_FS_CFG(24); ABO_FS_CFG(32);
#undef ABO_FS_CFG
    return ABO_OK;
}

static int ctx_init_resources(abo_ctx* c) {
    int prio_lo = 0, prio_hi = 0;
    CU(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    CU(cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_hi));    // main / panel stream
    CU(cudaStreamCreateWithPriority(&c->stream2, cudaStreamNonBlocking, prio_lo));   // look-ahead trailing updates
    CU(cudaStreamCreateWithPriority(&c->stream3, cudaStreamNonBlocking, prio_hi));   // bulk half of the panel chain / copy stream
    CU(cudaStreamCreateWithPriority(&c->stream4, cudaStreamNonBlocking, prio_lo));   // early part of the triangular inverse
    CU(cudaEventCreateWithFlags(&c->ev_inv, cudaEventDisableTiming));
    for (int q = 0; q < 3; ++q) CU(cudaEventCreateWithFlags(&c->ev_p[q], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_a, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c->ev_b, cudaEventDisableTiming));
    for (int q = 0; q < 2; ++q) {
        CU(cudaEventCreateWithFlags(&c->ev_h2d[q], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c->ev_pc[q], cudaEventDisableTiming));
    }
    return configure_kernels();
}

extern "C" int32_t abo_ctx_create(int32_t device, abo_ctx** out) {
    if (!out) return abo_fail(ABO_ERR_INVALID, "abo_ctx_create: out is NULL");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return abo_fail(ABO_ERR_CUDA, "no CUDA device available (%s); libabo_cuda has no CPU fallback",
                        e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return abo_fail(ABO_ERR_INVALID, "device %d out of range [0,%d)", device, ndev);
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return abo_fail(ABO_ERR_CUDA, "device %d is sm_%d%d; libabo_cuda is built for sm_100a only", device, prop.major,
                        prop.minor);
    abo_ctx* c = new (std::nothrow) abo_ctx();
    if (!c) return abo_fail(ABO_ERR_ALLOC, "host allocation failed");
    c->device = device;
    c->sms = prop.multiProcessorCount;
    int rc = ctx_init_resources(c);
    if (rc) { abo_ctx_destroy(c); return rc; }           // streams / events created so far are released (last error kept)
    *out = c;
    return ABO_OK;
}

static void gp_free_device(abo_gp* g);
// every stream of the context: workspace slots and caller buffers may be in use on any of them
void ctx_sync_all(abo_ctx* c) {
    for (cudaStream_t s_ : {c->stream, c->stream2, c->stream3, c->stream4}) if (s_) cudaStreamSynchronize(s_);
}

extern "C" int32_t abo_ctx_destroy(abo_ctx* c) {
    if (!c) return ABO_OK;
    const std::string keep = g_err;                      // a failing abo_ctx_create reports ITS error, not a teardown one
    cudaSetDevice(c->device);
    ctx_sync_all(c);
    for (abo_gp* g : c->live) { gp_free_device(g); g->ctx = nullptr; }   // orphaned: only abo_gp_destroy is valid on them
    c->live.clear();
    for (auto& b : c->ws) if (b.ptr) cudaFree(b.ptr);
    gp_pool_clear(c);
    for (auto e : c->prof_events) cudaEventDestroy(e);
    if (c->pinned) cudaFreeHost(c->pinned);
    abo_nccl_teardown(c);
    auto ev_free = [](cudaEvent_t e) { if (e) cudaEventDestroy(e); };
    ev_free(c->ev_a); ev_free(c->ev_b);
    for (int q = 0; q < 2; ++q) { ev_free(c->ev_h2d[q]); ev_free(c->ev_pc[q]); }
    for (cudaStream_t s_ : {c->stream, c->stream2, c->stream3, c->stream4}) if (s_) cudaStreamDestroy(s_);
    ev_free(c->ev_inv);
    for (int q = 0; q < 3; ++q) ev_free(c->ev_p[q]);
    cudaGetLastError();
    delete c;
    g_err = keep;
    return ABO_OK;
}

// release every cached device buffer of the context (pooled posterior sets, workspaces, pinned staging)
extern "C" int32_t abo_ctx_trim(abo_ctx* c) {
    if (!c) return abo_fail(ABO_ERR_INVALID, "null ctx");
    CU(cudaSetDevice(c->device));
    ctx_sync_all(c);
    gp_pool_clear(c);
    for (auto& b : c->ws) if (b.ptr) { cudaFree(b.ptr); b.ptr = nullptr; b.bytes = 0; }
    if (c->pinned) { cudaFreeHost(c->pinned); c->pinned = nullptr; c->pinned_bytes = 0; }
    return ABO_OK;
}

extern "C" int32_t abo_ctx_device(const abo_ctx* c, int32_t* device) {
    if (!c || !device) return abo_fail(ABO_ERR_INVALID, "null argument");
    *device = c->device;
    return ABO_OK;
}
extern "C" int32_t abo_ctx_stream(const abo_ctx* c, void** stream) {
    if (!c || !stream) return abo_fail(ABO_ERR_INVALID, "null argument");
    *stream = (void*)c->stream;
    return ABO_OK;
}
extern "C" int32_t abo_ctx_launch_count(const abo_ctx* c, int64_t* count) {
    if (!c || !count) return abo_fail(ABO_ERR_INVALID, "null argument");
    *count = c->launches;
    return ABO_OK;
}

// ---- per-kernel sweep timing --------------------------------------------------------------
int prof_mark(abo_ctx* c) {          // record the next event of the (start, stop) x 3 classes sequence
    if (!c->profile) return ABO_OK;
    if (c->prof_used == c->prof_events.size()) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        c->prof_events.push_back(e);
    }
    CU(cudaEventRecord(c->prof_events[c->prof_used++], c->stream));
    return ABO_OK;
}
int prof_collect(abo_ctx* c) {       // after a stream sync: fold the recorded pairs into the totals
    if (!c->profile) return ABO_OK;
    for (size_t i = 0; i + 1 < c->prof_used; i += 2) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, c->prof_events[i], c->prof_events[i + 1]));
        int cls = (int)((i / 2) % 3);
        c->prof_ms[cls] += ms;
        c->prof_n[cls] += 1;
    }
    c->prof_used = 0;
    return ABO_OK;
}
extern "C" int32_t abo_ctx_profile(abo_ctx* c, int32_t enable) {
    if (!c) return abo_fail(ABO_ERR_INVALID, "null ctx");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    c->profile = enable != 0;
    c->prof_used = 0;
    for (int i = 0; i < 3; ++i) { c->prof_ms[i] = 0; c->prof_n[i] = 0; }
    return ABO_OK;
}
extern "C" int32_t abo_ctx_profile_read(abo_ctx* c, double ms[3], int64_t launches[3]) {
    if (!c || !ms || !launches) return abo_fail(ABO_ERR_INVALID, "null argument");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    int rc = prof_collect(c);
    if (rc) return rc;
    for (int i = 0; i < 3; ++i) { ms[i] = c->prof_ms[i]; launches[i] = c->prof_n[i]; }
    return ABO_OK;
}

// ---- TMA tensor maps (driver entry point fetched through the runtime: no -lcuda link) --------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)ptr;
    }
    return fn;
}
// row-major matrix [rows][K] of doubles with leading dimension ld; box = 4 (k) x 128 (rows)
int make_tmap_k4(CUtensorMap* map, const double* base, int64_t K, int64_t rows, int64_t ld) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return abo_fail(ABO_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(double)};
    cuuint32_t box[2] = {4, 128};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, (void*)base, dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return abo_fail(ABO_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return ABO_OK;
}

extern "C" int32_t abo_debug_potf2_clocks(abo_ctx* c, int64_t out[16]) {
    if (!c || !out) return abo_fail(ABO_ERR_INVALID, "null argument");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    long long h[16];
    CU(cudaMemcpyFromSymbol(h, g_potf2_clk, sizeof h));
    for (int i = 0; i < 16; ++i) out[i] = h[i];
    return ABO_OK;
}

// grow-only workspace slots
int ws_get(abo_ctx* c, int slot, size_t bytes, void** out) {
    auto& b = c->ws[slot];
    if (b.bytes < bytes) {
        if (b.ptr) { ctx_sync_all(c); CU(cudaFree(b.ptr)); b.ptr = nullptr; b.bytes = 0; }
        cudaError_t e = cudaMalloc(&b.ptr, bytes);
        if (e != cudaSuccess) { cudaGetLastError(); return abo_fail(ABO_ERR_ALLOC, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); }
        b.bytes = bytes;
    }
    *out = b.ptr;
    return ABO_OK;
}

void ws_release(abo_ctx* c, int slot) {
    auto& b = c->ws[slot];
    if (b.ptr) { ctx_sync_all(c); cudaFree(b.ptr); b.ptr = nullptr; b.bytes = 0; }
}

int pinned_get(abo_ctx* c, size_t bytes, void** out) {
    if (c->pinned_bytes < bytes) {
        if (c->pinned) { ctx_sync_all(c); cudaFreeHost(c->pinned); c->pinned = nullptr; c->pinned_bytes = 0; }
        cudaError_t e = cudaMallocHost(&c->pinned, bytes);
        if (e != cudaSuccess) { cudaGetLastError(); return abo_fail(ABO_ERR_ALLOC, "cudaMallocHost(%zu) failed", bytes); }
        c->pinned_bytes = bytes;
    }
    *out = c->pinned;
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// blocked Cholesky (right-looking, NB = 128) of `batch` contiguously stacked matrices: potf2+inverse of the diagonal
// block (1 CTA per matrix), then panel TRSM (as a GEMM with the block inverse) and SYRK trailing update on the persistent
// TMA pipeline (both operands k-contiguous; K = 128 per step, so the missing pipeline fill / drain per tile is most of the
// gain).  A single matrix takes the same schedule, so a restart evaluated alone gives the same bits as in a batch.
// A: batch matrices, row-major, Npad x Npad (ld), matrix z at A + z Npad ld, lower triangle referenced.
// Dinv: batch x T x 128 x 128 block inverses.  info: batch ints (0 = ok).
// ------------------------------------------------------------------------------------------
int make_tmap_k4(CUtensorMap* map, const double* base, int64_t K, int64_t rows, int64_t ld);
template <int EPI = EPI_STORE>
static int launch_gemm_tma(abo_ctx* c, const CUtensorMap& tmA, const CUtensorMap& tmB, TmaGemmParams p, cudaStream_t st, int max_ctas = 0);
int potrf_blocked(abo_ctx* c, double* A, int64_t Npad, int64_t ld, double* Dinv, int* info, int batch) {
    const int T = (int)(Npad / NB);
    const int64_t strideA = Npad * ld, strideD = (int64_t)T * NB * NB;
    cudaStream_t st = c->stream;
    CUtensorMap tmA, tmD;
    int rc;
    if ((rc = make_tmap_k4(&tmA, A, Npad, (int64_t)batch * Npad, ld)) || (rc = make_tmap_k4(&tmD, Dinv, NB, (int64_t)batch * T * NB, NB)))
        return rc;
    // two-level blocking: inside an outer block of OB tile columns the SYRK touches the block's own columns only (K = 128);
    // everything to the right is updated ONCE per outer block with K = OB * 128, i.e. one read-modify-write of the trailing
    // tiles per OB panels instead of one per panel.  OB = 3 and 4 measure the same as 2 (DESIGN.md).
    constexpr int OB = 2;
    for (int jb = 0; jb < T; ++jb) {
        double* Ajj = A + (int64_t)jb * NB * (ld + 1);
        double* Dj = Dinv + (int64_t)jb * NB * NB;
        potf2_ws_kernel<<<batch, 512, PW_SMEM_BYTES, st>>>(Ajj, ld, strideA, Dj, strideD, info, jb * NB);
        KL(c);
        const int rem = (int)(Npad - (int64_t)(jb + 1) * NB);
        if (rem <= 0) break;
        const int ob0 = jb / OB * OB, obend = std::min(ob0 + OB, T);      // this panel's outer block [ob0, obend)
        TmaGemmParams g{};                             // L_ij = A_ij * inv(L_jj)^T, in place (a tile is read completely before it is written)
        g.Mt = rem / NB; g.Nt = 1; g.batch = batch; g.K = NB; g.flags = 0; g.alpha = 1.0; g.beta = 0.0;
        g.a_row0 = (jb + 1) * NB; g.a_rstep = (int)Npad; g.a_col0 = jb * NB; g.a_cstep = 0;
        g.b_row0 = jb * NB; g.b_rstep = T * NB; g.b_col0 = 0; g.b_cstep = 0;
        g.C = A; g.ldc = ld; g.c_off0 = (int64_t)(jb + 1) * NB * ld + (int64_t)jb * NB; g.c_zstep = strideA;
        if ((rc = launch_gemm_tma(c, tmA, tmD, g, st))) return rc;
        const int nin = obend - jb - 1;                // tile columns of the outer block still to the right of this panel
        if (nin > 0) {
            TmaGemmParams q{};                         // columns jb+1 .. obend-1: A -= L_panel L_panel^T (lower tiles), K = 128
            q.Mt = rem / NB; q.Nt = nin; q.batch = batch; q.K = NB; q.flags = LOWER_ONLY; q.alpha = -1.0; q.beta = 1.0;
            q.a_row0 = (jb + 1) * NB; q.a_rstep = (int)Npad; q.a_col0 = jb * NB; q.a_cstep = 0;
            q.b_row0 = q.a_row0; q.b_rstep = q.a_rstep; q.b_col0 = q.a_col0; q.b_cstep = 0;
            q.C = A; q.ldc = ld; q.c_off0 = (int64_t)(jb + 1) * NB * (ld + 1); q.c_zstep = strideA;
            if ((rc = launch_gemm_tma(c, tmA, tmA, q, st))) return rc;
        }
        if (jb == obend - 1 && obend < T) {
            TmaGemmParams q{};                         // columns >= obend: A -= L_block L_block^T, K = (obend - ob0) * 128
            q.Mt = T - obend; q.Nt = T - obend; q.batch = batch; q.K = (obend - ob0) * NB; q.flags = LOWER_ONLY; q.alpha = -1.0; q.beta = 1.0;
            q.a_row0 = obend * NB; q.a_rstep = (int)Npad; q.a_col0 = ob0 * NB; q.a_cstep = 0;
            q.b_row0 = q.a_row0; q.b_rstep = q.a_rstep; q.b_col0 = q.a_col0; q.b_cstep = 0;
            q.C = A; q.ldc = ld; q.c_off0 = (int64_t)obend * NB * (ld + 1); q.c_zstep = strideA;
            if ((rc = launch_gemm_tma(c, tmA, tmA, q, st))) return rc;
        }
    }
    return ABO_OK;
}

// launch with programmatic stream serialization (PDL): the kernel may become resident while its
// predecessor in the stream drains; the kernels call griddepcontrol.wait before touching memory
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, bool pdl,
                              Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ------------------------------------------------------------------------------------------
// Single-matrix Cholesky with two-level blocking and look-ahead (the "Cholesky TFLOP/s" path).
//   outer block = LA_OB tile columns (384): inside it the panels are factored right-looking
//   (potf2+inverse, TRSM-as-GEMM, SYRK restricted to the block's own columns, K = 128);
//   the rest of the trailing matrix is updated ONCE per outer block with K = 384 by the
//   TMA/mbarrier DMMA kernel (syrk_tma_kernel), split into
//       U_next : the next outer block's columns  -> panel stream (high priority)
//       U_rest : everything further right        -> second stream, overlaps the next panel
// The four schedule constants were scanned on B200 at n = 4096 and 8192 (outer block 2-4, PDL from 24-80 tiles, 64-row
// panel tiles from 2048 rows or never, 32-row slabs up to 30-120 tiles): every setting came within 3 %, the panel chain
// and not the schedule is the limit.
// ------------------------------------------------------------------------------------------
constexpr int LA_OB = 3;             // outer block in tiles: the trailing matrix is read and written once per 384 columns
constexpr int LA_PDL_TILES = 40;     // PDL once T - Jb <= 40: earlier, resident dependents take shared memory from the U_rest CTAs
constexpr int LA_SMALL_NEXT = 60;    // largest U_next slab (tiles) on 32-row tiles: one 128-row tile per CTA would idle most SMs
constexpr int LA_BIG_REM = 4096;     // panel GEMMs: 64-row tiles while >= 4096 rows remain (throughput), 32-row below (latency)
int potrf_lookahead(abo_ctx* c, double* A, int64_t Npad, int64_t ld, double* Dinv, int* info, int notify_tile, cudaStream_t notify_stream) {
    const int T = (int)(Npad / NB);
    cudaStream_t sp = c->stream, su = c->stream2;
    CUtensorMap tmL;
    int rc = make_tmap_k4(&tmL, A, Npad, Npad, ld);
    if (rc) return rc;
    CU(cudaEventRecord(c->ev_a, sp));                 // su must see everything enqueued on sp so far
    CU(cudaStreamWaitEvent(su, c->ev_a, 0));
    bool rest_pending = false;
    bool s3_pending = false;
    bool boundary_split = false;
    cudaStream_t s3 = c->stream3;
    // outer blocks ramp up (1, 2, LA_OB, LA_OB, ...): the first panels are not hidden behind any update, so
    // the trailing-update stream is given work as early as possible
    int step = 0;
    for (int Jb = 0, je = 0; Jb < T; Jb = je, ++step) {
        je = std::min(Jb + std::min(step + 1, LA_OB), T);
        const bool pdl = (T - Jb) <= LA_PDL_TILES;
        // ---- panel block: tile columns [Jb, je)
        for (int jp = Jb; jp < je; ++jp) {
            double* Ajj = A + (int64_t)jp * NB * (ld + 1);
            double* Dj = Dinv + (int64_t)jp * NB * NB;
            CU(launch_pdl(potf2_ws_kernel, dim3(1), dim3(512), PW_SMEM_BYTES, sp, pdl, Ajj, ld, (int64_t)0, Dj, (int64_t)0, info, jp * NB));
            KL(c);
            if (s3_pending) { CU(cudaStreamWaitEvent(sp, c->ev_p[2], 0)); s3_pending = false; }   // bulk of the previous panel
            const int rem = (T - jp - 1) * NB;
            if (rem <= 0) break;
            double* P = Ajj + (int64_t)NB * ld;
            const int ncol = (je - jp - 1) * NB;       // remaining columns of this outer block
            auto gemm_panel = [&](const GemmParams& q, cudaStream_t s_, bool pdl_) -> int {
                if (q.M <= 0 || q.N <= 0) return ABO_OK;
                if (q.M >= LA_BIG_REM) CU(launch_pdl(gemm_small_kernel<64, 8>, dim3(q.N / BN, q.M / 64, 1), dim3(256), GemmS<64, 8>::SMEM_BYTES, s_, pdl_, q));
                else CU(launch_pdl(gemm_small_kernel<32, 8>, dim3(q.N / BN, q.M / 32, 1), dim3(256), GemmS<32, 8>::SMEM_BYTES, s_, pdl_, q));
                KL(c);
                return ABO_OK;
            };
            GemmParams g{};                            // TRSM as GEMM: L_ij = A_ij * inv(L_jj)^T, in place
            g.A = P; g.lda = ld; g.B = Dj; g.ldb = NB; g.C = P; g.ldc = ld;
            g.M = rem; g.N = NB; g.K = NB; g.alpha = 1.0; g.beta = 0.0; g.flags = 0;
            GemmParams s{};                            // in-block SYRK: A_22 -= L_21 L_21^T (columns of this outer block)
            s.A = P; s.lda = ld; s.B = P; s.ldb = ld;
            s.C = Ajj + (int64_t)NB * (ld + 1); s.ldc = ld;
            s.M = rem; s.N = ncol; s.K = NB; s.alpha = -1.0; s.beta = 1.0; s.flags = LOWER_ONLY;
            int rc2;
            if (ncol <= 0 && rem > NB) {
                // last panel of the outer block: the next potf2 waits for tile row je of this TRSM and for the
                // update of tile (je, je) only (diag_next below); the other rows go to the bulk stream
                GemmParams g1 = g; g1.M = NB;
                CU(launch_pdl(gemm_k128_kernel<16, 128>, dim3(1, 8, 1), dim3(128), GemmK128<16, 128>::SMEM_BYTES, sp, pdl, g1)); KL(c);
                CU(cudaEventRecord(c->ev_p[1], sp));
                CU(cudaStreamWaitEvent(s3, c->ev_p[1], 0));
                GemmParams g2 = g; g2.A = P + (int64_t)NB * ld; g2.C = P + (int64_t)NB * ld; g2.M = rem - NB;
                if ((rc2 = gemm_panel(g2, s3, false))) return rc2;
                CU(cudaEventRecord(c->ev_p[2], s3));
                s3_pending = true;
                boundary_split = true;
            } else if (ncol <= 0 || rem <= NB) {
                if ((rc2 = gemm_panel(g, sp, pdl))) return rc2;
                if ((rc2 = gemm_panel(s, sp, pdl))) return rc2;
            } else {
                // split panel chain: only the next diagonal tile is on the critical path of the next
                // potf2; the bulk of the TRSM / in-block SYRK runs on a third stream concurrently with it
                // (the three critical kernels stay back to back on the panel stream so that PDL applies;
                //  the bulk stream picks up after them — it has a full potf2 of slack)
                GemmParams g1 = g; g1.M = NB;                              // tile row jp+1
                GemmParams s1 = s; s1.M = NB; s1.N = NB; s1.flags = 0;     // diagonal tile (jp+1, jp+1)
                // latency kernels: 8 / 16 CTAs, one load group
                CU(launch_pdl(gemm_k128_kernel<16, 128>, dim3(1, 8, 1), dim3(128), GemmK128<16, 128>::SMEM_BYTES, sp, pdl, g1)); KL(c);   // in place: whole rows per CTA
                CU(launch_pdl(gemm_k128_kernel<32, 32>, dim3(4, 4, 1), dim3(128), GemmK128<32, 32>::SMEM_BYTES, sp, pdl, s1)); KL(c);
                CU(cudaEventRecord(c->ev_p[1], sp));                       // potf2(jp), L[jp+1, jp] final
                CU(cudaStreamWaitEvent(s3, c->ev_p[1], 0));
                GemmParams g2 = g; g2.A = P + (int64_t)NB * ld; g2.C = P + (int64_t)NB * ld; g2.M = rem - NB;
                if ((rc2 = gemm_panel(g2, s3, false))) return rc2;         // remaining rows of the TRSM
                GemmParams s2 = s;                                         // remaining tiles: rows from tile jp+2
                s2.A = P + (int64_t)NB * ld; s2.C = s.C + (int64_t)NB * ld; s2.M = rem - NB; s2.lower_shift = NB;
                if ((rc2 = gemm_panel(s2, s3, false))) return rc2;
                CU(cudaEventRecord(c->ev_p[2], s3));
                s3_pending = true;
            }
        }
        if (s3_pending && !boundary_split) { CU(cudaStreamWaitEvent(sp, c->ev_p[2], 0)); s3_pending = false; }
        if (je >= T) break;
        SyrkParams u;
        u.C = A; u.ld = ld; u.kcol0 = Jb * NB; u.nk = (je - Jb) * (NB / 16); u.skip_first = 0;
        // ---- U_rest(b) on the second stream: needs panel(b) (event) and, by stream order, U_rest(b-1)
        const int jn = std::min(je + std::min(step + 2, LA_OB), T);
        CU(cudaEventRecord(c->ev_a, sp));
        if (notify_stream && notify_tile > 0 && je >= notify_tile) {
            // every column tile < je of L is final once the panel stream reaches this point (and the bulk rows of the last
            // TRSM have landed): work that only needs the leading columns may start on `notify_stream` now
            CU(cudaStreamWaitEvent(notify_stream, c->ev_a, 0));
            if (boundary_split) CU(cudaStreamWaitEvent(notify_stream, c->ev_p[2], 0));
            notify_tile = 0;
        }
        if (jn < T) {
            CU(cudaStreamWaitEvent(su, c->ev_a, 0));
            if (boundary_split) CU(cudaStreamWaitEvent(su, c->ev_p[2], 0));   // the bulk rows of the last TRSM
            u.row_t0 = jn; u.col_t0 = jn;
            syrk_tma_kernel<<<dim3(T - jn, T - jn), SW_THREADS, SY_SMEM_BYTES, su>>>(tmL, u);
            KL(c);
        }
        // ---- U_next(b) on the panel stream: the next block's columns; they were last touched by
        //      U_rest(b-1), so wait for it
        if (rest_pending) CU(cudaStreamWaitEvent(sp, c->ev_b, 0));
        cudaStream_t sn = sp;                              // stream of the (bulk of the) U_next update
        bool pdl_next = pdl && !rest_pending;
        if (boundary_split) {
            // critical chain: only tile (je, je) — K = width of the outer block — then straight on to potf2(je);
            // the rest of U_next follows the bulk TRSM on the third stream (it has that potf2 of slack)
            GemmParams dn{};
            dn.A = A + (int64_t)je * NB * ld + (int64_t)Jb * NB; dn.lda = ld;
            dn.B = dn.A; dn.ldb = ld;
            dn.C = A + (int64_t)je * NB * (ld + 1); dn.ldc = ld;
            dn.M = NB; dn.N = NB; dn.K = (je - Jb) * NB; dn.alpha = -1.0; dn.beta = 1.0; dn.flags = 0;
            CU(launch_pdl(gemm_k128_kernel<32, 32>, dim3(4, 4, 1), dim3(128), GemmK128<32, 32>::SMEM_BYTES, sp, pdl_next, dn)); KL(c);
            if (rest_pending) CU(cudaStreamWaitEvent(s3, c->ev_b, 0));
            sn = s3; pdl_next = false; u.skip_first = 1;
        }
        if ((T - je) * (jn - je) <= LA_SMALL_NEXT) {
            // few tiles: one 128x128xK tile per CTA would leave most SMs idle for a full tile time
            // (~55 us); 32-row tiles finish the slab in ~1/3 of that
            GemmParams nx{};
            nx.A = A + (int64_t)je * NB * ld + (int64_t)Jb * NB; nx.lda = ld;
            nx.B = nx.A; nx.ldb = ld;
            nx.C = A + (int64_t)je * NB * (ld + 1); nx.ldc = ld;
            nx.M = (T - je) * NB; nx.N = (jn - je) * NB; nx.K = (je - Jb) * NB;
            nx.alpha = -1.0; nx.beta = 1.0; nx.flags = LOWER_ONLY | (boundary_split ? SKIP_FIRST : 0);
            CU(launch_pdl(gemm_small_kernel<32, 8>, dim3(nx.N / BN, nx.M / 32, 1), dim3(256), GemmS<32, 8>::SMEM_BYTES, sn,
                          pdl_next, nx));
        } else {
            u.row_t0 = je; u.col_t0 = je;
            CU(launch_pdl(syrk_tma_kernel, dim3(jn - je, T - je), dim3(SW_THREADS), SY_SMEM_BYTES, sn, pdl_next, tmL, u));
        }
        KL(c);
        if (boundary_split) {                              // the next potf2's TRSM needs it: waited for right after that potf2
            CU(cudaEventRecord(c->ev_p[2], s3));
            s3_pending = true;
            boundary_split = false;
        }
        if (jn < T) { CU(cudaEventRecord(c->ev_b, su)); rest_pending = true; }
    }
    if (rest_pending) CU(cudaStreamWaitEvent(sp, c->ev_b, 0));
    if (notify_stream && notify_tile > 0) {
        // no outer-block boundary fell in [notify_tile, T) (the loop breaks at je = T before notifying): the notified
        // work waits for the whole factor instead; every side stream has joined the panel stream by now
        CU(cudaEventRecord(c->ev_a, sp));
        CU(cudaStreamWaitEvent(notify_stream, c->ev_a, 0));
    }
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// triangular inverse  X = L^-1  by recursive doubling on tiles, on the TMA pipeline (gemm_tma.cuh): the diagonal tiles
// are the block inverses from potf2; at level b (tiles) every pair computes  X21 = - X22 * (L21 * X11)  as two GEMMs that
// skip the structurally-zero k-ranges.  To keep every operand k-contiguous the recursion also carries U = X^T (written by
// the transposed-store epilogue) and keeps the intermediate W21 = L21 X11 only as its transpose:
//                    Wt = W21^T                   <- A = L21, B = U11 (rows of X11^T)
//                    X21 = -X22 W21               <- A = X22, B = W21^T ;  U12 = X21^T by the same launch
// Single matrix: all pairs of a level are one launch batched over the pairs; batched matrices (NLML): one
// launch per pair batched over the matrices.  Wt, U: scratch / output of the shape of L.
// ------------------------------------------------------------------------------------------
__global__ void place_diag_both_kernel(const double* __restrict__ Dinv, double* __restrict__ Linv, double* __restrict__ U, int64_t ld,
                                       int64_t strideD, int64_t strideL) {
    const int t = blockIdx.x;
    const double* src = Dinv + (int64_t)blockIdx.y * strideD + (int64_t)t * NB * NB;
    double* dst = Linv + (int64_t)blockIdx.y * strideL + (int64_t)t * NB * (ld + 1);
    double* dsu = U + (int64_t)blockIdx.y * strideL + (int64_t)t * NB * (ld + 1);
    for (int e = threadIdx.x; e < NB * NB; e += blockDim.x) {
        const int r = e >> 7, cc = e & 127;
        dst[(int64_t)r * ld + cc] = src[e];
        dsu[(int64_t)r * ld + cc] = src[cc * NB + r];
    }
}
template <int EPI>
static int launch_gemm_tma(abo_ctx* c, const CUtensorMap& tmA, const CUtensorMap& tmB, TmaGemmParams p, cudaStream_t st, int max_ctas) {
    if (p.Mt <= 0 || p.Nt <= 0 || p.batch <= 0) return ABO_OK;
    if ((p.flags & LOWER_ONLY) && p.Nt > p.Mt) return abo_fail(ABO_ERR_INVALID, "gemm_tma: LOWER_ONLY needs Nt <= Mt");
    const int64_t per = (p.flags & LOWER_ONLY) ? (int64_t)p.Nt * (p.Nt + 1) / 2 + (int64_t)(p.Mt - p.Nt) * p.Nt : (int64_t)p.Mt * p.Nt;
    const int64_t total = per * p.batch;
    if (total > 0x7fffffff) return abo_fail(ABO_ERR_INVALID, "too many tiles in one launch");
    p.total = (int)total;
    gemm_tma_kernel<EPI><<<(int)std::min<int64_t>(total, max_ctas > 0 ? max_ctas : c->sms), SW_THREADS, tg_smem_bytes<EPI>(), st>>>(tmA, tmB, p);
    KL(c);
    return ABO_OK;
}
// One pair of the recursion: block 11 = tile rows / columns [o, o + b), block 22 = tile rows [o + b, o + b + rr).  The launch
// covers zb such pairs, item z displaced by (z rstep, z cstep) elements in the tensor maps and by z zoff doubles in memory.
struct TrtriPair { int o, b, rr, zb, rstep, cstep; int64_t zoff; };
// Wt(o, o+b) = (L21 X11)^T : A = L21, B = U11 (k >= n)
static int trtri_pair_w(abo_ctx* c, const CUtensorMap& tmL, const CUtensorMap& tmU, double* Wt, int64_t ld, const TrtriPair& q,
                        cudaStream_t st, int max_ctas) {
    TmaGemmParams g{};
    g.batch = q.zb; g.alpha = 1.0; g.beta = 0.0;
    g.Mt = q.rr; g.Nt = q.b; g.K = q.b * NB; g.flags = KLO_N;
    g.a_row0 = (q.o + q.b) * NB; g.a_col0 = q.o * NB; g.a_rstep = q.rstep; g.a_cstep = q.cstep;
    g.b_row0 = q.o * NB; g.b_col0 = q.o * NB; g.b_rstep = q.rstep; g.b_cstep = q.cstep;
    g.C = nullptr; g.CT = Wt; g.ldct = ld; g.ct_off0 = (int64_t)q.o * NB * ld + (int64_t)(q.o + q.b) * NB; g.ct_zstep = q.zoff;
    return launch_gemm_tma(c, tmL, tmU, g, st, max_ctas);
}
// X21 = -X22 W21 (k <= m): A = X22, B = W21^T ; U12 = X21^T
static int trtri_pair_x(abo_ctx* c, const CUtensorMap& tmX, const CUtensorMap& tmW, double* Linv, double* U, int64_t ld,
                        const TrtriPair& q, cudaStream_t st, int max_ctas) {
    TmaGemmParams h{};
    h.batch = q.zb; h.alpha = -1.0; h.beta = 0.0;
    h.Mt = q.rr; h.Nt = q.b; h.K = q.rr * NB; h.flags = KHI_M;
    h.a_row0 = (q.o + q.b) * NB; h.a_col0 = (q.o + q.b) * NB; h.a_rstep = q.rstep; h.a_cstep = q.cstep;
    h.b_row0 = q.o * NB; h.b_col0 = (q.o + q.b) * NB; h.b_rstep = q.rstep; h.b_cstep = q.cstep;
    h.C = Linv; h.ldc = ld; h.c_off0 = (int64_t)(q.o + q.b) * NB * ld + (int64_t)q.o * NB; h.c_zstep = q.zoff;
    h.CT = U; h.ldct = ld; h.ct_off0 = (int64_t)q.o * NB * ld + (int64_t)(q.o + q.b) * NB; h.ct_zstep = q.zoff;
    return launch_gemm_tma(c, tmX, tmW, h, st, max_ctas);
}
// st / max_ctas: stream and CTA cap of every launch
static int trtri_tma_on(abo_ctx* c, const double* L, double* Linv, double* U, double* Wt, int64_t Npad, int64_t ld, int64_t strideM,
                        const double* Dinv, int64_t strideD, int batch, cudaStream_t st, int max_ctas) {
    const int T = (int)(Npad / NB);
    const int64_t rows = (batch == 1) ? Npad : (int64_t)batch * Npad;        // batched matrices are stacked (strideM = Npad * ld)
    if (batch > 1 && strideM != Npad * ld) return abo_fail(ABO_ERR_INVALID, "trtri_tma: batched matrices must be contiguous");
    place_diag_both_kernel<<<dim3(T, batch), 256, 0, st>>>(Dinv, Linv, U, ld, strideD, strideM);
    KL(c);
    if (T == 1) return ABO_OK;                                              // a single tile: no level, no tensor maps
    CUtensorMap tmL, tmX, tmU, tmW;
    int rc;
    if ((rc = make_tmap_k4(&tmL, L, Npad, rows, ld)) || (rc = make_tmap_k4(&tmX, Linv, Npad, rows, ld)) ||
        (rc = make_tmap_k4(&tmU, U, Npad, rows, ld)) || (rc = make_tmap_k4(&tmW, Wt, Npad, rows, ld)))
        return rc;
    for (int b = 1; b < T; b <<= 1) {
        const int npairs = (T - b + 2 * b - 1) / (2 * b), nfull = T / (2 * b);
        // groups of pairs with equal shapes: (first pair, count, rows of block 22)
        struct Grp { int q0, nq, rr; };
        std::vector<Grp> groups;
        if (nfull > 0) groups.push_back({0, nfull, b});
        if (npairs > nfull) groups.push_back({nfull, 1, T - 2 * b * nfull - b});
        for (const Grp& gq : groups) {
            const int launches = (batch == 1) ? 1 : gq.nq;                  // batched matrices: one launch per pair
            for (int li = 0; li < launches; ++li) {
                TrtriPair q;
                q.o = 2 * b * (gq.q0 + li); q.b = b; q.rr = gq.rr;
                q.zb = (batch == 1) ? gq.nq : batch;
                q.rstep = (batch == 1) ? 2 * b * NB : (int)Npad; q.cstep = (batch == 1) ? 2 * b * NB : 0;
                q.zoff = (batch == 1) ? (int64_t)2 * b * NB * (ld + 1) : strideM;
                if ((rc = trtri_pair_w(c, tmL, tmU, Wt, ld, q, st, max_ctas)) || (rc = trtri_pair_x(c, tmX, tmW, Linv, U, ld, q, st, max_ctas)))
                    return rc;
            }
        }
    }
    return ABO_OK;
}
int trtri_tma(abo_ctx* c, const double* L, double* Linv, double* U, double* Wt, int64_t Npad, int64_t ld, int64_t strideM,
              const double* Dinv, int64_t strideD, int batch) {
    return trtri_tma_on(c, L, Linv, U, Wt, Npad, ld, strideM, Dinv, strideD, batch, c->stream, 0);
}

// beta = Linv * delta ; alpha = Linv^T * beta      (alpha = (K + noise I)^-1 (y - m))
int solve_alpha(abo_ctx* c, const double* Linv, int64_t ld, int64_t N, const double* delta, double* beta,
                double* alpha, int64_t strideM, int64_t strideV, int batch) {
    cudaStream_t st = c->stream;
    {
        int64_t threads = N * 32;
        dim3 grid((unsigned)((threads + 255) / 256), batch);
        trmv_lower_kernel<<<grid, 256, 0, st>>>(Linv, ld, N, delta, beta, strideM, strideV);
        KL(c);
    }
    const int nchunks = (int)((N + TRMVT_ROWS - 1) / TRMVT_ROWS);
    double* part;
    int rc = ws_get(c, WS_VEC_PART, sizeof(double) * (size_t)nchunks * N * batch, (void**)&part);
    if (rc) return rc;
    {
        dim3 grid((unsigned)((N + 127) / 128), nchunks, batch);
        trmvT_lower_partial_kernel<<<grid, 128, 0, st>>>(Linv, ld, N, beta, part, strideM, strideV, (int64_t)nchunks * N);
        KL(c);
        dim3 g2((unsigned)((N + 127) / 128), batch);
        reduce_rows_kernel<<<g2, 128, 0, st>>>(part, nchunks, N, alpha, (int64_t)nchunks * N, strideV);
        KL(c);
    }
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// surrogate handle
// ------------------------------------------------------------------------------------------
// Device buffers are reference counted: abo_gp_clone shares them (O(1), Base.copy of a posterior in
// the BO loop, bayesian_opt.jl:116) and a handle that is about to WRITE takes a private set first
// (gp_alloc for a re-fit, gp_unshare for an append).  Released sets go to a small per-context pool.
constexpr size_t GP_POOL_MAX_SETS = 3;
constexpr size_t GP_POOL_MAX_BYTES = (size_t)24 << 30;
static size_t gp_set_bytes(int64_t cap_pad) { return 2 * sizeof(double) * (size_t)cap_pad * cap_pad; }

static void gp_free_device(abo_gp* g) {
    cudaSetDevice(g->ctx->device);
    double** ptrs[] = {&g->dXsT, &g->dL, &g->dLinv, &g->dAlpha, &g->dBeta, &g->dDelta, &g->dMeanC};
    if (g->share && --*g->share == 0) {
        delete g->share;
        abo_ctx* c = g->ctx;
        size_t pooled = 0;
        for (auto& e : c->gp_pool) pooled += gp_set_bytes(e.cap_pad);
        if (g->dL && c->gp_pool.size() < GP_POOL_MAX_SETS && pooled + gp_set_bytes(g->cap_pad) <= GP_POOL_MAX_BYTES) {
            abo_ctx::GpBufSet e{g->cap_pad, g->ldx, g->d, g->p, {}};
            for (int q = 0; q < 7; ++q) e.ptr[q] = *ptrs[q];
            c->gp_pool.push_back(e);
        } else {
            for (auto pp : ptrs) if (*pp) cudaFree(*pp);
        }
    }
    for (auto pp : ptrs) *pp = nullptr;
    g->share = nullptr;
    g->fitted = false;
    g->cap_pad = 0;
}

void gp_pool_clear(abo_ctx* c) {
    for (auto& e : c->gp_pool) for (double* q : e.ptr) if (q) cudaFree(q);
    c->gp_pool.clear();
}

int gp_alloc(abo_gp* g, int64_t Npad, int64_t ldx) {
    gp_free_device(g);
    abo_ctx* c = g->ctx;
    double** ptrs[] = {&g->dXsT, &g->dL, &g->dLinv, &g->dAlpha, &g->dBeta, &g->dDelta, &g->dMeanC};
    g->share = new (std::nothrow) int(1);
    if (!g->share) return abo_fail(ABO_ERR_ALLOC, "host allocation failed");
    for (size_t q = 0; q < c->gp_pool.size(); ++q) {
        auto& e = c->gp_pool[q];
        if (e.cap_pad == Npad && e.ldx == ldx && e.d == g->d && e.p == g->p) {
            for (int r = 0; r < 7; ++r) *ptrs[r] = e.ptr[r];
            c->gp_pool.erase(c->gp_pool.begin() + q);
            g->cap_pad = Npad; g->ld = Npad; g->ldx = ldx;
            return ABO_OK;
        }
    }
    size_t mat = sizeof(double) * (size_t)Npad * Npad;
    cudaError_t e = cudaSuccess;
    for (int attempt = 0; attempt < 2; ++attempt) {
        if ((e = cudaMalloc(&g->dL, mat)) == cudaSuccess && (e = cudaMalloc(&g->dLinv, mat)) == cudaSuccess &&
            (e = cudaMalloc(&g->dXsT, sizeof(double) * (size_t)ldx * g->d)) == cudaSuccess &&
            (e = cudaMalloc(&g->dAlpha, sizeof(double) * Npad)) == cudaSuccess &&
            (e = cudaMalloc(&g->dBeta, sizeof(double) * Npad)) == cudaSuccess &&
            (e = cudaMalloc(&g->dDelta, sizeof(double) * Npad)) == cudaSuccess &&
            (e = cudaMalloc(&g->dMeanC, sizeof(double) * g->p)) == cudaSuccess)
            break;
        cudaGetLastError();
        for (auto pp : ptrs) { if (*pp) cudaFree(*pp); *pp = nullptr; }
        if (attempt == 0 && !c->gp_pool.empty()) { gp_pool_clear(c); continue; }   // give the pooled sets back and retry
        delete g->share; g->share = nullptr;
        return abo_fail(ABO_ERR_ALLOC, "device allocation for a %lld x %lld posterior failed: %s", (long long)Npad,
                        (long long)Npad, cudaGetErrorString(e));
    }
    g->cap_pad = Npad;
    g->ld = Npad;
    g->ldx = ldx;
    return ABO_OK;
}

// private copy of shared buffers before an in-place update (copy-on-write): the lower tiles of L and
// L^-1 (the upper ones are never read), the coordinates and the vectors
__global__ void copy_lower_tiles_kernel(const double* __restrict__ a0, const double* __restrict__ a1, double* __restrict__ b0,
                                        double* __restrict__ b1, int64_t ld) {
    if (blockIdx.x > blockIdx.y) return;
    const double* src = blockIdx.z ? a1 : a0;
    double* dst = blockIdx.z ? b1 : b0;
    const int64_t base = (int64_t)blockIdx.y * NB * ld + (int64_t)blockIdx.x * NB;
    for (int e = threadIdx.x; e < NB * NB / 2; e += blockDim.x) {
        const int r = e / (NB / 2), c2 = e % (NB / 2);
        reinterpret_cast<double2*>(dst + base + (int64_t)r * ld)[c2] = reinterpret_cast<const double2*>(src + base + (int64_t)r * ld)[c2];
    }
}

int gp_unshare(abo_gp* g) {
    if (!gp_shared(g)) return ABO_OK;
    abo_ctx* c = g->ctx;
    cudaStream_t st = c->stream;
    abo_gp old = *g;                                    // keeps the shared pointers; its count is dropped below
    g->dXsT = g->dL = g->dLinv = g->dAlpha = g->dBeta = g->dDelta = g->dMeanC = nullptr;
    g->share = nullptr;
    const bool fitted = old.fitted;
    int rc = gp_alloc(g, old.cap_pad, old.ldx);         // gp_free_device on the nulled handle is a no-op
    if (rc) { *g = old; return rc; }
    const int T = (int)(old.cap_pad / NB);
    copy_lower_tiles_kernel<<<dim3(T, T, 2), 256, 0, st>>>(old.dL, old.dLinv, g->dL, g->dLinv, old.ld);
    KL(c);
    CU(cudaMemcpyAsync(g->dXsT, old.dXsT, sizeof(double) * old.ldx * old.d, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(g->dAlpha, old.dAlpha, sizeof(double) * old.cap_pad, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(g->dBeta, old.dBeta, sizeof(double) * old.cap_pad, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(g->dDelta, old.dDelta, sizeof(double) * old.cap_pad, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(g->dMeanC, old.dMeanC, sizeof(double) * old.p, cudaMemcpyDeviceToDevice, st));
    CU(cudaStreamSynchronize(st));
    --*old.share;                                       // > 0 by construction: the other holders keep the set
    g->fitted = fitted;
    return ABO_OK;
}

extern "C" int32_t abo_gp_create(abo_ctx* ctx, int32_t kernel_id, int32_t d, int32_t p, abo_gp** out) {
    if (!ctx || !out) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (kernel_id < 0 || kernel_id > 6) return abo_fail(ABO_ERR_INVALID, "unknown kernel id %d", kernel_id);
    if (d < 1) return abo_fail(ABO_ERR_INVALID, "d must be >= 1");
    if (p != 1 && p != d + 1) return abo_fail(ABO_ERR_INVALID, "p must be 1 (StandardGP) or d+1 (GradientGP)");
    if (p > 1 && (kernel_id == ABO_KERNEL_MATERN52 || kernel_id == ABO_KERNEL_MATERN72))
        return abo_fail(ABO_ERR_INVALID,
                        "KernelFunctions Matern kernels are not differentiable at 0 (NaN, test/test_kernels.jl:87); "
                        "use the Approx/AD variants for GradientGP");
    abo_gp* g = new (std::nothrow) abo_gp();
    if (!g) return abo_fail(ABO_ERR_ALLOC, "host allocation failed");
    g->ctx = ctx; g->kind = kernel_id; g->d = d; g->p = p;
    g->s = 1.0; g->scale = 1.0; g->noise = 0.0;
    g->sv.assign(d, 1.0); g->ard = false;
    g->mean_c.assign(p, 0.0);
    ctx->live.insert(g);
    *out = g;
    return ABO_OK;
}

extern "C" int32_t abo_gp_destroy(abo_gp* g) {
    if (!g) return ABO_OK;
    if (g->ctx) { g->ctx->live.erase(g); gp_free_device(g); }
    delete g;
    return ABO_OK;
}

extern "C" int32_t abo_gp_set_params(abo_gp* g, double inv_ls, double scale, double noise, const double* mean_c) {
    if (!g) return abo_fail(ABO_ERR_INVALID, "null gp");
    if (!(inv_ls > 0) || !(scale > 0) || !(noise >= 0) || !std::isfinite(inv_ls) || !std::isfinite(scale))
        return abo_fail(ABO_ERR_INVALID, "hyper-parameters must be positive and finite (noise >= 0)");
    g->s = inv_ls; g->scale = scale; g->noise = noise;
    g->sv.assign(g->d, inv_ls); g->ard = false;
    for (int a = 0; a < g->p; ++a) g->mean_c[a] = mean_c ? mean_c[a] : 0.0;
    g->fitted = false;
    return ABO_OK;
}

extern "C" int32_t abo_gp_set_params_ard(abo_gp* g, const double* inv_ls, double scale, double noise, const double* mean_c) {
    if (!g || !inv_ls) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (g->d > ARD_MAXD) return abo_fail(ABO_ERR_INVALID, "ARD length scales are supported for d <= %d", ARD_MAXD);
    for (int k = 0; k < g->d; ++k)
        if (!(inv_ls[k] > 0) || !std::isfinite(inv_ls[k])) return abo_fail(ABO_ERR_INVALID, "inverse length scales must be positive and finite");
    if (!(scale > 0) || !(noise >= 0) || !std::isfinite(scale)) return abo_fail(ABO_ERR_INVALID, "hyper-parameters must be positive and finite (noise >= 0)");
    g->sv.assign(inv_ls, inv_ls + g->d);
    g->s = inv_ls[0]; g->scale = scale; g->noise = noise; g->ard = true;
    for (int a = 0; a < g->p; ++a) g->mean_c[a] = mean_c ? mean_c[a] : 0.0;
    g->fitted = false;
    return ABO_OK;
}

static KSpec gp_spec(const abo_gp* g) {
    KSpec k;
    k.kind = g->kind; k.d = g->d; k.p = g->p; k.s = g->s; k.scale = g->scale; k.noise = g->noise;
    for (int q = 0; q < ARD_MAXD; ++q) k.sv[q] = (q < g->d && q < (int)g->sv.size()) ? g->sv[q] : g->s;
    return k;
}

static int gp_fit_run(abo_gp* g, const double* X, const double* y, int64_t n, int64_t* info_out);
constexpr int FIT_OVERLAP_MIN_TILES = 32;   // smallest system (tiles) whose leading inverse runs alongside the factorisation
constexpr int FIT_OVERLAP_CTAS = 112;       // CTA cap of the overlapped launches: 36 of the 148 SMs stay with the factorisation
extern "C" int32_t abo_gp_fit(abo_gp* g, const double* X, const double* y, int64_t n, int64_t* info_out) {
    const int rc = gp_fit_run(g, X, y, n, info_out);
    if (rc && g && g->ctx) {
        // an error return must not leave the factorisation's side streams or the overlapped inverse on stream4 running:
        // they write L, L^-1 and workspace slots that the next call may reuse.  Drain every stream, keep the first error.
        const std::string keep = g_err;
        ctx_sync_all(g->ctx);
        cudaGetLastError();
        g_err = keep;
    }
    return rc;
}
static int gp_fit_run(abo_gp* g, const double* X, const double* y, int64_t n, int64_t* info_out) {
    if (!g || !X || !y) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (n < 1) return abo_fail(ABO_ERR_DIM, "need at least one observation");
    if (!g->ctx) return abo_fail(ABO_ERR_INVALID, "the context of this handle has been destroyed");
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t N = n * g->p;
    const int64_t Npad = (N + NB - 1) / NB * NB;
    const int64_t ldx = (n + NB - 1) / NB * NB + NB;      // room for appended points
    g->fitted = false;
    if (Npad != g->cap_pad || ldx > g->ldx || gp_shared(g)) { int rc = gp_alloc(g, Npad, ldx); if (rc) return rc; }
    g->n = n; g->N = N; g->Npad = Npad;

    // stage X, y
    double *dXraw, *dYraw;
    int rc;
    if ((rc = ws_get(c, WS_STAGE_X, sizeof(double) * (size_t)n * g->d, (void**)&dXraw))) return rc;
    if ((rc = ws_get(c, WS_STAGE_Y, sizeof(double) * (size_t)N, (void**)&dYraw))) return rc;
    CU(cudaMemcpyAsync(dXraw, X, sizeof(double) * n * g->d, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dYraw, y, sizeof(double) * N, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(g->dMeanC, g->mean_c.data(), sizeof(double) * g->p, cudaMemcpyHostToDevice, st));
    {
        int64_t tot = g->ldx * g->d;
        scale_transpose_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(dXraw, g->dXsT, n, g->d, g->ldx, gp_spec(g));
        KL(c);
        fill_kernel<<<(unsigned)((Npad + 255) / 256), 256, 0, st>>>(g->dDelta, Npad, 0.0);
        KL(c);
        delta_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(dYraw, g->dMeanC, n, g->p, g->dDelta);
        KL(c);
    }
    const int T = (int)(Npad / NB);
    KmatBatch bt{nullptr, nullptr, 0, 0, 0};
    launch_kmat(gp_spec(g), g->dXsT, g->ldx, N, g->dL, g->ld, bt, T, 1, st);
    KL(c);

    double* Dinv; int* dinfo; double* W;
    if ((rc = ws_get(c, WS_DINV, sizeof(double) * (size_t)T * NB * NB, (void**)&Dinv))) return rc;
    if ((rc = ws_get(c, WS_INFO, sizeof(int) * 16, (void**)&dinfo))) return rc;
    if ((rc = ws_get(c, WS_TRTRI, sizeof(double) * (size_t)Npad * Npad, (void**)&W))) return rc;
    CU(cudaMemsetAsync(dinfo, 0, sizeof(int) * 16, st));
    // Conditioning schedule: the triangular inverse of the LEADING b_top tile columns and the first product of the top level
    // (W21 = L21 X11) only need the leading columns of L, which are final half-way through the factorisation — they run on a
    // low-priority stream with a capped grid while the factorisation's chain-bound tail leaves most SMs idle; the trailing
    // block's inverse and the second product (X21 = -X22 W21) follow once the factorisation is complete.
    double* U;
    if ((rc = ws_get(c, WS_TRTRI_U, sizeof(double) * (size_t)Npad * Npad, (void**)&U))) return rc;
    int b_top = 1;
    while (2 * b_top < T) b_top *= 2;                                  // largest power of two below T: the top-level pair is (0, b_top)
    const TrtriPair top{0, b_top, T - b_top, 1, 0, 0, 0};
    const bool overlap = T >= FIT_OVERLAP_MIN_TILES;
    if ((rc = potrf_lookahead(c, g->dL, Npad, g->ld, Dinv, dinfo, overlap ? b_top : 0, overlap ? c->stream4 : nullptr))) return rc;
    if (overlap) {
        cudaStream_t s4 = c->stream4;
        const int64_t nl = (int64_t)b_top * NB;
        if ((rc = trtri_tma_on(c, g->dL, g->dLinv, U, W, nl, g->ld, 0, Dinv, 0, 1, s4, FIT_OVERLAP_CTAS))) return rc;
        CUtensorMap tmL, tmU;
        if ((rc = make_tmap_k4(&tmL, g->dL, Npad, Npad, g->ld)) || (rc = make_tmap_k4(&tmU, U, Npad, Npad, g->ld))) return rc;
        if ((rc = trtri_pair_w(c, tmL, tmU, W, g->ld, top, s4, FIT_OVERLAP_CTAS))) return rc;
        CU(cudaEventRecord(c->ev_inv, s4));
    }
    int hinfo = 0;
    CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (info_out) *info_out = hinfo;
    if (hinfo != 0)                                                   // abo_gp_fit drains stream4 on the way out
        return abo_fail(ABO_ERR_NOT_POSDEF, "matrix is not positive definite; Cholesky factorization failed at pivot %d", hinfo);
    if (overlap) {
        const int64_t off = (int64_t)b_top * NB * (g->ld + 1);
        if ((rc = trtri_tma_on(c, g->dL + off, g->dLinv + off, U + off, W + off, Npad - (int64_t)b_top * NB, g->ld, 0,
                               Dinv + (int64_t)b_top * NB * NB, 0, 1, st, 0))) return rc;
        CU(cudaStreamWaitEvent(st, c->ev_inv, 0));
        CUtensorMap tmX, tmW;
        if ((rc = make_tmap_k4(&tmX, g->dLinv, Npad, Npad, g->ld)) || (rc = make_tmap_k4(&tmW, W, Npad, Npad, g->ld))) return rc;
        if ((rc = trtri_pair_x(c, tmX, tmW, g->dLinv, U, g->ld, top, st, 0))) return rc;
    } else if ((rc = trtri_tma(c, g->dL, g->dLinv, U, W, Npad, g->ld, 0, Dinv, 0, 1))) return rc;
    if ((rc = solve_alpha(c, g->dLinv, g->ld, Npad, g->dDelta, g->dBeta, g->dAlpha, 0, 0, 1))) return rc;
    CU(cudaStreamSynchronize(st));
    g->fitted = true;
    return ABO_OK;
}

extern "C" int32_t abo_gp_clone(const abo_gp* g, abo_gp** out) {
    if (!g || !out) return abo_fail(ABO_ERR_INVALID, "null argument");
    abo_gp* n = new (std::nothrow) abo_gp(*g);          // shares the device buffers; a writer un-shares first
    if (!n) return abo_fail(ABO_ERR_ALLOC, "host allocation failed");
    if (n->share) ++*n->share;
    if (n->ctx) n->ctx->live.insert(n);
    *out = n;
    return ABO_OK;
}

extern "C" int32_t abo_gp_n(const abo_gp* g, int64_t* n) {
    if (!g || !n) return abo_fail(ABO_ERR_INVALID, "null argument");
    *n = g->fitted ? g->n : 0;
    return ABO_OK;
}

extern "C" int32_t abo_gp_alpha(const abo_gp* g, double* alpha) {
    if (!g || !alpha) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior");
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    double* tmp;
    int rc = ws_get(c, WS_STAGE_Y, sizeof(double) * (size_t)g->N, (void**)&tmp);
    if (rc) return rc;
    to_out_major_kernel<<<(unsigned)((g->N + 255) / 256), 256, 0, c->stream>>>(g->dAlpha, g->n, g->p, tmp);
    KL(c);
    CU(cudaMemcpyAsync(alpha, tmp, sizeof(double) * g->N, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    return ABO_OK;
}

extern "C" int32_t abo_gp_factor(const abo_gp* g, int32_t which, double* out) {
    if (!g || !out) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior");
    CU(cudaSetDevice(g->ctx->device));
    const double* src = which == 0 ? g->dL : g->dLinv;
    CU(cudaMemcpy2DAsync(out, sizeof(double) * g->N, src, sizeof(double) * g->ld, sizeof(double) * g->N, g->N,
                         cudaMemcpyDeviceToHost, g->ctx->stream));
    CU(cudaStreamSynchronize(g->ctx->stream));
    for (int64_t i = 0; i < g->N; ++i)                  // tiles above the diagonal are never written on the device
        for (int64_t j = i + 1; j < g->N; ++j) out[i * g->N + j] = 0.0;
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// candidate sweep
// ------------------------------------------------------------------------------------------
template <int DT>
static void launch_ks(abo_ctx* c, const abo_gp* g, const double* dXc, int64_t c_begin, int64_t m_total, int bo,
                      double* Ks, double* pmean, int64_t mc_eff, int64_t mc, int npb, cudaStream_t stream) {
    if (g->p == 1)
        ks_build_kernel<DT, false><<<dim3(npb, (unsigned)(mc_eff / KS_CB)), 128, 0, stream>>>(
            gp_spec(g), g->dXsT, g->ldx, g->n, g->N, g->Npad, g->dAlpha, dXc, c_begin, m_total, bo, Ks, pmean, mc);
    else
        ks_build_kernel<DT, true><<<dim3(npb, (unsigned)(mc_eff / KS_CB)), 128, 0, stream>>>(
            gp_spec(g), g->dXsT, g->ldx, g->n, g->N, g->Npad, g->dAlpha, dXc, c_begin, m_total, bo, Ks, pmean, mc);
}

static int launch_ks_d(abo_ctx* c, const abo_gp* g, const double* dXc, int64_t c0, int64_t m, int bo, double* Ks, double* pmean,
                       int64_t mc_eff, int64_t mc, int npb, cudaStream_t st) {
    const int d = g->d;
    if (d <= 4) launch_ks<4>(c, g, dXc, c0, m, bo, Ks, pmean, mc_eff, mc, npb, st);
    else if (d <= 8) launch_ks<8>(c, g, dXc, c0, m, bo, Ks, pmean, mc_eff, mc, npb, st);
    else if (d <= 12) launch_ks<12>(c, g, dXc, c0, m, bo, Ks, pmean, mc_eff, mc, npb, st);
    else if (d <= 16) launch_ks<16>(c, g, dXc, c0, m, bo, Ks, pmean, mc_eff, mc, npb, st);
    else if (d <= 20) launch_ks<20>(c, g, dXc, c0, m, bo, Ks, pmean, mc_eff, mc, npb, st);
    else if (d <= 24) launch_ks<24>(c, g, dXc, c0, m, bo, Ks, pmean, mc_eff, mc, npb, st);
    else if (d <= 32) launch_ks<32>(c, g, dXc, c0, m, bo, Ks, pmean, mc_eff, mc, npb, st);
    else
        ks_build_generic_kernel<<<dim3(npb, (unsigned)(mc_eff / KS_CB)), 128, 0, st>>>(
            gp_spec(g), g->dXsT, g->ldx, g->n, g->N, g->Npad, g->dAlpha, dXc, c0, m, bo, Ks, pmean, mc);
    KL(c);
    return ABO_OK;
}

static double phi_prime0(int kind) {
    if (kind == K_SE) return -0.5;
    if (kind == K_M52 || kind == K_AM52 || kind == K_ADM52) return -5.0 / 6.0;
    return -7.0 / 10.0;
}

// ---- fused single-kernel sweep (sweep_fused.cuh): scalar GPs up to FS_MAX_NPAD observations (measured faster than the
//      three-kernel path at every size: n = 8192 97.9 % vs 95.6 % of the Dgemm peak for the whole step) ------------
static bool fused_applies(const abo_gp* g, int bo) {
    return g->p == 1 && bo == 0 && g->d <= 32 && g->Npad <= FS_MAX_NPAD;
}

// The acquisition of one sweep over a candidate output: its AcqSpec and, for ABO_ACQ_MES, the y*.  The MesSpec travels by
// value in the kernel parameters: no upload.
struct AcqSweep {
    AcqSpec a;
    MesSpec mes;                                                     // ABO_ACQ_MES only
};

// posterior mean / variance only (acq = -1) of candidate output bo: its prior mean and variance, -2 s_b^2 sigma^2 phi'(0) for
// the derivative output b of a GradientGP
static AcqSpec prior_spec(const abo_gp* g, int bo) {
    const double sb = (bo > 0 && bo - 1 < (int)g->sv.size() && g->d <= ARD_MAXD) ? g->sv[bo - 1] : g->s;
    return AcqSpec{-1, 0.0, 0.0, g->mean_c[bo], (bo == 0) ? g->scale : -2.0 * sb * sb * g->scale * phi_prime0(g->kind)};
}

// `a` with the acquisition acq_id: EI / PI params = {xi, best_y}, UCB {beta} (p1 = 0), MES {K, y*_1 .. y*_K} (the y* go to
// the MesSpec), GradientNormUCB {beta, unused}
static AcqSpec with_acq(AcqSpec a, int acq_id, const double* params) {
    a.acq = acq_id;
    a.p0 = params[0];
    a.p1 = (acq_id != ACQ_UCB) ? params[1] : 0.0;
    return a;
}

// (acq_id, params) of abo_acq_eval[_dev] / abo_acq_eval_grad, for candidate output bo.  ABO_ACQ_MES: K an integer-valued
// double in [1, MES_MAX_K], every y* finite.
static int acq_parse(const abo_gp* g, int acq_id, const double* params, int bo, AcqSweep* s) {
    if ((acq_id < ACQ_EI || acq_id > ACQ_UCB) && acq_id != ACQ_MES) return abo_fail(ABO_ERR_INVALID, "unknown acquisition id %d", acq_id);
    if (acq_id == ACQ_MES) {
        const double K = params[0];
        if (!(K >= 1.0 && K <= (double)MES_MAX_K && K == std::floor(K)))
            return abo_fail(ABO_ERR_INVALID, "MES needs params[0] = K, an integer in [1, %d]", MES_MAX_K);
        s->mes.K = (int)K;
        for (int k = 0; k < s->mes.K; ++k) {
            if (!std::isfinite(params[1 + k])) return abo_fail(ABO_ERR_INVALID, "MES y*[%d] is not finite", k);
            s->mes.ystar[k] = params[1 + k];
        }
    }
    s->a = with_acq(prior_spec(g, bo), acq_id, params);
    return ABO_OK;
}

static int sweep_fused_device(abo_gp* g, const double* dXc, int64_t m, const AcqSweep& s, double* d_mean, double* d_var,
                              double* d_score) {
    abo_ctx* c = g->ctx;
    cudaStream_t st = c->stream;
    FusedParams fp;
    fp.spec = gp_spec(g); fp.acq = s.a;
    fp.XsT = g->dXsT; fp.ldx = g->ldx; fp.n = g->n;
    fp.T = (int)((g->n + NB - 1) / NB);
    fp.Kld = (int)((g->n + 15) / 16 * 16);
    fp.Xc = dXc; fp.m = m; fp.beta = g->dBeta;
    fp.mean_out = d_mean; fp.var_out = d_var; fp.score_out = d_score;
    fp.ntiles = (int)((m + NB - 1) / NB);
    const int grid = std::min(c->sms, fp.ntiles);
    int rc;
    // private K* scratch: [CTA][2][128][Kld]; sized for the full grid so that the tensor map is stable between calls
    if ((rc = ws_get(c, WS_KS, sizeof(double) * (size_t)c->sms * 2 * NB * fp.Kld, (void**)&fp.scratch))) return rc;
    CUtensorMap tmA, tmB;
    if ((rc = make_tmap_k4(&tmA, g->dLinv, g->Npad, g->Npad, g->ld))) return rc;
    if ((rc = make_tmap_k4(&tmB, fp.scratch, fp.Kld, (int64_t)c->sms * 2 * NB, fp.Kld))) return rc;
    if ((rc = prof_mark(c)) || (rc = prof_mark(c))) return rc;            // class 0 (K* builder): inside the fused kernel
    if ((rc = prof_mark(c))) return rc;
    const auto run = [&](auto mes) {
        constexpr bool MES = std::is_same<decltype(mes), MesSpec>::value;
#define ABO_FS_RUN(DT) sweep_fused_kernel<DT, MES><<<grid, FS_THREADS, fused_smem_bytes<DT>(), st>>>(tmA, tmB, fp, mes)
        const int d = g->d;
        if (d <= 4) ABO_FS_RUN(4); else if (d <= 8) ABO_FS_RUN(8); else if (d <= 12) ABO_FS_RUN(12); else if (d <= 16) ABO_FS_RUN(16);
        else if (d <= 20) ABO_FS_RUN(20); else if (d <= 24) ABO_FS_RUN(24); else ABO_FS_RUN(32);
#undef ABO_FS_RUN
    };
    if (s.a.acq == ACQ_MES) run(s.mes); else run(NoMes{});
    KL(c);
    if ((rc = prof_mark(c))) return rc;
    if ((rc = prof_mark(c)) || (rc = prof_mark(c))) return rc;            // class 2 (epilogue): inside the fused kernel
    if (c->profile && c->prof_used >= 6 * 512) {
        CU(cudaStreamSynchronize(st));
        if ((rc = prof_collect(c))) return rc;
    }
    return ABO_OK;
}

// mean / var / scores for m device-resident candidates and candidate output bo, `s` the acquisition of output bo; any of the
// three outputs may be null (device pointers, length m)
int sweep_device(abo_gp* g, const double* dXc, int64_t m, int bo, const AcqSweep& s, double* d_mean, double* d_var,
                 double* d_score) {
    if (fused_applies(g, bo)) return sweep_fused_device(g, dXc, m, s, d_mean, d_var, d_score);
    abo_ctx* c = g->ctx;
    cudaStream_t st = c->stream;
    const int64_t Npad = g->Npad;
    const int T = (int)(Npad / NB);
    // chunk: enough tiles per launch (>= ~2048) that the persistent kernel's tail is small, K* buffer
    // bounded by 512 MB
    int64_t mc = (int64_t)NB * ((2048 + T - 1) / T);
    mc = std::min<int64_t>(mc, ((int64_t)(512ll << 20) / (Npad * 8)) / NB * NB);
    mc = std::max<int64_t>(NB, std::min<int64_t>(mc, 65536));
    mc = std::min<int64_t>(mc, (m + NB - 1) / NB * NB);
    const int64_t vpts = (Npad + g->p - 1) / g->p;                 // virtual points incl. padding columns
    const int npb = (int)((vpts + 127) / 128);
    // (Building the K* tile of chunk i+1 on a second stream while chunk i is contracted was measured: 514.5k vs
    //  513.9k candidates/s — DMMA and DFMA share the FP64 datapath, there is nothing to overlap — and removed.)
    double *Ks, *pmean, *sumsq;
    int rc;
    if ((rc = ws_get(c, WS_KS, sizeof(double) * (size_t)mc * Npad, (void**)&Ks))) return rc;
    if ((rc = ws_get(c, WS_PMEAN, sizeof(double) * (size_t)npb * mc, (void**)&pmean))) return rc;
    if ((rc = ws_get(c, WS_SUMSQ, sizeof(double) * (size_t)T * mc, (void**)&sumsq))) return rc;
    CUtensorMap tmA, tmB;
    if ((rc = make_tmap_k4(&tmA, g->dLinv, Npad, Npad, g->ld))) return rc;
    if ((rc = make_tmap_k4(&tmB, Ks, Npad, mc, Npad))) return rc;
    for (int64_t c0 = 0; c0 < m; c0 += mc) {
        const int64_t mvalid = std::min(mc, m - c0);
        const int64_t mc_eff = (mvalid + NB - 1) / NB * NB;
        if ((rc = prof_mark(c))) return rc;
        if ((rc = launch_ks_d(c, g, dXc, c0, m, bo, Ks, pmean, mc_eff, mc, npb, st))) return rc;
        if ((rc = prof_mark(c))) return rc;
        if ((rc = prof_mark(c))) return rc;
        TmaGemmParams sp{};                                 // sumsq[ib][c] = sum over row tile ib of (L^-1 K*^T)^2
        sp.batch = 1; sp.Mt = T; sp.Nt = (int)(mc_eff / NB); sp.K = (int)Npad; sp.flags = KHI_M;
        sp.C = sumsq; sp.ldc = mc;
        if ((rc = launch_gemm_tma<EPI_COLSUMSQ>(c, tmA, tmB, sp, st))) return rc;
        if ((rc = prof_mark(c))) return rc;
        if ((rc = prof_mark(c))) return rc;
        const auto epilogue = [&](auto mes) {
            acq_epilogue_kernel<std::is_same<decltype(mes), MesSpec>::value><<<(unsigned)((mvalid + 255) / 256), 256, 0, st>>>(
                s.a, pmean, npb, sumsq, T, mc, mvalid, d_mean ? d_mean + c0 : nullptr, d_var ? d_var + c0 : nullptr,
                d_score ? d_score + c0 : nullptr, mes);
        };
        if (s.a.acq == ACQ_MES) epilogue(s.mes); else epilogue(NoMes{});
        KL(c);
        if ((rc = prof_mark(c))) return rc;
        if (c->profile && c->prof_used >= 6 * 512) {       // bound the event pool
            CU(cudaStreamSynchronize(st));
            if ((rc = prof_collect(c))) return rc;
        }
    }
    CU(cudaGetLastError());
    return ABO_OK;
}

// host candidates per piece of sweep_host_pieces
constexpr int64_t HOST_PIECE = 262144;
static int sweep_host_pieces(abo_gp* g, const double* Xc, int64_t m, const AcqSweep& s, double* h_mean, double* h_var,
                             double* h_scores, int64_t k, int64_t* top_idx, double* top_val);

extern "C" int32_t abo_gp_posterior(abo_gp* g, const double* Xc, int64_t m, int32_t outputs, double* mean, double* var) {
    if (!g || !Xc) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior (call update first)");
    if (outputs != 1 && outputs != g->p) return abo_fail(ABO_ERR_INVALID, "outputs must be 1 or p");
    if (m <= 0) return ABO_OK;
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    if (outputs == 1 && m > HOST_PIECE && !c->profile)
        return sweep_host_pieces(g, Xc, m, AcqSweep{prior_spec(g, 0)}, mean, var, nullptr, 0, nullptr, nullptr);
    cudaStream_t st = c->stream;
    double *dXc, *dm, *dv;
    int rc;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)m * g->d, (void**)&dXc))) return rc;
    if ((rc = ws_get(c, WS_OUT_A, sizeof(double) * (size_t)m * outputs, (void**)&dm))) return rc;
    if ((rc = ws_get(c, WS_OUT_B, sizeof(double) * (size_t)m * outputs, (void**)&dv))) return rc;
    CU(cudaMemcpyAsync(dXc, Xc, sizeof(double) * m * g->d, cudaMemcpyHostToDevice, st));
    for (int bo = 0; bo < outputs; ++bo)
        if ((rc = sweep_device(g, dXc, m, bo, AcqSweep{prior_spec(g, bo)}, dm + (int64_t)bo * m, dv + (int64_t)bo * m, nullptr)))
            return rc;
    if (mean) CU(cudaMemcpyAsync(mean, dm, sizeof(double) * m * outputs, cudaMemcpyDeviceToHost, st));
    if (var) CU(cudaMemcpyAsync(var, dv, sizeof(double) * m * outputs, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ABO_OK;
}

// W = L^-1 K*^T  [Npad][ncol]  (k <= row): both operands k-contiguous -> the persistent TMA GEMM.
// W and / or its transpose Wt [ncol][Npad] (nullable each).
static int linv_times_ks(abo_ctx* c, const abo_gp* g, const double* Ks, int64_t ncol, double* W, cudaStream_t st, double* Wt = nullptr) {
    CUtensorMap tmX, tmK;
    int rc;
    if ((rc = make_tmap_k4(&tmX, g->dLinv, g->Npad, g->Npad, g->ld)) || (rc = make_tmap_k4(&tmK, Ks, g->Npad, ncol, g->Npad))) return rc;
    TmaGemmParams w{};
    w.batch = 1; w.alpha = 1.0; w.beta = 0.0; w.Mt = (int)(g->Npad / NB); w.Nt = (int)(ncol / NB); w.K = (int)g->Npad; w.flags = KHI_M;
    w.C = W; w.ldc = ncol;
    w.CT = Wt; w.ldct = g->Npad;
    return launch_gemm_tma(c, tmX, tmK, w, st);
}

// ------------------------------------------------------------------------------------------
// acquisition value + analytic gradient for a batch of points
// ------------------------------------------------------------------------------------------
extern "C" int32_t abo_acq_eval_grad(abo_gp* g, int32_t acq_id, const double* params, const double* Xc, int64_t m,
                                     double* scores, double* grad, double* mean, double* var) {
    if (!g || !Xc || !params || !scores || !grad) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior (call update first)");
    AcqSweep s;
    if (const int rc = acq_parse(g, acq_id, params, 0, &s)) return rc;
    if (g->d > AG_MAXD) return abo_fail(ABO_ERR_INVALID, "abo_acq_eval_grad supports d <= %d", AG_MAXD);
    if (m <= 0) return ABO_OK;
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t Npad = g->Npad;
    const int d = g->d;
    const int64_t mc = 2048;                                   // points per pass
    const int64_t vpts = (Npad + g->p - 1) / g->p;
    const int npb = (int)((vpts + 127) / 128);                 // K* builder point blocks (incl. padding columns)
    const int npbg = (int)((g->n + 127) / 128);                // gradient kernel point blocks
    double *dXc, *Ks, *pmean, *W, *Z, *part, *out;
    int rc;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)m * d, (void**)&dXc))) return rc;
    if ((rc = ws_get(c, WS_KS, sizeof(double) * (size_t)mc * Npad, (void**)&Ks))) return rc;
    if ((rc = ws_get(c, WS_PMEAN, sizeof(double) * (size_t)npb * mc, (void**)&pmean))) return rc;
    if ((rc = ws_get(c, WS_GRAD_W, sizeof(double) * (size_t)mc * Npad, (void**)&W))) return rc;
    if ((rc = ws_get(c, WS_GRAD_Z, sizeof(double) * (size_t)mc * Npad, (void**)&Z))) return rc;
    if ((rc = ws_get(c, WS_GRAD_PART, sizeof(double) * (size_t)npbg * mc * 2 * AG_MAXD, (void**)&part))) return rc;
    // out: colsq[mc] | score[m] | mean[m] | var[m] | grad[m*d]
    if ((rc = ws_get(c, WS_GRAD_OUT, sizeof(double) * (size_t)(mc + 3 * m + m * d), (void**)&out))) return rc;
    double *colsq = out, *dS = out + mc, *dM = dS + m, *dV = dM + m, *dG = dV + m;
    CU(cudaMemcpyAsync(dXc, Xc, sizeof(double) * m * d, cudaMemcpyHostToDevice, st));
    for (int64_t c0 = 0; c0 < m; c0 += mc) {
        const int64_t mvalid = std::min(mc, m - c0);
        const int64_t mpad = (mvalid + NB - 1) / NB * NB;
        if ((rc = launch_ks_d(c, g, dXc, c0, m, 0, Ks, pmean, mpad, mc, npb, st))) return rc;
        KL(c);
        if ((rc = linv_times_ks(c, g, Ks, mpad, W, st))) return rc;      // W = L^-1 K*^T   (k <= row)
        colsumsq_kernel<<<(unsigned)((mpad + 127) / 128), 128, 0, st>>>(W, Npad, mpad, colsq);
        KL(c);
        GemmParams z{};                                        // Z = L^-T W      (k >= row)
        z.A = g->dLinv; z.lda = g->ld; z.B = W; z.ldb = mpad; z.C = Z; z.ldc = mpad;
        z.M = (int)Npad; z.N = (int)mpad; z.K = (int)Npad; z.alpha = 1.0; z.beta = 0.0; z.flags = KLO_M;
        CU((launch_gemm(z, 1, st)));
        KL(c);
        acq_grad_partial_kernel<<<dim3(npbg, (unsigned)mpad), 128, 0, st>>>(gp_spec(g), g->dXsT, g->ldx, g->n, g->dAlpha, Z,
                                                                           mpad, dXc + c0 * d, mvalid, part);
        KL(c);
        const auto finish = [&](auto mes) {
            acq_grad_finish_kernel<std::is_same<decltype(mes), MesSpec>::value><<<(unsigned)((mvalid + 127) / 128), 128, 0, st>>>(
                s.a, d, pmean, npb, colsq, part, npbg, mc, mpad, mvalid, dS + c0, dG + c0 * d, dM + c0, dV + c0, mes);
        };
        if (s.a.acq == ACQ_MES) finish(s.mes); else finish(NoMes{});
        KL(c);
    }
    CU(cudaMemcpyAsync(scores, dS, sizeof(double) * m, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(grad, dG, sizeof(double) * m * d, cudaMemcpyDeviceToHost, st));
    if (mean) CU(cudaMemcpyAsync(mean, dM, sizeof(double) * m, cudaMemcpyDeviceToHost, st));
    if (var) CU(cudaMemcpyAsync(var, dV, sizeof(double) * m, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ABO_OK;
}

extern "C" int32_t abo_gp_posterior_cov(abo_gp* g, const double* Xc, int64_t m, int32_t outputs, double* cov) {
    if (!g || !Xc || !cov) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior (call update first)");
    if (outputs != 1 && outputs != g->p) return abo_fail(ABO_ERR_INVALID, "outputs must be 1 or p");
    if (m <= 0) return ABO_OK;
    const int64_t mp = (m + KS_CB - 1) / KS_CB * KS_CB;           // rows per output block (builder granularity)
    const int64_t Mtot = mp * outputs, Mpad = (Mtot + NB - 1) / NB * NB;
    if (m * outputs > 8192) return abo_fail(ABO_ERR_INVALID, "posterior covariance is limited to m*outputs <= 8192");
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t Npad = g->Npad;
    const int d = g->d;
    const int64_t vpts = (Npad + g->p - 1) / g->p;
    const int npb = (int)((vpts + 127) / 128);
    double *dXc, *Ks, *pmean, *W, *G, *dcov;
    int rc;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)m * d, (void**)&dXc))) return rc;
    if ((rc = ws_get(c, WS_KS, sizeof(double) * (size_t)Mpad * Npad, (void**)&Ks))) return rc;
    if ((rc = ws_get(c, WS_PMEAN, sizeof(double) * (size_t)npb * Mpad, (void**)&pmean))) return rc;
    if ((rc = ws_get(c, WS_GRAD_W, sizeof(double) * (size_t)Mpad * Npad, (void**)&W))) return rc;
    if ((rc = ws_get(c, WS_GRAD_Z, sizeof(double) * (size_t)Mpad * Mpad, (void**)&G))) return rc;
    if ((rc = ws_get(c, WS_GRAD_OUT, sizeof(double) * (size_t)(m * outputs) * (m * outputs), (void**)&dcov))) return rc;
    CU(cudaMemcpyAsync(dXc, Xc, sizeof(double) * m * d, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(Ks, 0, sizeof(double) * (size_t)Mpad * Npad, st));
    for (int bo = 0; bo < outputs; ++bo) {
        double* Kb = Ks + (size_t)bo * mp * Npad;
        double* pm = pmean + (size_t)bo * mp;                      // (unused partial means)
        if ((rc = launch_ks_d(c, g, dXc, 0, m, bo, Kb, pm, mp, Mpad, npb, st))) return rc;
    }
    if ((rc = linv_times_ks(c, g, Ks, Mpad, W, st))) return rc;          // W = L^-1 K*^T
    GemmParams q{};                                                // G = W^T W
    q.A = W; q.lda = Mpad; q.B = W; q.ldb = Mpad; q.C = G; q.ldc = Mpad;
    q.M = (int)Mpad; q.N = (int)Mpad; q.K = (int)Npad; q.alpha = 1.0; q.beta = 0.0; q.flags = 0;
    CU((launch_gemm(q, 1, st)));
    KL(c);
    const int64_t Mo = m * outputs;
    cov_finish_kernel<<<(unsigned)((Mo * Mo + 255) / 256), 256, 0, st>>>(gp_spec(g), dXc, m, outputs, mp, G, Mpad, dcov, Mo, 0, 0.0);
    KL(c);
    CU(cudaMemcpyAsync(cov, dcov, sizeof(double) * Mo * Mo, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// Monte-Carlo batch expected improvement over B batches of q points (qei.cuh).  Once per call: the S x q base normals
// (key offset 2^62).  Per chunk of whole batches (about 2048 points):
//   K* value rows -> W = L^-1 K*^T (TMA GEMM) -> q x q Gram blocks of W^T W and the means -> per-batch Cholesky, estimate
//   and, with a gradient, C = d qEI / d Sigma -> Z = L^-T W (DMMA GEMM) -> R = (C + C^T) Z per batch (into the K* buffer)
//   -> acq_grad_partial_kernel on R -> the per-point gradient.
// ------------------------------------------------------------------------------------------
constexpr int64_t QEI_MAX_S = 4096;
constexpr uint64_t QEI_KEY_OFFSET = 1ull << 62;
extern "C" int32_t abo_acq_qei(abo_gp* g, const double* params, int32_t q, const double* Xb, int64_t B, int64_t S,
                               uint64_t seed, double jitter, double* values, double* grad, double* jitter_used) {
    if (!g || !params || !Xb || !values) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior (call update first)");
    if (q < 1 || q > QEI_MAXQ) return abo_fail(ABO_ERR_INVALID, "qEI needs 1 <= q <= %d", QEI_MAXQ);
    if (S < 1 || S > QEI_MAX_S) return abo_fail(ABO_ERR_INVALID, "qEI needs 1 <= S <= %lld", (long long)QEI_MAX_S);
    if (g->d > AG_MAXD) return abo_fail(ABO_ERR_INVALID, "abo_acq_qei supports d <= %d", AG_MAXD);
    if (!(jitter > 0) || !std::isfinite(jitter)) return abo_fail(ABO_ERR_INVALID, "jitter must be positive and finite");
    if (B <= 0) return ABO_OK;
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t Npad = g->Npad, M = B * q;
    const int d = g->d;
    const int64_t nbc = std::max<int64_t>(1, 2048 / q);                 // batches per chunk
    const int64_t mc = (nbc * q + NB - 1) / NB * NB;                    // columns per chunk, padded
    const int64_t vpts = (Npad + g->p - 1) / g->p;
    const int npb = (int)((vpts + 127) / 128);
    const int npbg = (int)((g->n + 127) / 128);
    const int ldz = (q + 3) / 4 * 4;
    const bool want_grad = grad != nullptr;
    double *dXb, *Ks, *pmean, *W, *Z = nullptr, *part = nullptr, *out, *zn, *bs;
    int rc;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)M * d, (void**)&dXb)) ||
        (rc = ws_get(c, WS_KS, sizeof(double) * (size_t)mc * Npad, (void**)&Ks)) ||
        (rc = ws_get(c, WS_PMEAN, sizeof(double) * (size_t)npb * mc, (void**)&pmean)) ||
        (rc = ws_get(c, WS_GRAD_W, sizeof(double) * (size_t)mc * Npad, (void**)&W)) ||
        (rc = ws_get(c, WS_QEI_Z, sizeof(double) * (size_t)S * ldz, (void**)&zn)) ||
        // per chunk: Gram [nbc q q] | mu [nbc q] | C [nbc q q] | d mu [nbc q]
        (rc = ws_get(c, WS_QEI_BATCH, sizeof(double) * (size_t)nbc * q * (2 * q + 2), (void**)&bs)) ||
        // values [B] | tau [B] | grad [B q d]
        (rc = ws_get(c, WS_GRAD_OUT, sizeof(double) * (size_t)(2 * B + (want_grad ? M * d : 0)), (void**)&out)))
        return rc;
    if (want_grad &&
        ((rc = ws_get(c, WS_GRAD_Z, sizeof(double) * (size_t)mc * Npad, (void**)&Z)) ||
         (rc = ws_get(c, WS_GRAD_PART, sizeof(double) * (size_t)npbg * mc * 2 * AG_MAXD, (void**)&part))))
        return rc;
    double *Gm = bs, *mu = Gm + nbc * q * q, *Cb = mu + nbc * q, *dmu = Cb + nbc * q * q;
    double *dV = out, *dT = out + B, *dG = out + 2 * B;
    const double delta = params[1] - params[0];                        // (best_y - xi), EI's improvement convention
    CU(cudaMemcpyAsync(dXb, Xb, sizeof(double) * M * d, cudaMemcpyHostToDevice, st));
    philox_normal_kernel<<<(unsigned)((S * ldz / 4 + 255) / 256), 256, 0, st>>>(seed, QEI_KEY_OFFSET, 0, 1.0, S, q, S, ldz, ldz, zn);
    KL(c);
    const size_t smem = sizeof(double) * 4 * (size_t)q * (q + 1);
    for (int64_t b0 = 0; b0 < B; b0 += nbc) {
        const int64_t nb = std::min(nbc, B - b0), c0 = b0 * q, ncols = nb * q;
        const int64_t mpad = (ncols + NB - 1) / NB * NB;
        if ((rc = launch_ks_d(c, g, dXb, c0, M, 0, Ks, pmean, mpad, mc, npb, st))) return rc;
        if ((rc = linv_times_ks(c, g, Ks, mpad, W, st))) return rc;                  // W = L^-1 K*^T   [Npad][mpad]
        qei_gram_kernel<<<(unsigned)nb, 128, 0, st>>>(W, Npad, mpad, q, pmean, npb, mc, g->mean_c[0], Gm, mu);
        KL(c);
        qei_batch_kernel<<<(unsigned)nb, 32, smem, st>>>(gp_spec(g), dXb + c0 * d, q, Gm, mu, zn, S, ldz, delta, jitter,
                                                         want_grad ? 1 : 0, dV + b0, dT + b0, dmu, Cb);
        KL(c);
        if (!want_grad) continue;
        GemmParams z{};                                                                // Z = L^-T W      (k >= row)
        z.A = g->dLinv; z.lda = g->ld; z.B = W; z.ldb = mpad; z.C = Z; z.ldc = mpad;
        z.M = (int)Npad; z.N = (int)mpad; z.K = (int)Npad; z.alpha = 1.0; z.beta = 0.0; z.flags = KLO_M;
        CU((launch_gemm(z, 1, st)));
        KL(c);
        double* R = Ks;                                                                // K* is consumed: R takes its place
        qei_combine_kernel<<<dim3((unsigned)((ncols + 127) / 128), (unsigned)Npad), 128, 0, st>>>(Z, mpad, q, ncols, Cb, R);
        KL(c);
        acq_grad_partial_kernel<<<dim3(npbg, (unsigned)mpad), 128, 0, st>>>(gp_spec(g), g->dXsT, g->ldx, g->n, g->dAlpha, R,
                                                                           mpad, dXb + c0 * d, ncols, part);
        KL(c);
        qei_grad_finish_kernel<<<(unsigned)((ncols + 127) / 128), 128, 0, st>>>(gp_spec(g), dXb + c0 * d, q, ncols, part, npbg,
                                                                                mpad, dmu, Cb, dT + b0, dG + c0 * d);
        KL(c);
    }
    CU(cudaMemcpyAsync(values, dV, sizeof(double) * B, cudaMemcpyDeviceToHost, st));
    if (jitter_used) CU(cudaMemcpyAsync(jitter_used, dT, sizeof(double) * B, cudaMemcpyDeviceToHost, st));
    if (want_grad) CU(cudaMemcpyAsync(grad, dG, sizeof(double) * M * d, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// joint posterior samples of the value output over a candidate set (sample.cuh):
//   K* (value rows) -> W^T = (L^-1 K*^T)^T -> G = W^T W (lower tiles) -> Sigma + tau I (lower tiles, identity padding)
//   -> look-ahead Cholesky (strict upper part of its diagonal tiles zeroed) -> L_Sigma Z^T, stored transposed: draws F [S][m] sample-major -> + mu, per-draw argmin.
// Every product is a full-k GEMM tile per (candidate tile, draw tile): no reduction order depends on S, so the first S'
// draws of a call are those of a call with S' draws, bit for bit.
// ------------------------------------------------------------------------------------------
constexpr int64_t SAMPLE_MAX_M = 16384, SAMPLE_MAX_S = 4096;
constexpr int SAMPLE_JITTER_STEPS = 7;       // tau_k = jitter * sigma^2 * 10^k, k = 0 .. 6
static int gp_posterior_sample_run(abo_gp* g, const double* Xc, int64_t m, int64_t S, uint64_t seed, double jitter,
                                   double* samples, int64_t* argmin_idx, double* argmin_val, double* jitter_used);
extern "C" int32_t abo_gp_posterior_sample(abo_gp* g, const double* Xc, int64_t m, int64_t S, uint64_t seed, double jitter,
                                           double* samples, int64_t* argmin_idx, double* argmin_val, double* jitter_used) {
    const int rc = gp_posterior_sample_run(g, Xc, m, S, seed, jitter, samples, argmin_idx, argmin_val, jitter_used);
    if (rc && g && g->ctx) {
        // as abo_gp_fit: no factorisation side stream may still be writing workspace slots the next call reuses
        const std::string keep = g_err;
        ctx_sync_all(g->ctx);
        cudaGetLastError();
        g_err = keep;
    }
    return rc;
}
static int gp_posterior_sample_run(abo_gp* g, const double* Xc, int64_t m, int64_t S, uint64_t seed, double jitter,
                                   double* samples, int64_t* argmin_idx, double* argmin_val, double* jitter_used) {
    if (!g || !Xc) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior (call update first)");
    if (!(jitter > 0) || !std::isfinite(jitter)) return abo_fail(ABO_ERR_INVALID, "jitter must be positive and finite");
    if (m > SAMPLE_MAX_M || S > SAMPLE_MAX_S)
        return abo_fail(ABO_ERR_INVALID, "joint samples are limited to m <= %lld candidates and S <= %lld draws",
                        (long long)SAMPLE_MAX_M, (long long)SAMPLE_MAX_S);
    if (m <= 0 || S <= 0) return ABO_OK;
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int64_t Npad = g->Npad, Mpad = (m + NB - 1) / NB * NB, Spad = (S + NB - 1) / NB * NB;
    const int T = (int)(Mpad / NB);
    const int npb = (int)(((Npad + g->p - 1) / g->p + 127) / 128);
    double *dXc, *Ks, *pmean, *Wt, *G, *Sig, *Z, *F, *mu, *amin, *Dinv;
    int* dinfo;
    int rc;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)m * g->d, (void**)&dXc)) ||
        (rc = ws_get(c, WS_KS, sizeof(double) * (size_t)Mpad * Npad, (void**)&Ks)) ||
        (rc = ws_get(c, WS_PMEAN, sizeof(double) * (size_t)npb * Mpad, (void**)&pmean)) ||
        (rc = ws_get(c, WS_GRAD_W, sizeof(double) * (size_t)Mpad * Npad, (void**)&Wt)) ||
        (rc = ws_get(c, WS_SAMPLE_G, sizeof(double) * (size_t)Mpad * Mpad, (void**)&G)) ||
        (rc = ws_get(c, WS_SAMPLE_SIGMA, sizeof(double) * (size_t)Mpad * Mpad, (void**)&Sig)) ||
        (rc = ws_get(c, WS_SAMPLE_Z, sizeof(double) * (size_t)Spad * Mpad, (void**)&Z)) ||
        (rc = ws_get(c, WS_SAMPLE_F, sizeof(double) * (size_t)Spad * Mpad, (void**)&F)) ||
        (rc = ws_get(c, WS_OUT_B, sizeof(double) * (size_t)Mpad, (void**)&mu)) ||
        (rc = ws_get(c, WS_OUT_A, sizeof(double) * (size_t)2 * S, (void**)&amin)) ||
        (rc = ws_get(c, WS_DINV, sizeof(double) * (size_t)T * NB * NB, (void**)&Dinv)) ||
        (rc = ws_get(c, WS_INFO, sizeof(int) * 16, (void**)&dinfo)))
        return rc;
    CU(cudaMemcpyAsync(dXc, Xc, sizeof(double) * m * g->d, cudaMemcpyHostToDevice, st));
    // K* value rows for all Mpad candidate rows (rows >= m are built at the origin; the padding of Sigma overwrites them)
    if ((rc = launch_ks_d(c, g, dXc, 0, m, 0, Ks, pmean, Mpad, Mpad, npb, st))) return rc;
    if ((rc = linv_times_ks(c, g, Ks, Mpad, nullptr, st, Wt))) return rc;             // W^T [Mpad][Npad]
    {
        CUtensorMap tmW;
        if ((rc = make_tmap_k4(&tmW, Wt, Npad, Mpad, Npad))) return rc;
        TmaGemmParams q{};                                                               // G = W^T W, lower tiles
        q.Mt = T; q.Nt = T; q.batch = 1; q.K = (int)Npad; q.flags = LOWER_ONLY; q.alpha = 1.0; q.beta = 0.0;
        q.C = G; q.ldc = Mpad;
        if ((rc = launch_gemm_tma(c, tmW, tmW, q, st))) return rc;
    }
    {
        // mu = m + sum of the partial means
        acq_epilogue_kernel<false><<<(unsigned)((m + 255) / 256), 256, 0, st>>>(prior_spec(g, 0), pmean, npb, nullptr, 0, Mpad, m, mu,
                                                                                nullptr, nullptr, NoMes{});
        KL(c);
    }
    philox_normal_kernel<<<(unsigned)((Spad * Mpad / 4 + 255) / 256), 256, 0, st>>>(seed, 0, 0, 1.0, S, m, Spad, Mpad, Mpad, Z);
    KL(c);
    double tau = 0.0;
    for (int k = 0;; ++k) {
        double p10 = 1.0;
        for (int e = 0; e < k; ++e) p10 *= 10.0;
        tau = jitter * g->scale * p10;
        cov_finish_kernel<<<(unsigned)((Mpad * Mpad + 255) / 256), 256, 0, st>>>(gp_spec(g), dXc, m, 1, Mpad, G, Mpad, Sig, Mpad,
                                                                                 Mpad, tau);
        KL(c);
        CU(cudaMemsetAsync(dinfo, 0, sizeof(int) * 16, st));
        if ((rc = potrf_lookahead(c, Sig, Mpad, Mpad, Dinv, dinfo))) return rc;
        int hinfo = 0;
        CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (hinfo == 0) break;
        ctx_sync_all(c);
        if (k + 1 == SAMPLE_JITTER_STEPS)
            return abo_fail(ABO_ERR_NOT_POSDEF, "posterior covariance + %g I is not positive definite (pivot %d)", tau, hinfo);
    }
    zero_diag_upper_kernel<<<T, 256, 0, st>>>(Sig, Mpad);
    KL(c);
    {
        CUtensorMap tmL, tmZ;
        if ((rc = make_tmap_k4(&tmL, Sig, Mpad, Mpad, Mpad)) || (rc = make_tmap_k4(&tmZ, Z, Mpad, Spad, Mpad))) return rc;
        TmaGemmParams f{};                                                               // F = (L_Sigma Z^T)^T  [Spad][Mpad]
        f.Mt = T; f.Nt = (int)(Spad / NB); f.batch = 1; f.K = (int)Mpad; f.flags = KHI_M; f.alpha = 1.0; f.beta = 0.0;
        f.C = nullptr; f.CT = F; f.ldct = Mpad;
        if ((rc = launch_gemm_tma(c, tmL, tmZ, f, st))) return rc;
    }
    long long* aidx = reinterpret_cast<long long*>(amin);
    sample_finish_kernel<<<(unsigned)S, SF_THREADS, 0, st>>>(F, Mpad, mu, 0.0, m, 0, 0, aidx, amin + S);
    KL(c);
    if (samples)
        CU(cudaMemcpy2DAsync(samples, sizeof(double) * m, F, sizeof(double) * Mpad, sizeof(double) * m, S, cudaMemcpyDeviceToHost, st));
    if (argmin_idx) CU(cudaMemcpyAsync(argmin_idx, aidx, sizeof(int64_t) * S, cudaMemcpyDeviceToHost, st));
    if (argmin_val) CU(cudaMemcpyAsync(argmin_val, amin + S, sizeof(double) * S, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (jitter_used) *jitter_used = tau;
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// pathwise posterior draws over any number of candidates (sample.cuh), f_s(x) = mean_c + k(x, X)(alpha - v_s) + phi(x) theta'_s:
//   once per call   features (Om, b) -> Phi(X) [Npad][Lpad], training rows in point-major output order
//                   -> Bc[s][Npad + l] = theta'_s[l] and Rt[s][i] = eps_s[i] (Philox) -> Rt += Theta' Phi(X)^T (TMA GEMM)
//                   -> Y = L^-1 Rt^T (TMA GEMM) -> V = L^-T Y (the cp.async DMMA GEMM, which reads L^-1 transposed)
//                   -> Bc[s][k] = alpha[k] - V[k][s], k < Npad
//   per chunk       K* value rows and Phi* of mc candidates -> F = Bc [K* | Phi*]^T [Spad][mc]: two TMA GEMM launches over
//                   k in [0, Npad) and [Npad, Npad + Lpad), the second accumulating -> + mean_c, running per-draw argmin.
// Each element of F is one fixed-order reduction over k of quantities that depend on its own candidate and draw only.
// ------------------------------------------------------------------------------------------
constexpr int64_t PATH_MAX_S = 4096, PATH_MAX_L = 16384;
constexpr size_t PATH_CHUNK_BYTES = (size_t)6 << 30;     // K*, Phi* and F of one candidate chunk
struct PathPlan {
    int64_t Lpad, Spad, ldb, mc;
    int npb;
    double *Om, *bf, *Phi, *Bc, *Ks, *pmean, *F, *amin;
    CUtensorMap tmB, tmK, tmP;
};

static int pathwise_prepare(abo_gp* g, int64_t m, int64_t S, int64_t L, uint64_t seed, PathPlan& P) {
    abo_ctx* c = g->ctx;
    cudaStream_t st = c->stream;
    const int64_t Npad = g->Npad, N = g->N;
    const int d = g->d;
    const int64_t Lpad = (L + NB - 1) / NB * NB, Spad = (S + NB - 1) / NB * NB, ldb = Npad + Lpad;
    // chunk: three waves of (draw tile, candidate tile) work items, K* + Phi* + F within PATH_CHUNK_BYTES
    const int64_t ts = Spad / NB;
    int64_t mc = NB * ((3 * c->sms + ts - 1) / ts);
    mc = std::min<int64_t>(mc, (int64_t)(PATH_CHUNK_BYTES / (sizeof(double) * (size_t)(Npad + Lpad + Spad))) / NB * NB);
    mc = std::max<int64_t>(NB, std::min<int64_t>(mc, (m + NB - 1) / NB * NB));
    P.Lpad = Lpad; P.Spad = Spad; P.ldb = ldb; P.mc = mc;
    P.npb = (int)(((Npad + g->p - 1) / g->p + 127) / 128);
    double *R, *Y;
    int rc;
    if ((rc = ws_get(c, WS_PATH_FEAT, sizeof(double) * (size_t)Lpad * (d + 1), (void**)&P.Om)) ||
        (rc = ws_get(c, WS_PATH_PHI, sizeof(double) * (size_t)std::max(Npad, mc) * Lpad, (void**)&P.Phi)) ||
        (rc = ws_get(c, WS_PATH_COEF, sizeof(double) * (size_t)Spad * ldb, (void**)&P.Bc)) ||
        (rc = ws_get(c, WS_PATH_R, sizeof(double) * (size_t)Spad * Npad, (void**)&R)) ||
        (rc = ws_get(c, WS_PATH_Y, sizeof(double) * (size_t)Npad * Spad, (void**)&Y)) ||
        (rc = ws_get(c, WS_KS, sizeof(double) * (size_t)mc * Npad, (void**)&P.Ks)) ||
        (rc = ws_get(c, WS_PMEAN, sizeof(double) * (size_t)P.npb * mc, (void**)&P.pmean)) ||
        (rc = ws_get(c, WS_PATH_F, sizeof(double) * (size_t)Spad * mc, (void**)&P.F)) ||
        (rc = ws_get(c, WS_OUT_A, sizeof(double) * (size_t)2 * S, (void**)&P.amin)))
        return rc;
    P.bf = P.Om + Lpad * d;
    const int kdf = g->kind == K_SE ? 0 : (g->kind == K_M52 || g->kind == K_AM52 || g->kind == K_ADM52) ? 5 : 7;
    rff_params_kernel<<<(unsigned)(Lpad / 128), 128, 0, st>>>(seed, d, kdf, L, Lpad, P.Om, P.bf);
    KL(c);
    const int64_t vpts = (Npad + g->p - 1) / g->p;
    rff_build_kernel<<<dim3((unsigned)(Lpad / 128), (unsigned)((vpts + RFF_PB - 1) / RFF_PB)), 128, 0, st>>>(
        gp_spec(g), P.Om, P.bf, Lpad, g->dXsT, 1, g->ldx, 0, g->n, g->p, Npad, P.Phi);
    KL(c);
    const uint64_t draw_key = 1ull << 63;
    philox_normal_kernel<<<(unsigned)((Spad * Lpad / 4 + 255) / 256), 256, 0, st>>>(seed, draw_key, 0, std::sqrt(2.0 * g->scale / (double)L),
                                                                                   S, L, Spad, Lpad, ldb, P.Bc + Npad);
    KL(c);
    philox_normal_kernel<<<(unsigned)((Spad * Npad / 4 + 255) / 256), 256, 0, st>>>(seed, draw_key, L, std::sqrt(g->noise),
                                                                                   S, N, Spad, Npad, Npad, R);
    KL(c);
    CUtensorMap tmPX;
    if ((rc = make_tmap_k4(&P.tmB, P.Bc, ldb, Spad, ldb)) || (rc = make_tmap_k4(&tmPX, P.Phi, Lpad, Npad, Lpad))) return rc;
    {
        TmaGemmParams q{};                                                   // Rt = E + Theta' Phi(X)^T  [Spad][Npad]
        q.Mt = (int)(Spad / NB); q.Nt = (int)(Npad / NB); q.batch = 1; q.K = (int)Lpad; q.a_col0 = (int)Npad;
        q.alpha = 1.0; q.beta = 1.0; q.C = R; q.ldc = Npad;
        if ((rc = launch_gemm_tma(c, P.tmB, tmPX, q, st))) return rc;
    }
    if ((rc = linv_times_ks(c, g, R, Spad, Y, st))) return rc;             // Y = L^-1 R  [Npad][Spad]
    {
        GemmParams z{};                                                      // V = L^-T Y  [Npad][Spad], into R's slot
        z.A = g->dLinv; z.lda = g->ld; z.B = Y; z.ldb = Spad; z.C = R; z.ldc = Spad;
        z.M = (int)Npad; z.N = (int)Spad; z.K = (int)Npad; z.alpha = 1.0; z.beta = 0.0; z.flags = KLO_M;
        CU((launch_gemm(z, 1, st)));
        KL(c);
    }
    pathwise_coef_kernel<<<dim3((unsigned)(Npad / 32), (unsigned)(Spad / 32)), dim3(32, 8), 0, st>>>(g->dAlpha, N, R, Npad, Spad,
                                                                                                  P.Bc, ldb);
    KL(c);
    if ((rc = make_tmap_k4(&P.tmK, P.Ks, Npad, mc, Npad)) || (rc = make_tmap_k4(&P.tmP, P.Phi, Lpad, mc, Lpad))) return rc;
    return ABO_OK;
}

// the draws at m device-resident candidates dXc, global indices off .. off + m - 1; samples (nullable) is the caller's
// S x ldo output (host or device memory, `kind`), written at column off
static int pathwise_chunks(abo_gp* g, const PathPlan& P, const double* dXc, int64_t m, int64_t S, int64_t off, double* samples,
                           int64_t ldo, cudaMemcpyKind kind, int64_t* nchunk) {
    abo_ctx* c = g->ctx;
    cudaStream_t st = c->stream;
    const int64_t Npad = g->Npad, mc = P.mc;
    long long* aidx = reinterpret_cast<long long*>(P.amin);
    int rc;
    for (int64_t c0 = 0; c0 < m; c0 += mc) {
        const int64_t mvalid = std::min(mc, m - c0), mc_eff = (mvalid + NB - 1) / NB * NB;
        if ((rc = launch_ks_d(c, g, dXc, c0, m, 0, P.Ks, P.pmean, mc_eff, mc, P.npb, st))) return rc;
        rff_build_kernel<<<dim3((unsigned)(P.Lpad / 128), (unsigned)(mc_eff / RFF_PB)), 128, 0, st>>>(
            gp_spec(g), P.Om, P.bf, P.Lpad, dXc + c0 * g->d, g->d, 1, 1, mvalid, 1, mc_eff, P.Phi);
        KL(c);
        TmaGemmParams q{};                                                   // F = Bc[:, 0:Npad] K*^T   [Spad][mc]
        q.Mt = (int)(P.Spad / NB); q.Nt = (int)(mc_eff / NB); q.batch = 1; q.K = (int)Npad;
        q.alpha = 1.0; q.beta = 0.0; q.C = P.F; q.ldc = mc;
        if ((rc = launch_gemm_tma(c, P.tmB, P.tmK, q, st))) return rc;
        q.K = (int)P.Lpad; q.a_col0 = (int)Npad; q.beta = 1.0;               //   += Bc[:, Npad:] Phi*^T
        if ((rc = launch_gemm_tma(c, P.tmB, P.tmP, q, st))) return rc;
        sample_finish_kernel<<<(unsigned)S, SF_THREADS, 0, st>>>(P.F, mc, nullptr, g->mean_c[0], mvalid, off + c0, *nchunk > 0 ? 1 : 0,
                                                                 aidx, P.amin + S);
        KL(c);
        if (samples)
            CU(cudaMemcpy2DAsync(samples + off + c0, sizeof(double) * ldo, P.F, sizeof(double) * mc, sizeof(double) * mvalid, S,
                                 kind, st));
        ++*nchunk;
    }
    return ABO_OK;
}

static int gp_pathwise_run(abo_gp* g, const double* Xc, bool dev, int64_t m, int64_t S, int64_t L, uint64_t seed, double* samples,
                           int64_t* argmin_idx, double* argmin_val) {
    if (!g || !Xc) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior (call update first)");
    if (S > PATH_MAX_S || L < 1 || L > PATH_MAX_L)
        return abo_fail(ABO_ERR_INVALID, "pathwise samples need S <= %lld draws and 1 <= L <= %lld features", (long long)PATH_MAX_S,
                        (long long)PATH_MAX_L);
    if (g->d > RFF_MAXD) return abo_fail(ABO_ERR_INVALID, "pathwise samples support d <= %d", RFF_MAXD);
    if (m <= 0 || S <= 0) return ABO_OK;
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    PathPlan P;
    int rc;
    if ((rc = pathwise_prepare(g, dev ? m : std::min(m, HOST_PIECE), S, L, seed, P))) return rc;
    int64_t nchunk = 0;
    if (dev) {
        if ((rc = pathwise_chunks(g, P, Xc, m, S, 0, samples, m, cudaMemcpyDeviceToDevice, &nchunk))) return rc;
    } else {
        double* dXc;
        if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)std::min(m, HOST_PIECE) * g->d, (void**)&dXc))) return rc;
        for (int64_t off = 0; off < m; off += HOST_PIECE) {                 // stream order: piece i + 1 overwrites dXc after piece i
            const int64_t cnt = std::min(HOST_PIECE, m - off);
            CU(cudaMemcpyAsync(dXc, Xc + off * g->d, sizeof(double) * cnt * g->d, cudaMemcpyHostToDevice, st));
            if ((rc = pathwise_chunks(g, P, dXc, cnt, S, off, samples, m, cudaMemcpyDeviceToHost, &nchunk))) return rc;
        }
    }
    if (argmin_idx) CU(cudaMemcpyAsync(argmin_idx, P.amin, sizeof(int64_t) * S, cudaMemcpyDeviceToHost, st));
    if (argmin_val) CU(cudaMemcpyAsync(argmin_val, P.amin + S, sizeof(double) * S, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return ABO_OK;
}

static int pathwise_entry(abo_gp* g, const double* Xc, bool dev, int64_t m, int64_t S, int64_t L, uint64_t seed, double* samples,
                          int64_t* argmin_idx, double* argmin_val) {
    const int rc = gp_pathwise_run(g, Xc, dev, m, S, L, seed, samples, argmin_idx, argmin_val);
    if (rc && g && g->ctx) {
        // as abo_gp_posterior_sample: nothing may still be writing workspace slots or the caller's buffers
        const std::string keep = g_err;
        ctx_sync_all(g->ctx);
        cudaGetLastError();
        g_err = keep;
    }
    return rc;
}
extern "C" int32_t abo_gp_pathwise_sample(abo_gp* g, const double* Xc, int64_t m, int64_t S, int64_t L, uint64_t seed,
                                          double* samples, int64_t* argmin_idx, double* argmin_val) {
    return pathwise_entry(g, Xc, false, m, S, L, seed, samples, argmin_idx, argmin_val);
}
extern "C" int32_t abo_gp_pathwise_sample_dev(abo_gp* g, const double* d_Xc, int64_t m, int64_t S, int64_t L, uint64_t seed,
                                              double* d_samples, int64_t* argmin_idx, double* argmin_val) {
    return pathwise_entry(g, d_Xc, true, m, S, L, seed, d_samples, argmin_idx, argmin_val);
}

// ---- stable descending top-k with Julia isless semantics (NaN largest, -0.0 < 0.0)

// Device-side selection (kernels.cuh: sel_*): enqueue the K best of dS[0..m) on `st` into workspace slot 0 / 1, and
// read the K (index, value) pairs back.  Nothing but K pairs crosses PCIe for the top-k.
struct SelSlot { SelState* st; unsigned int* ties; unsigned long long* excl; long long* idx; double* val; };
static int sel_slot(abo_ctx* c, int slot, int64_t max_m, int64_t max_k, SelSlot* out) {
    const size_t nblk = (size_t)((max_m + SEL_CHUNK - 1) / SEL_CHUNK);
    const size_t a0 = (sizeof(SelState) + 255) / 256 * 256, a1 = (nblk * 4 + 255) / 256 * 256, a2 = (nblk * 8 + 255) / 256 * 256,
                 a3 = ((size_t)max_k * 8 + 255) / 256 * 256;
    const size_t per = a0 + a1 + a2 + 2 * a3;
    char* base;
    int rc = ws_get(c, WS_SELECT, 2 * per, (void**)&base);
    if (rc) return rc;
    base += (size_t)slot * per;
    out->st = (SelState*)base; out->ties = (unsigned int*)(base + a0); out->excl = (unsigned long long*)(base + a0 + a1);
    out->idx = (long long*)(base + a0 + a1 + a2); out->val = (double*)(base + a0 + a1 + a2 + a3);
    return ABO_OK;
}
static int device_topk_launch(abo_ctx* c, const SelSlot& q, const double* dS, int64_t m, int64_t K, cudaStream_t st) {
    const int nblk = (int)((m + SEL_CHUNK - 1) / SEL_CHUNK);
    const int hgrid = (int)std::min<int64_t>((m + 255) / 256, (int64_t)c->sms * 8);
    sel_init_kernel<<<1, 256, 0, st>>>(q.st, (long long)K);
    KL(c);
    for (int pass = 0; pass < 8; ++pass) {
        sel_hist_kernel<<<hgrid, 256, 0, st>>>(dS, m, pass, q.st);
        KL(c);
        sel_pick_kernel<<<1, 256, 0, st>>>(q.st);
        KL(c);
    }
    sel_tiecount_kernel<<<nblk, 256, 0, st>>>(dS, m, q.st, q.ties);
    KL(c);
    sel_tiescan_kernel<<<1, 32, 0, st>>>(q.ties, nblk, q.excl);
    KL(c);
    sel_gather_kernel<<<nblk, 256, 0, st>>>(dS, m, q.st, q.excl, q.idx, q.val);
    KL(c);
    return ABO_OK;
}
struct TopItem { uint64_t key; int64_t idx; double val; };
constexpr int64_t SEL_MIN_M = 65536;          // below this the host picks the K best from the read-back scores
// copy the K pairs of a slot to the host (on `st`, synchronised) and append them with global indices
static int device_topk_read(const SelSlot& q, int64_t K, int64_t idx_offset, std::vector<TopItem>& items, cudaStream_t st) {
    std::vector<long long> hi((size_t)K);
    std::vector<double> hv((size_t)K);
    CU(cudaMemcpyAsync(hi.data(), q.idx, sizeof(long long) * K, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(hv.data(), q.val, sizeof(double) * K, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (int64_t i = 0; i < K; ++i) items.push_back(TopItem{ordkey(hv[(size_t)i]), (int64_t)hi[(size_t)i] + idx_offset, hv[(size_t)i]});
    return ABO_OK;
}
// sortperm(rev = true) order: key descending, index ascending
static void topk_emit(std::vector<TopItem>& items, int64_t k, int64_t* top_idx, double* top_val) {
    std::sort(items.begin(), items.end(), [](const TopItem& a, const TopItem& b) { return a.key != b.key ? a.key > b.key : a.idx < b.idx; });
    const int64_t cnt = std::min<int64_t>(k, (int64_t)items.size());
    for (int64_t i = 0; i < cnt; ++i) { top_idx[i] = items[(size_t)i].idx; top_val[i] = items[(size_t)i].val; }
}

static int scores_select_readback(abo_ctx* c, const double* dS, int64_t m, double* h_scores, int64_t k, int64_t* top_idx, double* top_val);
static int acq_eval_common(abo_gp* g, const AcqSweep& s, const double* dXc, int64_t m, double* d_scores, double* h_scores,
                           int64_t k, int64_t* top_idx, double* top_val) {
    abo_ctx* c = g->ctx;
    int rc;
    double* dS = d_scores;
    if (!dS && (rc = ws_get(c, WS_OUT_A, sizeof(double) * (size_t)m, (void**)&dS))) return rc;
    if ((rc = sweep_device(g, dXc, m, 0, s, nullptr, nullptr, dS))) return rc;
    return scores_select_readback(c, dS, m, h_scores, k, top_idx, top_val);
}
// scores on the device -> (optionally) the host, and the stable top-k of them
static int scores_select_readback(abo_ctx* c, const double* dS, int64_t m, double* h_scores, int64_t k, int64_t* top_idx, double* top_val) {
    cudaStream_t st = c->stream;
    int rc;
    const int64_t K = std::min(k, m);
    if (K > 0 && m <= SEL_MIN_M) {
        // small sets (the 10 000-point grid of optimize_acquisition): the 19 selection launches would cost more than
        // reading 8 m bytes back; pick the K best on the host
        double* hs = h_scores;
        if (!hs) { if ((rc = pinned_get(c, sizeof(double) * (size_t)m, (void**)&hs))) return rc; }
        CU(cudaMemcpyAsync(hs, dS, sizeof(double) * m, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        // heap of the K best seen so far (top = the worst kept); scanning in index order, an element enters only if its key
        // is strictly larger than the worst kept one, so equal keys keep the smaller index (sortperm is stable)
        auto better = [](const TopItem& a, const TopItem& b) { return a.key != b.key ? a.key > b.key : a.idx < b.idx; };
        std::vector<TopItem> keep;
        keep.reserve((size_t)K);
        int64_t i = 0;
        for (; i < K; ++i) keep.push_back(TopItem{ordkey(hs[i]), i, hs[i]});
        std::make_heap(keep.begin(), keep.end(), better);
        for (; i < m; ++i) {
            const uint64_t key = ordkey(hs[i]);
            if (key > keep.front().key) {
                std::pop_heap(keep.begin(), keep.end(), better);
                keep.back() = TopItem{key, i, hs[i]};
                std::push_heap(keep.begin(), keep.end(), better);
            }
        }
        std::sort(keep.begin(), keep.end(), better);
        for (int64_t q = 0; q < K; ++q) { top_idx[q] = keep[(size_t)q].idx; top_val[q] = keep[(size_t)q].val; }
        return ABO_OK;
    }
    SelSlot q{};
    if (K > 0) {
        if ((rc = sel_slot(c, 0, m, K, &q))) return rc;
        if ((rc = device_topk_launch(c, q, dS, m, K, st))) return rc;
    }
    if (h_scores) CU(cudaMemcpyAsync(h_scores, dS, sizeof(double) * m, cudaMemcpyDeviceToHost, st));
    if (K > 0) {
        std::vector<TopItem> items;
        items.reserve((size_t)K);
        if ((rc = device_topk_read(q, K, 0, items, st))) return rc;
        topk_emit(items, K, top_idx, top_val);
    } else {
        CU(cudaStreamSynchronize(st));
    }
    return ABO_OK;
}

// the arguments every acquisition entry point takes; with `s`, (acq_id, params) parsed into it
static int acq_check(abo_gp* g, const double* params, const void* Xc, int64_t m, int64_t k, int64_t* top_idx, double* top_val,
                     int acq_id = -1, AcqSweep* s = nullptr) {
    if (!g || !Xc || !params) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (!g->fitted) return abo_fail(ABO_ERR_NOT_FITTED, "surrogate has no posterior (call update first)");
    if (s) { if (const int rc = acq_parse(g, acq_id, params, 0, s)) return rc; }
    if (m < 0 || k < 0) return abo_fail(ABO_ERR_INVALID, "negative size");
    if (k > 0 && (!top_idx || !top_val)) return abo_fail(ABO_ERR_INVALID, "top-k buffers are NULL");
    return ABO_OK;
}

// Large host candidate sets go through in pieces so that the copies hide behind the sweep: while piece i
// is being evaluated the host stages piece i+1 (H2D on the copy stream), then reads back the results of
// piece i-1 (scores if asked for, and the K best of the piece, selected on the device).  Per-candidate results
// do not depend on the piece size.
// s.a.acq < 0: posterior mean / variance of output 0 (h_mean / h_var, each may be NULL).
static int sweep_host_pieces_run(abo_gp* g, const double* Xc, int64_t m, const AcqSweep& s, double* h_mean, double* h_var,
                                 double* h_scores, int64_t k, int64_t* top_idx, double* top_val);
static int sweep_host_pieces(abo_gp* g, const double* Xc, int64_t m, const AcqSweep& s, double* h_mean, double* h_var,
                             double* h_scores, int64_t k, int64_t* top_idx, double* top_val) {
    const int rc = sweep_host_pieces_run(g, Xc, m, s, h_mean, h_var, h_scores, k, top_idx, top_val);
    if (rc) {
        // an error return must not leave copies or kernels in flight that target the caller's host buffers or the
        // workspace slots (the next call may re-allocate them): drain both streams, keep the first error message
        const std::string keep = g_err;
        ctx_sync_all(g->ctx);
        cudaGetLastError();
        g_err = keep;
    }
    return rc;
}
static int sweep_host_pieces_run(abo_gp* g, const double* Xc, int64_t m, const AcqSweep& s, double* h_mean, double* h_var,
                                 double* h_scores, int64_t k, int64_t* top_idx, double* top_val) {
    abo_ctx* c = g->ctx;
    const int acq_id = s.a.acq;
    cudaStream_t st = c->stream, sc = c->stream3;
    const int d = g->d;
    const int64_t piece = HOST_PIECE;
    const int64_t np = (m + piece - 1) / piece;
    int rc;
    double *dXc, *dA, *dB = nullptr;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)m * d, (void**)&dXc))) return rc;
    if ((rc = ws_get(c, WS_OUT_A, sizeof(double) * (size_t)m, (void**)&dA))) return rc;
    if (acq_id < 0 && (rc = ws_get(c, WS_OUT_B, sizeof(double) * (size_t)m, (void**)&dB))) return rc;
    // acquisition: dA = scores; posterior: dA = mean, dB = variance
    const int64_t Kp = (acq_id >= 0 && k > 0) ? std::min(k, piece) : 0;      // per piece: its own K best, selected on the device
    SelSlot slot[2] = {};
    if (Kp > 0) { if ((rc = sel_slot(c, 0, piece, Kp, &slot[0])) || (rc = sel_slot(c, 1, piece, Kp, &slot[1]))) return rc; }
    std::vector<TopItem> items;
    if (Kp > 0) items.reserve((size_t)(Kp * np));
    auto off = [&](int64_t i) { return i * piece; };
    auto cnt = [&](int64_t i) { return std::min(piece, m - i * piece); };
    auto drain = [&](int64_t i) -> int {                 // results of piece i -> host
        double* hosts[2] = {acq_id >= 0 ? h_scores : h_mean, acq_id >= 0 ? nullptr : h_var};
        double* devs[2] = {dA, dB};
        if (!hosts[0] && !hosts[1] && Kp == 0) return ABO_OK;
        CU(cudaStreamWaitEvent(sc, c->ev_pc[i & 1], 0));
        for (int q = 0; q < 2; ++q)
            if (hosts[q]) CU(cudaMemcpyAsync(hosts[q] + off(i), devs[q] + off(i), sizeof(double) * cnt(i), cudaMemcpyDeviceToHost, sc));
        if (Kp > 0) return device_topk_read(slot[i & 1], std::min(Kp, cnt(i)), off(i), items, sc);
        CU(cudaStreamSynchronize(sc));
        return ABO_OK;
    };
    CU(cudaMemcpyAsync(dXc, Xc, sizeof(double) * cnt(0) * d, cudaMemcpyHostToDevice, sc));
    CU(cudaEventRecord(c->ev_h2d[0], sc));
    for (int64_t i = 0; i < np; ++i) {
        CU(cudaStreamWaitEvent(st, c->ev_h2d[i & 1], 0));
        if (acq_id >= 0) rc = sweep_device(g, dXc + off(i) * d, cnt(i), 0, s, nullptr, nullptr, dA + off(i));
        else rc = sweep_device(g, dXc + off(i) * d, cnt(i), 0, s, dA + off(i), dB + off(i), nullptr);
        if (rc) return rc;
        if (Kp > 0 && (rc = device_topk_launch(c, slot[i & 1], dA + off(i), cnt(i), std::min(Kp, cnt(i)), st))) return rc;
        CU(cudaEventRecord(c->ev_pc[i & 1], st));
        if (i + 1 < np) {
            CU(cudaMemcpyAsync(dXc + off(i + 1) * d, Xc + off(i + 1) * d, sizeof(double) * cnt(i + 1) * d, cudaMemcpyHostToDevice, sc));
            CU(cudaEventRecord(c->ev_h2d[(i + 1) & 1], sc));
        }
        if (i >= 1 && (rc = drain(i - 1))) return rc;
    }
    if ((rc = drain(np - 1))) return rc;
    CU(cudaStreamSynchronize(st));
    if (Kp > 0) topk_emit(items, std::min(k, m), top_idx, top_val);
    return ABO_OK;
}

extern "C" int32_t abo_acq_eval(abo_gp* g, int32_t acq_id, const double* params, const double* Xc, int64_t m,
                                double* scores, int64_t k, int64_t* top_idx, double* top_val) {
    AcqSweep s;
    int rc = acq_check(g, params, Xc, m, k, top_idx, top_val, acq_id, &s);
    if (rc) return rc;
    if (m == 0) return ABO_OK;
    abo_ctx* c = g->ctx;
    CU(cudaSetDevice(c->device));
    if (m > HOST_PIECE && !c->profile) return sweep_host_pieces(g, Xc, m, s, nullptr, nullptr, scores, k, top_idx, top_val);
    double* dXc;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)m * g->d, (void**)&dXc))) return rc;
    CU(cudaMemcpyAsync(dXc, Xc, sizeof(double) * m * g->d, cudaMemcpyHostToDevice, c->stream));
    return acq_eval_common(g, s, dXc, m, nullptr, scores, k, top_idx, top_val);
}

extern "C" int32_t abo_acq_eval_dev(abo_gp* g, int32_t acq_id, const double* params, const double* d_Xc, int64_t m,
                                    double* d_scores, int64_t k, int64_t* top_idx, double* top_val) {
    AcqSweep s;
    int rc = acq_check(g, params, d_Xc, m, k, top_idx, top_val, acq_id, &s);
    if (rc) return rc;
    if (m == 0) return ABO_OK;
    CU(cudaSetDevice(g->ctx->device));
    return acq_eval_common(g, s, d_Xc, m, d_scores, nullptr, k, top_idx, top_val);
}

extern "C" int32_t abo_fill_distance(abo_ctx* c, const double* X, int64_t n, int32_t d, const double* S, int64_t m,
                                     double* h_fill) {
    if (!c || !X || !S || !h_fill) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (n < 1 || m < 1 || d < 1 || d > 96) return abo_fail(ABO_ERR_INVALID, "bad sizes (d <= 96)");
    CU(cudaSetDevice(c->device));
    cudaStream_t st = c->stream;
    const int nblk = (int)((m + 255) / 256);
    double *dX, *dS, *dB;
    int rc;
    if ((rc = ws_get(c, WS_STAGE_X, sizeof(double) * (size_t)n * d, (void**)&dX))) return rc;
    if ((rc = ws_get(c, WS_CAND, sizeof(double) * (size_t)m * d, (void**)&dS))) return rc;
    if ((rc = ws_get(c, WS_OUT_A, sizeof(double) * (size_t)nblk, (void**)&dB))) return rc;
    CU(cudaMemcpyAsync(dX, X, sizeof(double) * n * d, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(dS, S, sizeof(double) * m * d, cudaMemcpyHostToDevice, st));
    fill_distance_kernel<<<nblk, 256, sizeof(double) * 256 * d, st>>>(dX, n, d, dS, m, dB);
    KL(c);
    std::vector<double> hb(nblk);
    CU(cudaMemcpyAsync(hb.data(), dB, sizeof(double) * nblk, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    double r = 0.0;
    for (double v : hb) r = std::max(r, v);
    *h_fill = r;
    return ABO_OK;
}

// ------------------------------------------------------------------------------------------
// standalone factorisation (Cholesky TFLOP/s metric)
// ------------------------------------------------------------------------------------------
extern "C" int32_t abo_potrf_dev(abo_ctx* c, double* d_A, int64_t n, int64_t ld, int64_t* info) {
    if (!c || !d_A) return abo_fail(ABO_ERR_INVALID, "null argument");
    if (n < 1 || n % NB != 0 || ld < n || ld % 2 != 0)
        return abo_fail(ABO_ERR_INVALID, "abo_potrf_dev needs n a multiple of 128 and an even ld >= n");
    CU(cudaSetDevice(c->device));
    const int T = (int)(n / NB);
    double* Dinv; int* dinfo;
    int rc;
    if ((rc = ws_get(c, WS_DINV, sizeof(double) * (size_t)T * NB * NB, (void**)&Dinv))) return rc;
    if ((rc = ws_get(c, WS_INFO, sizeof(int) * 16, (void**)&dinfo))) return rc;
    CU(cudaMemsetAsync(dinfo, 0, sizeof(int) * 16, c->stream));
    if ((rc = potrf_lookahead(c, d_A, n, ld, Dinv, dinfo))) return rc;
    int hinfo = 0;
    CU(cudaMemcpyAsync(&hinfo, dinfo, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    if (info) *info = hinfo;
    if (hinfo) return abo_fail(ABO_ERR_NOT_POSDEF, "matrix is not positive definite; Cholesky factorization failed at pivot %d", hinfo);
    return ABO_OK;
}

#include "abo_extra.cuh"
#include "abo_multi.cuh"

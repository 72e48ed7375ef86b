// abo_internal.h — private structures shared by the translation units of libabo_cuda.so
#pragma once
#include <cstdint>
#include <cstring>
#include <utility>
#include <unordered_set>
#include <vector>
#include <cuda_runtime.h>

int abo_fail(int code, const char* fmt, ...);

#define CU(...)                                                                                       \
    do {                                                                                              \
        cudaError_t e_ = (__VA_ARGS__);                                                                      \
        if (e_ != cudaSuccess) {                                                                      \
            cudaGetLastError();                                                                       \
            return abo_fail(4 /*ABO_ERR_CUDA*/, "%s failed: %s (%s:%d)", #__VA_ARGS__, cudaGetErrorString(e_), \
                            __FILE__, __LINE__);                                                      \
        }                                                                                             \
    } while (0)

// after every kernel launch: count it and surface launch-configuration errors
#define KL(ctx)                                                                                       \
    do {                                                                                              \
        (ctx)->launches++;                                                                            \
        cudaError_t e_ = cudaGetLastError();                                                          \
        if (e_ != cudaSuccess)                                                                        \
            return abo_fail(4, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

enum WsSlot {
    WS_STAGE_X = 0, WS_STAGE_Y, WS_DINV, WS_INFO, WS_TRTRI, WS_VEC_PART, WS_KS, WS_PMEAN, WS_SUMSQ, WS_CAND,
    WS_OUT_A, WS_OUT_B, WS_NLML_K, WS_NLML_LINV, WS_NLML_W, WS_NLML_X, WS_NLML_VEC, WS_NLML_PAR, WS_APPEND,
    WS_TOPK, WS_SELECT, WS_GRAD_W, WS_GRAD_Z, WS_GRAD_PART, WS_GRAD_OUT, WS_TRTRI_U, WS_NLML_U,
    WS_SAMPLE_G, WS_SAMPLE_SIGMA, WS_SAMPLE_Z, WS_SAMPLE_F,       // joint posterior sampler: W^T W, Sigma + tau I -> its factor, Z^T, draws
    WS_PATH_FEAT, WS_PATH_PHI, WS_PATH_COEF, WS_PATH_R, WS_PATH_Y, WS_PATH_F,  // pathwise sampler: features, Phi, [alpha - V | Theta'], R -> V, Y, draws
    WS_QEI_Z, WS_QEI_BATCH,                                        // batch expected improvement: base normals, per-batch Gram / mu / C / d mu
    WS_COUNT
};

struct WsBuf { void* ptr = nullptr; size_t bytes = 0; };

struct abo_ctx {
    int device = 0;
    int sms = 0;
    cudaStream_t stream = nullptr, stream2 = nullptr, stream3 = nullptr, stream4 = nullptr;   // 4: triangular inverse of the leading block, overlapping the factorisation's tail
    cudaEvent_t ev_inv = nullptr;
    cudaEvent_t ev_p[3] = {nullptr, nullptr, nullptr};            // panel-chain split of the Cholesky
    cudaEvent_t ev_a = nullptr, ev_b = nullptr;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_pc[2] = {nullptr, nullptr};  // candidate pieces: staged / evaluated
    WsBuf ws[WS_COUNT];
    void* pinned = nullptr;
    size_t pinned_bytes = 0;
    int64_t launches = 0;
    // optional per-kernel timing of the sweep (abo_ctx_profile)
    bool profile = false;
    std::vector<cudaEvent_t> prof_events;     // pairs, class = (index / 2) % 3
    size_t prof_used = 0;
    double prof_ms[3] = {0, 0, 0};
    int64_t prof_n[3] = {0, 0, 0};
    // NCCL (one rank per context)
    void* nccl_comm = nullptr;
    int rank = 0, nranks = 1;
    // handles created on this context: abo_ctx_destroy orphans the ones still alive (bindings whose finalizers
    // run in arbitrary order — Python at interpreter exit, Julia's GC — may destroy the context first)
    std::unordered_set<abo_gp*> live;
    // released posterior buffer sets kept for re-use (a BO loop allocates and frees one per iteration)
    struct GpBufSet { int64_t cap_pad, ldx; int d, p; double* ptr[7]; };
    std::vector<GpBufSet> gp_pool;
};

struct abo_gp {
    abo_ctx* ctx = nullptr;
    int kind = 0, d = 1, p = 1;
    double s = 1.0, scale = 1.0, noise = 0.0;
    std::vector<double> sv;               // per-dimension inverse length scales (ARD); all equal to s when isotropic
    bool ard = false;
    std::vector<double> mean_c;
    int64_t n = 0, N = 0, Npad = 0;      // points, system size n*p, padded to 128
    int64_t cap_pad = 0, ld = 0, ldx = 0;
    bool fitted = false;
    double *dXsT = nullptr, *dL = nullptr, *dLinv = nullptr, *dAlpha = nullptr, *dBeta = nullptr,
           *dDelta = nullptr, *dMeanC = nullptr;
    int* share = nullptr;                 // reference count of the device buffers (clones share them until one writes)
};

// Julia `isless` order on Float64 as an unsigned key: NaN largest, -0.0 < 0.0
static inline uint64_t ordkey(double v) {
    if (v != v) return ~0ull;
    uint64_t u;
    memcpy(&u, &v, 8);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}

int gp_alloc(abo_gp* g, int64_t Npad, int64_t ldx);
int gp_unshare(abo_gp* g);
void gp_pool_clear(abo_ctx* c);
static inline bool gp_shared(const abo_gp* g) { return g->share && *g->share > 1; }
void ctx_sync_all(abo_ctx* c);
void ws_release(abo_ctx* c, int slot);
int ws_get(abo_ctx* c, int slot, size_t bytes, void** out);
int pinned_get(abo_ctx* c, size_t bytes, void** out);
int potrf_lookahead(abo_ctx* c, double* A, int64_t Npad, int64_t ld, double* Dinv, int* info, int notify_tile = 0, cudaStream_t notify_stream = nullptr);
int potrf_blocked(abo_ctx* c, double* A, int64_t Npad, int64_t ld, double* Dinv, int* info, int batch);
int trtri_tma(abo_ctx* c, const double* L, double* Linv, double* U, double* Wt, int64_t Npad, int64_t ld, int64_t strideM,
              const double* Dinv, int64_t strideD, int batch);
int solve_alpha(abo_ctx* c, const double* Linv, int64_t ld, int64_t N, const double* delta, double* beta,
                double* alpha, int64_t strideM, int64_t strideV, int batch);
void abo_nccl_teardown(abo_ctx* c);
int prof_mark(abo_ctx* c);
int prof_collect(abo_ctx* c);

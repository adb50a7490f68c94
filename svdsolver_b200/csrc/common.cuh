// Shared declarations of the svdb200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>
#include "../../include/svdb200.h"

namespace svdb200 {

constexpr int kMaxBand = 128;          // stage-1 panel width / stage-2 band supported by the kernels
constexpr int kMaxPanelCtas = 148;     // one CTA per SM in the cooperative panel kernel
constexpr int kLookaheadReserve = 20;  // SMs the persistent tcgen05 rank update leaves free while a look-ahead panel runs beside it

// Run-time choices set through the C ABI setters.  Sub-handles (batch pool, stage-1 chains of the list pipeline) copy
// them from their parent before every use.
struct Settings {
    int stage2_complete = 0;                // 0: the reference's window schedule (parity), 1: complete chase
    // singular values of the bidiagonal: 0 auto (zero-shift QR up to qr_auto_limit, bisection above), 1 QR, 2 bisection
    int qr_method = 0;
    size_t qr_auto_limit = 1024;
    int use_tc05 = 1;                       // 0 off, 1 when the update is large enough, 2 always (tests)
    long long tc05_min_elems = 8LL << 20;   // smallest M*N the tcgen05 kernels are used for in mode 1
    int panel_blk = 1;                      // blocked panel kernel (one exchange per 8 columns, stage1_panel_blk.cu) where the shape allows
    int panel_chol = 1;                     // Cholesky-QR panel with reconstructed Householder vectors (stage1_panel_chol.cu)
    double chol_guard = 1e-3;               // smallest accepted pivot ratio R_jj^2 / G_jj; below, the exchange-based kernels redo the panel
};

// Device buffer allocated after svdb200_create, on first use or grown by reserve(); freed with its owner.
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
};

struct Ctx {
    int device = 0;
    int dtype = SVDB200_F64;
    size_t max_n = 0, band = 0, esz = 8;
    int num_sms = 148;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    // device workspace (element type = dtype)
    DevBuf a_dev;                  // max_n * max_n : staging for host-pointer calls (first use)
    void* v = nullptr;             // max_n * band  : V (QR) / U^T (LQ), row-major, unit diagonal explicit
    void* v2 = nullptr;            // max_n * band  : V S^T (QR) ; band * max_n : S U (LQ)
    void* vb = nullptr; void* v2b = nullptr;   // second reflector pair (LQ panels) for the look-ahead
    cudaStream_t aux_stream = nullptr;         // high-priority stream the look-ahead panels run on
    cudaEvent_t lev[4] = {};
    void* w = nullptr;             // band * max_n  : W = V^T A  /  max_n * band : W = A U^T
    void* wpart = nullptr;         // split-K partials
    size_t wpart_elems = 0;
    void* s = nullptr;             // band * band   : S (= -T of compact WY), upper triangular
    void* tau = nullptr;           // band
    unsigned panel_epoch = 0;      // sequence base of the flag-stamped panel all-reduce words (one per launch)
    void* red = nullptr;           // panel all-reduce scratch: 2 * kMaxPanelCtas * (2*band + 8)
    void* red2 = nullptr;          // blocked panel kernel: flag-stamped words exchanged between clusters through L2 (512 KB)
    unsigned int* bar = nullptr;   // software grid barrier state (2 words) + misc counters
    int* prog = nullptr;           // stage-2 per-sweep progress counters (max_n)
    DevBuf band_ws;                // max_n * 3 band: stage 2 from band storage, packed 3-band-diagonal layout (first use)
    DevBuf rect_ws;                // m * n: A^T of a wide m x n matrix (m < n), reduced there; grown on demand
    void* d = nullptr; void* e = nullptr; void* sigma = nullptr;   // max_n each
    long long* qr_info = nullptr;  // [0] sweeps, [1] status
    void* tileq = nullptr;         // tile order: per-chain-step Q matrices, (max_n/band) * 4*band*band
    void* tilestate = nullptr;     // tile order: S_kk,V_kk,... persistent small state
    // host-side bookkeeping
    long long launches = 0;
    cudaEvent_t ev[8] = {};
    double ms_stage1 = 0, ms_stage2 = 0, ms_qr = 0, ms_h2d = 0, ms_d2h = 0;
    std::string last_error;
    int coop_supported = 0;
    int cluster_ok = 16;           // largest thread-block-cluster size the panel kernel may use (0: none)
    // per-kernel-class profiling (svdb200_set_profile)
    int profile = 0;
    double prof_ms[SVDB200_PROFILE_CLASSES] = {};
    double prof_work[SVDB200_PROFILE_CLASSES] = {};
    long long prof_launches[SVDB200_PROFILE_CLASSES] = {};
    cudaEvent_t pev[2] = {};
    // pool of sub-handles for the batched driver (created on first use for a given n, band)
    std::vector<Ctx*> pool;
    size_t pool_n = 0, pool_band = 0;
    // tcgen05 FP32 path (gemm_tc05.cu): hi/lo split scratch for the O(n b) operands, allocated on first use
    DevBuf tcsplit;
    Settings cfg;
    // pipelined multi-matrix driver (bidiagonalize_many): stage 2 of matrix i on s2_stream beside stage 1 of matrix i+1
    static constexpr int kLanes = 2;        // chains in flight: each = one stage 1 (own sub-handle) and one stage-2 kernel
                                            // (more chains measured slower: they disturb each other's stage-2 sweep pipelines)
    cudaStream_t s2_stream[kLanes] = {};
    int* s2_prog[kLanes] = {};              // progress counters per lane
    cudaEvent_t s2ev[4 + kLanes] = {};
    int onestage = 0;                       // stage-1 driver in the one-stage Golub-Kahan order (band 1, no skipped row reflector)
    int s2_ready = 0;                       // the pipeline's streams / counters / sub-handles below exist (all or nothing)
    void* chol_ws = nullptr;                // Cholesky-QR panel workspace: status word, [M1 | M2], partial Gram matrices (1 MB)
    const int* panel_run_if = nullptr;      // set while a gated fallback panel launch is being enqueued
    int reserve_now = 0;                    // set by the stage-1 drivers around the part of an update that overlaps a panel
    int overlap_safe = 0;                   // stage 1 may only use kernels without cross-cluster / grid-wide waits
    Ctx* s1ctx[kLanes] = {};                // sub-handles (own workspace + streams): stage 1 of two matrices at a time
    void* a_stage[2 * kLanes] = {};         // staging buffers + bidiagonal rows for the host-pointer variant
    void* de2 = nullptr;
    DevBuf bis_ws;                             // bisection workspace: params + 2 * max_n squared off-diagonals (double)
    std::vector<void*> band_capture;           // test hook of bidiagonalize_many_*: device buffers that receive matrix i's band
    // batched small-matrix driver: per-matrix progress counters, reflector / W workspaces, d / e rows
    DevBuf batch_prog;
    DevBuf batch_ws;
};

// Brackets one kernel launch with events when profiling is on (serialises host and device; the
// kernel's own duration is unaffected).
struct ProfScope {
    Ctx* c; int cls; double work;
    ProfScope(Ctx* c_, int cls_, double work_) : c(c_), cls(cls_), work(work_) {
        if (c->profile) cudaEventRecord(c->pev[0], c->stream);
    }
    ~ProfScope() {
        if (!c->profile) return;
        cudaEventRecord(c->pev[1], c->stream);
        cudaEventSynchronize(c->pev[1]);
        float ms = 0;
        cudaEventElapsedTime(&ms, c->pev[0], c->pev[1]);
        c->prof_ms[cls] += ms; c->prof_work[cls] += work; c->prof_launches[cls] += 1;
    }
};

inline int cuda_status(Ctx* c, cudaError_t e, const char* what) {
    if (e == cudaSuccess) return 0;
    if (c) {
        c->last_error = std::string(what) + ": " + cudaGetErrorString(e);
    }
    return SVDB200_CUDA_ERR + (int)e;
}

#define SVDB_CHECK(ctx, expr)                                            \
    do {                                                                 \
        cudaError_t _e = (expr);                                         \
        if (_e != cudaSuccess) return ::svdb200::cuda_status((ctx), _e, #expr); \
    } while (0)
#define SVDB_TRY(expr)                 \
    do {                               \
        int _s = (expr);               \
        if (_s != 0) return _s;        \
    } while (0)

// At least `bytes` in b: returns at once when b is big enough; otherwise b is replaced by an allocation of exactly `bytes`
// (after the handle's stream has finished, since work enqueued earlier may still use the old buffer).
inline int reserve(Ctx* c, DevBuf& b, size_t bytes) {
    if (b.bytes >= bytes) return 0;
    if (b.p) {
        SVDB_CHECK(c, cudaStreamSynchronize(c->stream));
        SVDB_CHECK(c, cudaFree(b.p));
        b.p = nullptr;
        b.bytes = 0;
    }
    SVDB_CHECK(c, cudaMalloc(&b.p, bytes));
    b.bytes = bytes;
    return 0;
}

// ---- exactly-rounded, never-contracted arithmetic for the bit-faithful kernels -------------------
// (the reference is compiled without FMA contraction: ISO C++ mode => -ffp-contract=off; SURVEY 0.7)
template <typename T> struct RN;
template <> struct RN<float> {
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
    static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
    static __device__ __forceinline__ float sqrt(float a) { return __fsqrt_rn(a); }
    static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
    static __device__ __forceinline__ float abs(float a) { return fabsf(a); }
};
template <> struct RN<double> {
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
    static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
    static __device__ __forceinline__ double sqrt(double a) { return __dsqrt_rn(a); }
    static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
    static __device__ __forceinline__ double abs(double a) { return fabs(a); }
};

// Householder scalars exactly as svd_serial.h:194-201: s, u1, 1/u1, tau in double, rounded to T.
template <typename T>
__device__ __forceinline__ void householder_scalars(T x0, T norm_x, T& alpha, T& tau) {
    double s = -copysign(1.0, (double)x0);
    double u1 = __dsub_rn((double)x0, __dmul_rn(s, (double)norm_x));
    alpha = (T)__ddiv_rn(1.0, u1);
    tau = (T)__ddiv_rn(__dmul_rn(-s, u1), (double)norm_x);
}

// L2-coherent accesses for data exchanged between CTAs inside one launch (bypass the non-coherent L1)
template <typename T> __device__ __forceinline__ T ld_cg(const T* p) { return __ldcg(p); }
template <typename T> __device__ __forceinline__ void st_cg(T* p, T v) { __stcg(p, v); }
__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_u(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Software grid barrier for cooperative launches (all CTAs co-resident). bar[0] = arrival counter,
// bar[1] = generation. Monotone generation => no reset race.
__device__ __forceinline__ void grid_barrier(unsigned* bar, unsigned nctas, unsigned& gen) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        unsigned target = gen + 1;
        unsigned prev = atomicAdd(&bar[0], 1u);
        if (prev == nctas * target - 1) {
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(&bar[1]), "r"(target) : "memory");
        } else {
            while (ld_acquire_u(&bar[1]) < target) { __nanosleep(20); }
        }
        __threadfence();
    }
    gen += 1;
    __syncthreads();
}

// ---- internal entry points (one per .cu) ----------------------------------------------------------
template <typename T> int stage2_chase(Ctx* c, T* a, size_t n, size_t band, T* d, T* e);
template <typename T> int extract_bidiagonal(Ctx* c, const T* a, size_t n, T* d, T* e);
template <typename T> int stage2_chase_packed(Ctx* c, const T* ab, size_t n, size_t band, T* d, T* e);   // ab: LAPACK upper band storage
template <typename T, bool kPacked> int stage2_chase_fast(Ctx* c, T* a, size_t n, size_t band, int* prog);   // 0 ran, 1 shape not covered
template <typename T> int bidiag_qr(Ctx* c, T* d, T* e, size_t n, T* sigma);
template <typename T> int bidiag_bisect(Ctx* c, const T* d, const T* e, size_t n, T* sigma);
template <typename T> int bidiag_sqr(Ctx* c, T* d, T* e, size_t n, T* sigma);
template <typename T> int stage1_panel_order(Ctx* c, T* a, size_t rows, size_t n, size_t band);   // a: rows x n, rows >= n
template <typename T> int transpose(Ctx* c, const T* src, size_t rows, size_t cols, T* dst);        // rect.cu
template <typename T> int transpose_batched(Ctx* c, const T* src, size_t sS, size_t rows, size_t cols, T* dst, size_t sD, size_t count);
template <typename T> int stage1_tile_order(Ctx* c, T* a, size_t n, size_t band);
template <typename T> int gemm_tn(Ctx* c, const T* v, const T* cm, size_t ldc, size_t mrows, size_t ncols, size_t b, T* w);
template <typename T> int gemm_nn(Ctx* c, const T* cm, size_t ldc, size_t mrows, size_t ncols, size_t b, const T* ut, T* w);
template <typename T> int rank_update(Ctx* c, T* cm, size_t ldc, size_t mrows, size_t ncols, size_t b, const T* p, const T* q, size_t ldq);
// batched (uniform-shape) building blocks: element strides sX between consecutive matrices
template <typename T> int rank_update_batched(Ctx* c, T* cm, size_t ldc, size_t sC, int M, int N, int K, const T* p, size_t sP, const T* q, size_t ldq, size_t sQ, int count);
template <typename T> int gemm_tn_batched(Ctx* c, const T* v, size_t sV, const T* cm, size_t ldc, size_t sC, int M, int N, int B, T* w, size_t sW, int count);
template <typename T> int gemm_nn_batched(Ctx* c, const T* cm, size_t ldc, size_t sC, int M, int N, int B, const T* ut, size_t sU, T* w, size_t sW, int count);
template <typename T, bool kTrans> int panel_batched(Ctx* c, T* a, size_t lda, size_t sA, int m, int b, T* V, T* V2, size_t sV, int count);
bool panel_batched_fits(int m, int b, size_t esz);   // panel_batched takes panels of height (or length) m at width b
template <typename T> int stage2_chase_batched(Ctx* c, T* a, size_t sA, size_t n, size_t band, T* d, T* e, int count);
template <typename T> int bidiag_bisect_batched(Ctx* c, const T* d, const T* e, size_t n, T* sigma, int count);
template <typename T> int fill_uniform(Ctx* c, T* a, size_t count, unsigned long long seed, double lo, double hi);
template <typename T> int mse_metric(Ctx* c, const T* a, const T* b, size_t n, size_t band, T* out_host);
template <typename T> int batched_svdvals(Ctx* c, T* a, size_t count, size_t n, size_t band, T* sigma);
template <typename T> int batched_chain(Ctx* c, T* a, size_t count, size_t m, size_t n, size_t band, int what, T* d, T* e, T* sigma);
int probe_peak(Ctx* c, int kind, double* tflops);
int probe_tc05_tf32(Ctx* c, double* tflops);
int panel_reg_debug_read(long long* out16);
int panel_blk_debug_read(long long* out16);
int panel_chol_debug_read(long long* out16);
int stage2_debug_read(long long* out16);
int stage2_fast_debug_read(long long* out24);
int tc05_selftest(Ctx* c, int a_mn, int b_mn, const float* a, const float* b, float* out, float* dump);

}  // namespace svdb200

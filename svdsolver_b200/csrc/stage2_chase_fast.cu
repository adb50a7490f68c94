// Stage 2 (band -> bidiagonal), band 32: the latency-optimised variant of stage2_chase_kernel (stage2_chase.cu; replaces
// csc586::parallel::brd_p2<T>, svd_parallel.h:640-695).  Same window schedule, same bit-faithful arithmetic (explicit H,
// k-ascending unfused sums, reflector scalars in double), same per-sweep progress counters and lag-4 rule -- what changes
// is what sits on the critical path of a window op.  Measured for the previous kernel (f64, cycles per op): window product
// 3.3 K, reflector scalars on one thread 1.2 K, build H + store the new block + barriers 1.1 K, load issue 0.7 K.  Here:
//   * a ninth HELPER warp prepares the NEXT op's reflector while the main warps still multiply: the next op's
//     Householder vector is one column (RIGHT -> LEFT) / one row (LEFT -> RIGHT) of the block this op forwards, so the
//     helper recomputes those 32 dot products (same products, same order => same bits), runs the sequential sum of
//     squares, the double-precision scalars and writes the explicit H into the other H buffer.  The next op starts with
//     its H ready: scalars and H leave the critical path;
//   * the window product is split by operand: warps 0-3 multiply the block that is already in shared memory (forwarded
//     by the previous op) while warps 4-7 fetch the new block from L2, store it and multiply it -- the L2 latency of the
//     fetch hides behind the first half instead of behind the scalars.
// Only interior windows (full c x c blocks) take this path; the top pair of a sweep and the clamped windows at the matrix
// edge run the generic code of the original kernel (inside this kernel, on the same shared-memory layout).
#include <algorithm>
#include <climits>
#include "common.cuh"
#include "stage2_common.cuh"

namespace svdb200 {

namespace {
using namespace s2;

#ifndef SVDB_S2_TIMING
#define SVDB_S2_TIMING 0
#endif
// per-phase cycle counters of interior RIGHT ops of CTA 1 (debug builds: -DSVDB_S2_TIMING=1); every slot has one writer
__device__ long long g_s2f_dbg[16];
#define S2F_T() (SVDB_S2_TIMING ? clock64() : 0ll)
#define S2F_ADD(k, v)                                                   \
    do {                                                                \
        if (SVDB_S2_TIMING && blockIdx.x == 1) g_s2f_dbg[k] += (v);     \
    } while (0)

constexpr int kC = 32;                 // band
constexpr int kMain = 256;             // main threads: warps 0-3 = F half, warps 4-7 = N half
constexpr int kFastThreads = kMain + 32;

__device__ __forceinline__ void bar_n_helper() { asm volatile("bar.sync 1, 160;" ::: "memory"); }   // N warps + helper warp

// Helper warp: reflector of the next op from its Householder vector xv (lane l holds x_l), exactly as
// reflector_scalars + build_h do it (sequential unfused sum of squares in index order; scalars in double; H = I - tau w w^T
// with w_0 = 1, w_i = x_i * alpha).  The shared-memory pipe is busy with the operands of the window product, so every
// value another lane holds is fetched in ONE batch of vector loads (x goes through a 32-element staging row) instead of one
// shuffle per step: the dependent chains then run on registers only.
template <typename T>
__device__ __forceinline__ void helper_reflector(T xv, T* __restrict__ xst, T* __restrict__ Hn, int ldh, bool guard) {
    const int lane = threadIdx.x & 31;
    xst[lane] = xv;
    __syncwarp();
    T x[kC];
    if constexpr (sizeof(T) == 4) {
#pragma unroll
        for (int r = 0; r < kC; r += 4) {
            const float4 v = *reinterpret_cast<const float4*>(xst + r);
            x[r] = v.x; x[r + 1] = v.y; x[r + 2] = v.z; x[r + 3] = v.w;
        }
    } else {
#pragma unroll
        for (int r = 0; r < kC; r += 2) {
            const double2 v = *reinterpret_cast<const double2*>(xst + r);
            x[r] = v.x; x[r + 1] = v.y;
        }
    }
    T acc = (T)0;
#pragma unroll
    for (int r = 0; r < kC; ++r) acc = RN<T>::add(acc, RN<T>::mul(x[r], x[r]));
    T alpha, tau;
    if (guard && acc == (T)0) { alpha = (T)0; tau = (T)0; }
    else householder_scalars<T>(x[0], RN<T>::sqrt(acc), alpha, tau);
    const T mtau = -tau;
    const T wl = (lane == 0) ? (T)1 : RN<T>::mul(xv, alpha);
#pragma unroll
    for (int i = 0; i < kC; ++i) {
        const T wi = (i == 0) ? (T)1 : RN<T>::mul(x[i], alpha);
        T h = RN<T>::mul(RN<T>::add((T)0, RN<T>::mul(wi, wl)), mtau);
        if (i == lane) h = RN<T>::add((T)1, h);
        Hn[i * ldh + lane] = h;
    }
    __syncwarp();
}

template <typename T>
__global__ void __launch_bounds__(kFastThreads, 1) stage2_fast_kernel(T* __restrict__ A, int n, int* __restrict__ prog, int complete) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int c = kC, w = c + 1;
    constexpr int ldr = c + 1, ldl = 2 * c + 1, ldh = c + 1;
    T* WR = reinterpret_cast<T*>(smem_raw);     // RIGHT window [2c][c+1]: rows [0,c) forwarded block F, rows [c,2c) new block N
    T* WL = WR + 2 * c * ldr;                   // LEFT  window [c][2c+1]: cols [0,c) F, cols [c,2c) N
    T* Hb0 = WL + c * ldl;                      // two H buffers [c][c+1]: the current op's and the next op's
    T* Hb1 = Hb0 + c * ldh;
    T* sc = Hb1 + c * ldh;                      // alpha, tau (generic path)
    T* xst = sc + 8;                            // helper: staging row for the next Householder vector (16-byte aligned)
    const int tid = threadIdx.x;
    const bool is_main = tid < kMain, is_helper = !is_main;
    const bool f_warp = tid < kMain / 2, n_warp = is_main && !f_warp;
    const size_t N = (size_t)n;
    const int tx = tid % c, ty = tid / c;       // generic path: c columns x tys rows of main threads
    constexpr int tys = kMain / c;
    const int ht = tid - kMain / 2;             // N warps: 0..127
    const int G = gridDim.x;
    const int rel_tid = 32;
    T* Hc = Hb0;
    T* Hn = Hb1;
    for (int i = blockIdx.x; i < n - 1; i += G) {
        int seen = 0;
        const int top_j2 = min(i + 2 * w - 1, n);
        const int npairs = complete ? (n - i - 1 + c - 1) / c : 1 + (n - top_j2) / c + 1;
        int fr = 0;
        bool hready = false;                    // Hc already holds the H of the op about to run (written by the helper)
        for (int p = 0; p < npairs; ++p) {
            const int r0 = (p == 0) ? i : min(i + 1 + (p - 1) * c, n);
            const int r1 = min(i + 1 + p * c, n), r2 = min(i + 1 + (p + 1) * c, n), c3 = min(i + 1 + (p + 2) * c, n);
            if (r2 <= r1) break;
            // ================= RIGHT(p): rows [r0,r2) x cols [r1,r2), window = [F; N] ===================
            {
                const int q = 2 * p;
                const long long t_op0 = S2F_T();
                if (i > 0 && tid == 0) seen = wait_progress(&prog[i - 1], q + 4, seen);
                const long long t_polled = S2F_T();
                __syncthreads();
                const long long t_start = S2F_T();
                const int nc = r2 - r1, nr = r2 - r0, have = fr;
                const bool interior = (have == c) && (nr == 2 * c) && (nc == c);
                if (interior) {
                    if (tid == 0) { S2F_ADD(0, t_polled - t_op0); S2F_ADD(9, t_start - t_polled); S2F_ADD(7, 1); if (!hready) S2F_ADD(10, 1); }
                    T nv[8];
                    if (n_warp) {                 // new block: rows [c,2c) of the window, 8 elements per thread
#pragma unroll
                        for (int u = 0; u < 8; ++u) nv[u] = ld_cg(&A[(size_t)(r1 + (ht >> 5) + 4 * u) * N + (r1 + (ht & 31))]);
                    }
                    if (!hready) {                // first interior op of a sweep: H the classic way
                        if (tid == 0) reflector_scalars<T>(WR, 1, c, sc, complete != 0);
                        __syncthreads();
                        if (is_main) build_h<T>(WR, 1, c, sc, Hc, ldh, tx, ty, tys);
                        __syncthreads();
                    }
                    const long long t_h = S2F_T();
                    long long t_done = 0;
                    if (f_warp) {                 // F half: finished rows [r0,r1) -> global
                        window_product<T, kC>(WR, ldr, Hc, ldh, c, c, c, 16, 8,
                                              [&](int r, int cc, T v) { st_cg(&A[(size_t)(r0 + r) * N + (r1 + cc)], v); }, tid);
                        t_done = S2F_T();
                        if (tid == 0) { S2F_ADD(11, t_h - t_start); S2F_ADD(1, t_done - t_h); }
                    } else if (n_warp) {
#pragma unroll
                        for (int u = 0; u < 8; ++u) WR[(c + (ht >> 5) + 4 * u) * ldr + (ht & 31)] = nv[u];
                        const long long t_ld = S2F_T();
                        bar_n_helper();
                        const long long t_b = S2F_T();
                        window_product<T, kC>(WR + c * ldr, ldr, Hc, ldh, c, c, c, 16, 8,
                                              [&](int r, int cc, T v) { WL[r * ldl + cc] = v; }, ht);
                        t_done = S2F_T();
                        if (tid == kMain / 2) { S2F_ADD(3, t_ld - t_start); S2F_ADD(12, t_b - t_ld); S2F_ADD(4, t_done - t_b); }
                    } else {                      // helper: x' = column 0 of N * H  (LEFT(p)'s Householder vector)
                        bar_n_helper();
                        const long long t_b = S2F_T();
                        const int lane = tid & 31;
                        T xo[kC], yo[kC];
#pragma unroll
                        for (int k = 0; k < c; ++k) { xo[k] = WR[(c + lane) * ldr + k]; yo[k] = Hc[k * ldh]; }
                        T acc = (T)0;
#pragma unroll
                        for (int k = 0; k < c; ++k) acc = RN<T>::add(acc, RN<T>::mul(xo[k], yo[k]));
                        const long long t_x = S2F_T();
                        helper_reflector<T>(acc, xst, Hn, ldh, complete != 0);
                        t_done = S2F_T();
                        if (tid == kMain) { S2F_ADD(6, t_b - t_start); S2F_ADD(13, t_x - t_b); S2F_ADD(5, t_done - t_x); }
                    }
                    __syncthreads();
                    if (tid == 0) { S2F_ADD(2, S2F_T() - t_done); S2F_ADD(8, S2F_T() - t_op0); }
                    { T* t = Hc; Hc = Hn; Hn = t; }
                    hready = true;
                } else {
                    // -------- generic path (top pair, clamped windows): the original kernel's code on the main threads
                    T nv[kNewPerThread];
                    const int newcnt = (nr - have) * nc;
                    if (have == 0) {
                        if (is_main)
                            for (int e = tid; e < newcnt; e += kMain)
                                WR[(e / nc) * ldr + e % nc] = ld_cg(&A[(size_t)(r0 + e / nc) * N + (r1 + e % nc)]);
                        __syncthreads();
                    } else if (is_main) {
#pragma unroll
                        for (int u = 0; u < kNewPerThread; ++u) {
                            int r = ty + u * tys;
                            if (r < nr - have && tx < nc) nv[u] = ld_cg(&A[(size_t)(r0 + have + r) * N + (r1 + tx)]);
                        }
                    }
                    if (!hready && tid == 0) reflector_scalars<T>(WR, 1, nc, sc, complete != 0);
                    __syncthreads();
                    if (is_main) {
                        if (!hready) build_h<T>(WR, 1, nc, sc, Hc, ldh, tx, ty, tys);
                        if (have != 0) {
#pragma unroll
                            for (int u = 0; u < kNewPerThread; ++u) {
                                int r = ty + u * tys;
                                if (r < nr - have && tx < nc) WR[(have + r) * ldr + tx] = nv[u];
                            }
                        }
                    }
                    __syncthreads();
                    const int keep = r1 - r0;
                    if (is_main)
                        window_product<T, kC>(WR, ldr, Hc, ldh, nr, nc, nc, (c + 1) / 2, (c + 1) / 2,
                                              [&](int r, int cc, T v) {
                                                  if (r < keep) st_cg(&A[(size_t)(r0 + r) * N + (r1 + cc)], v);
                                                  else WL[(r - keep) * ldl + cc] = v;
                                              }, tid);
                    __syncthreads();
                    hready = false;
                }
                if (tid == rel_tid) st_release(&prog[i], q + 1);
            }
            // ================= LEFT(p): rows [r1,r2) x cols [r1,c3), window = [F | N] ====================
            const int nn = c3 - r2;
            const bool fwd = (p + 1 < npairs) && nn > 0;
            {
                const int q = 2 * p + 1;
                if (i > 0 && tid == 0) seen = wait_progress(&prog[i - 1], q + 4, seen);
                __syncthreads();
                const int nr = r2 - r1, fc = r2 - r1, nc = fc + nn;
                const bool interior = (nr == c) && (nn == c) && fwd;
                if (interior) {
                    T nv[8];
                    if (n_warp) {                 // new block: cols [c,2c) of the window
#pragma unroll
                        for (int u = 0; u < 8; ++u) nv[u] = ld_cg(&A[(size_t)(r1 + (ht >> 5) + 4 * u) * N + (r2 + (ht & 31))]);
                    }
                    if (!hready) {
                        if (tid == 0) reflector_scalars<T>(WL, ldl, c, sc, complete != 0);
                        __syncthreads();
                        if (is_main) build_h<T>(WL, ldl, c, sc, Hc, ldh, tx, ty, tys);
                        __syncthreads();
                    }
                    if (f_warp) {                 // F half: finished cols [r1,r2) -> global
                        window_product<T, kC>(Hc, ldh, WL, ldl, c, c, c, 16, 8,
                                              [&](int r, int cc, T v) { st_cg(&A[(size_t)(r1 + r) * N + (r1 + cc)], v); }, tid);
                    } else if (n_warp) {
#pragma unroll
                        for (int u = 0; u < 8; ++u) WL[((ht >> 5) + 4 * u) * ldl + c + (ht & 31)] = nv[u];
                        bar_n_helper();
                        window_product<T, kC>(Hc, ldh, WL + c, ldl, c, c, c, 16, 8,
                                              [&](int r, int cc, T v) { WR[r * ldr + cc] = v; }, ht);
                    } else {                      // helper: x'' = row 0 of H * N  (RIGHT(p+1)'s Householder vector)
                        bar_n_helper();
                        const int lane = tid & 31;
                        T xo[kC], yo[kC];
#pragma unroll
                        for (int k = 0; k < c; ++k) { xo[k] = Hc[k]; yo[k] = WL[k * ldl + c + lane]; }
                        T acc = (T)0;
#pragma unroll
                        for (int k = 0; k < c; ++k) acc = RN<T>::add(acc, RN<T>::mul(xo[k], yo[k]));
                        helper_reflector<T>(acc, xst, Hn, ldh, complete != 0);
                    }
                    fr = c;
                    __syncthreads();
                    { T* t = Hc; Hc = Hn; Hn = t; }
                    hready = true;
                } else {
                    T nv[kNewPerThread];
                    if (is_main) {
#pragma unroll
                        for (int u = 0; u < kNewPerThread; ++u) {
                            int r = ty + u * tys;
                            if (r < nr && tx < nn) nv[u] = ld_cg(&A[(size_t)(r1 + r) * N + (r2 + tx)]);
                        }
                    }
                    if (!hready && tid == 0) reflector_scalars<T>(WL, ldl, nr, sc, complete != 0);
                    __syncthreads();
                    if (is_main) {
                        if (!hready) build_h<T>(WL, ldl, nr, sc, Hc, ldh, tx, ty, tys);
#pragma unroll
                        for (int u = 0; u < kNewPerThread; ++u) {
                            int r = ty + u * tys;
                            if (r < nr && tx < nn) WL[r * ldl + fc + tx] = nv[u];
                        }
                    }
                    __syncthreads();
                    if (is_main)
                        window_product<T, kC>(Hc, ldh, WL, ldl, nr, nc, nr, c, (c + 3) / 4,
                                              [&](int r, int cc, T v) {
                                                  if (cc < fc || !fwd) st_cg(&A[(size_t)(r1 + r) * N + (r1 + cc)], v);
                                                  else WR[r * ldr + (cc - fc)] = v;
                                              }, tid);
                    fr = fwd ? nr : 0;
                    __syncthreads();
                    hready = false;
                }
                if (tid == rel_tid && fwd) st_release(&prog[i], q + 1);
            }
            if (!fwd) break;
        }
        if (tid == rel_tid) st_release(&prog[i], INT_MAX);
    }
}

}  // namespace

int stage2_fast_debug_read(long long* out16) {
    long long z[16] = {};
    if (cudaMemcpyFromSymbol(out16, g_s2f_dbg, sizeof(z)) != cudaSuccess) return 1;
    cudaMemcpyToSymbol(g_s2f_dbg, z, sizeof(z));
    return 0;
}

// returns 0 when it ran, 1 when the shape is outside this kernel's range (the caller runs stage2_chase_kernel)
template <typename T>
int stage2_chase_fast(Ctx* c, T* a, size_t n, size_t band, int* prog) {
    if (band != (size_t)kC || n < 2 * band + 2) return 1;
    const size_t smem = (size_t)(2 * kC * (kC + 1) + kC * (2 * kC + 1) + 2 * kC * (kC + 1) + 8 + kC + 8) * sizeof(T);
    auto kern = stage2_fast_kernel<T>;
    SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    SVDB_CHECK(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kFastThreads, smem));
    if (per_sm < 1) return 1;
    long long inflight = (long long)(n / band) / 2 + 2;
    long long G = std::min(inflight, std::min((long long)per_sm * c->num_sms, (long long)n - 1));
    if (G < 1) G = 1;
    int ni = (int)n, complete = c->cfg.stage2_complete;
    void* args[] = {&a, &ni, &prog, &complete};
    SVDB_CHECK(c, cudaLaunchCooperativeKernel((void*)kern, dim3((unsigned)G), dim3(kFastThreads), args, smem, c->stream));
    c->launches++;
    return 0;
}
template int stage2_chase_fast<float>(Ctx*, float*, size_t, size_t, int*);
template int stage2_chase_fast<double>(Ctx*, double*, size_t, size_t, int*);

}  // namespace svdb200

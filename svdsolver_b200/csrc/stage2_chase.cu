// Stage 2: band -> bidiagonal by bulge chasing.  Replaces csc586::parallel::brd_p2<T>
// (svd_parallel.h:640-695; kernels band_rd_top 569-589, band_rd_right 600-608, band_rd_left 617-624).
//
// B200 design
//   * one CTA per in-flight sweep; sweeps are pipelined across SMs.  Window op q of sweep i+1
//     (ops numbered RIGHT(p) = 2p, LEFT(p) = 2p+1) overlaps ops of sweep i only up to index q+3
//     (brute-force check in tests/test_oracle.py), so it may start once sweep i has completed
//     q+4 ops: one per-sweep progress counter in global memory (st.release / ld.acquire);
//   * consecutive ops of a sweep share half of their window: RIGHT(p) = [F; N] hands its lower
//     block to LEFT(p) = [F | N], which hands its right block to RIGHT(p+1).  The forwarded block F
//     never leaves shared memory; only the new block N (c x c) is fetched from L2 -- and that fetch
//     is overlapped with the norm / Householder / H computation, which needs F only -- and only the
//     finished block is written back.  All inter-CTA data goes through L2 (ld.global.cg /
//     st.global.cg), never the non-coherent L1;
//   * arithmetic is BIT-FAITHFUL to the reference: explicit H = I - tau w w^T, window*H / H*window
//     with k-ascending sums from 0, separate (never fused) multiply and add, reflector scalars in
//     double -- so the kernel reproduces data/bidiagonal_* exactly when fed data/band_* (SURVEY 0.7);
//   * the reference's window schedule is reproduced including its boundary behaviour (SURVEY 0.3).
#include <algorithm>
#include <climits>
#include "common.cuh"
#include "stage2_common.cuh"

namespace svdb200 {

namespace {

#ifndef SVDB_S2_TIMING
#define SVDB_S2_TIMING 0
#endif
__device__ long long g_s2_dbg[16];
#define S2_TICK(k)                                                          \
    do {                                                                    \
        if (SVDB_S2_TIMING && blockIdx.x == 1 && threadIdx.x == 0) {        \
            long long _t = clock64();                                       \
            g_s2_dbg[k] += _t - tick;                                       \
            tick = _t;                                                      \
        }                                                                   \
    } while (0)

using namespace s2;

// kC: the band as a compile-time constant (32 / 64: the sizes the configs use), 0 = any band at run time
template <typename T, int kMaxThreads, int kMinBlocks, int kC>
__global__ void __launch_bounds__(kMaxThreads, kMinBlocks) stage2_chase_kernel(T* __restrict__ A0, int n, int band, int* __restrict__ prog0,
                                                                      int count, int G, int complete) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int c = kC > 0 ? kC : band, w = c + 1;
    const int ldr = c + 1, ldl = 2 * c + 1, ldh = c + 1;
    T* WR = reinterpret_cast<T*>(smem_raw);     // RIGHT window [2c][c+1]
    T* WL = WR + 2 * c * ldr;                   // LEFT  window [c][2c+1]
    T* H = WL + c * ldl;                        // [c][c+1]
    T* sc = H + c * ldh;                        // alpha, tau
    const int tid = threadIdx.x, nt = blockDim.x;
    const size_t N = (size_t)n;
    const int tx = tid % c, ty = tid / c, tys = nt / c;   // 2-D view of the CTA: c columns x tys rows (nt >= c)

    // Batched use: the grid is split into groups of G CTAs; a group pipelines the sweeps of one matrix at a time
    // (matrices group, group + #groups, ...).  Progress counters are per matrix and pre-zeroed, so a CTA that runs
    // ahead into its group's next matrix only ever waits on counters of that matrix.  Single matrix: count = 1,
    // G = gridDim.x.
    const int grp = blockIdx.x / G, rank = blockIdx.x - grp * G, ngroups = gridDim.x / G;
    for (int mat = grp; mat < count; mat += ngroups) {
    T* __restrict__ A = A0 + (size_t)mat * N * N;
    int* __restrict__ prog = prog0 + (size_t)mat * N;
    long long tick = SVDB_S2_TIMING ? clock64() : 0;
    (void)tick;
    const int rel_tid = nt > 32 ? 32 : 0;                   // the progress counter is published by a thread off thread 0's path
    for (int i = rank; i < n - 1; i += G) {
        int seen = 0;                                         // last observed progress of sweep i-1 (thread 0 only)
        const int top_j2 = min(i + 2 * w - 1, n);
        // reference schedule: svd_parallel.h:664 (floor, the ceil there acts on an integer quotient).  complete: pairs
        // while their window is non-empty -- chases every bulge to the matrix edge (see svdb200_set_stage2_schedule).
        const int npairs = complete ? (n - i - 1 + c - 1) / c : 1 + (n - top_j2) / c + 1;
        int fr = 0;                               // rows of the forwarded block sitting in WR (0: none)
        for (int p = 0; p < npairs; ++p) {
            const int r0 = (p == 0) ? i : min(i + 1 + (p - 1) * c, n);
            const int r1 = min(i + 1 + p * c, n), r2 = min(i + 1 + (p + 1) * c, n), c3 = min(i + 1 + (p + 2) * c, n);
            if (r2 <= r1) break;                  // empty pair (only possible as the very last one)
            // ================= RIGHT(p): rows [r0,r2) x cols [r1,r2), window = [F; N] ===================
            {
                const int q = 2 * p;
                S2_TICK(0);
                if (i > 0) {
                    if (tid == 0) seen = wait_progress(&prog[i - 1], q + 4, seen);
                    S2_TICK(1);
                    __syncthreads();
                }
                S2_TICK(2);
                const int nc = r2 - r1, nr = r2 - r0;
                const int have = fr;              // rows [0,have) of WR already hold F
                T nv[kNewPerThread];
                const int newcnt = (nr - have) * nc;
                if (have == 0) {                  // top pair: the whole window (x included) comes from L2
                    for (int e = tid; e < newcnt; e += nt)
                        WR[(e / nc) * ldr + e % nc] = ld_cg(&A[(size_t)(r0 + e / nc) * N + (r1 + e % nc)]);
                    __syncthreads();
                } else {                          // issue the fetch of N, consume it after H is built
#pragma unroll
                    for (int u = 0; u < kNewPerThread; ++u) {
                        int r = ty + u * tys;
                        if (r < nr - have && tx < nc) nv[u] = ld_cg(&A[(size_t)(r0 + have + r) * N + (r1 + tx)]);
                    }
                }
                S2_TICK(3);
                if (tid == 0) reflector_scalars<T>(WR, 1, nc, sc, complete != 0);
                S2_TICK(4);
                __syncthreads();
                build_h<T>(WR, 1, nc, sc, H, ldh, tx, ty, tys);
                if (have != 0) {
#pragma unroll
                    for (int u = 0; u < kNewPerThread; ++u) {
                        int r = ty + u * tys;
                        if (r < nr - have && tx < nc) WR[(have + r) * ldr + tx] = nv[u];
                    }
                }
                __syncthreads();
                S2_TICK(5);
                // rows [r0,r1) are finished for this sweep; rows [r1,r2) become LEFT(p)'s left block
                const int keep = r1 - r0;
                window_product<T, kC>(WR, ldr, H, ldh, nr, nc, nc, (c + 1) / 2, (c + 1) / 2,
                                  [&](int r, int cc, T v) {
                                      if (r < keep) st_cg(&A[(size_t)(r0 + r) * N + (r1 + cc)], v);
                                      else WL[(r - keep) * ldl + cc] = v;
                                  }, tid);
                S2_TICK(6);
                __syncthreads();
                S2_TICK(7);
                if (tid == rel_tid) st_release(&prog[i], q + 1);
            }
            // ================= LEFT(p): rows [r1,r2) x cols [r1,c3), window = [F | N] ====================
            const int nn = c3 - r2;
            const bool fwd = (p + 1 < npairs) && nn > 0;   // is there a RIGHT(p+1) to hand the right block to
            {
                const int q = 2 * p + 1;
                if (i > 0) {
                    if (tid == 0) seen = wait_progress(&prog[i - 1], q + 4, seen);
                    __syncthreads();
                }
                const int nr = r2 - r1, fc = r2 - r1, nc = fc + nn;
                T nv[kNewPerThread];
#pragma unroll
                for (int u = 0; u < kNewPerThread; ++u) {
                    int r = ty + u * tys;
                    if (r < nr && tx < nn) nv[u] = ld_cg(&A[(size_t)(r1 + r) * N + (r2 + tx)]);
                }
                if (tid == 0) reflector_scalars<T>(WL, ldl, nr, sc, complete != 0);
                __syncthreads();
                build_h<T>(WL, ldl, nr, sc, H, ldh, tx, ty, tys);
#pragma unroll
                for (int u = 0; u < kNewPerThread; ++u) {
                    int r = ty + u * tys;
                    if (r < nr && tx < nn) WL[r * ldl + fc + tx] = nv[u];
                }
                __syncthreads();
                // cols [r1,r2) are finished; cols [r2,c3) become the top block of RIGHT(p+1)
                window_product<T, kC>(H, ldh, WL, ldl, nr, nc, nr, c, (c + 3) / 4,
                                  [&](int r, int cc, T v) {
                                      if (cc < fc || !fwd) st_cg(&A[(size_t)(r1 + r) * N + (r1 + cc)], v);
                                      else WR[r * ldr + (cc - fc)] = v;
                                  }, tid);
                fr = fwd ? nr : 0;
                __syncthreads();
                if (tid == rel_tid && fwd) st_release(&prog[i], q + 1);
            }
            if (!fwd) break;
        }
        if (tid == rel_tid) st_release(&prog[i], INT_MAX);
    }
    }
}

}  // namespace
int stage2_debug_read(long long* out16) {
    long long z[16] = {};
    if (cudaMemcpyFromSymbol(out16, g_s2_dbg, sizeof(z)) != cudaSuccess) return 1;
    cudaMemcpyToSymbol(g_s2_dbg, z, sizeof(z));
    return 0;
}
namespace {

template <typename T>
__global__ void extract_bidiagonal_kernel(const T* __restrict__ A, int n, T* __restrict__ d, T* __restrict__ e) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    A += (size_t)blockIdx.y * n * n;                 // batched: one matrix per blockIdx.y, d/e rows of length n
    if (d) d += (size_t)blockIdx.y * n;
    if (e) e += (size_t)blockIdx.y * n;
    if (i < n) {
        if (d) d[i] = A[(size_t)i * n + i];
        if (e && i + 1 < n) e[i] = A[(size_t)i * n + i + 1];
    }
}

}  // namespace

template <typename T>
int stage2_chase_batched(Ctx* c, T* a, size_t n, size_t band, T* d, T* e, int count) {
    if (n < 2 || band < 1 || count < 1) return SVDB200_E_SHAPE;
    if (n > (size_t)INT_MAX / 4) return SVDB200_E_CAPACITY;
    const int cb = (int)band;
    ProfScope ps(c, 4, 4.0 * (double)band * (double)n * (double)n * sizeof(T) * count);
    size_t smem = (size_t)(2 * cb * (cb + 1) + cb * (2 * cb + 1) + cb * (cb + 1) + 8) * sizeof(T);
    int nt = stage2_threads(cb);
    if (nt > 1024) return SVDB200_E_CAPACITY;      // band <= 64
    if (cb * cb > kNewPerThread * nt) return SVDB200_E_CAPACITY;
    if (smem > 227 * 1024) return SVDB200_E_CAPACITY;
    // small bands run with <= 256 threads: instantiate that case without the 64-register cap; a batch wants
    // several CTAs per SM instead (the window product is FP64-issue bound for ~40 % of an op, the rest is latency)
    const bool light = count > 1;
    auto kern = nt <= 256 ? (light ? stage2_chase_kernel<T, 256, 3, 0> : stage2_chase_kernel<T, 256, 1, 0>)
                          : stage2_chase_kernel<T, 1024, 1, 0>;
    if (cb == 32) kern = light ? stage2_chase_kernel<T, 256, 3, 32> : stage2_chase_kernel<T, 256, 1, 32>;   // band-specialised
    else if (cb == 64) kern = stage2_chase_kernel<T, 1024, 1, 64>;                                           // (same arithmetic)
    SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    SVDB_CHECK(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, nt, smem));
    if (per_sm < 1) return SVDB200_E_CAPACITY;
    // No more sweeps of one matrix can be in flight than the pipeline admits (one every 2 pairs).
    long long inflight = (long long)(n / band) / 2 + 2;
    if (count > 1) inflight = std::max<long long>(1, (long long)(n / band + 1) / 2);   // no idle CTAs in a batch
    long long slots = (long long)per_sm * c->num_sms;
    long long G = std::min(inflight, std::min(slots, (long long)n - 1));
    if (G < 1) G = 1;
    long long groups = std::min((long long)count, slots / G);
    if (groups < 1) groups = 1;
    const long long grid = groups * G;
    int* prog = c->prog;
    if (count > 1) {
        const size_t need = (size_t)count * n;
        if (c->batch_prog_elems < need) {
            if (c->batch_prog) cudaFree(c->batch_prog);
            c->batch_prog = nullptr; c->batch_prog_elems = 0;
            SVDB_CHECK(c, cudaMalloc(&c->batch_prog, sizeof(int) * need));
            c->batch_prog_elems = need;
        }
        prog = c->batch_prog;
    }
    SVDB_CHECK(c, cudaMemsetAsync(prog, 0, sizeof(int) * n * (size_t)count, c->stream));
    int ni = (int)n, bi = cb, cnt = count, gi = (int)G, complete = c->cfg.stage2_complete;
    int fast = 1;                                                      // 0 = the latency-optimised band-32 kernel ran
    if (count == 1) {
        fast = stage2_chase_fast<T>(c, a, n, band, prog);
        if (fast != 0 && fast != 1) return fast;
    }
    if (fast != 0) {
        void* args[] = {&a, &ni, &bi, &prog, &cnt, &gi, &complete};
        SVDB_CHECK(c, cudaLaunchCooperativeKernel((void*)kern, dim3((unsigned)grid), dim3(nt), args, smem, c->stream));
        c->launches++;
    }
    if (d || e) {
        extract_bidiagonal_kernel<T><<<dim3((unsigned)((n + 255) / 256), (unsigned)count), 256, 0, c->stream>>>(a, ni, d, e);
        SVDB_CHECK(c, cudaGetLastError());
        c->launches++;
    }
    return 0;
}

template <typename T>
int stage2_chase(Ctx* c, T* a, size_t n, size_t band, T* d, T* e) { return stage2_chase_batched<T>(c, a, n, band, d, e, 1); }

// d = diag(A), e = diag(A, 1) of a device matrix (what Bidiagonal{A.diag(), A.diag(1)} returns, svd_serial.h:264)
template <typename T>
int extract_bidiagonal(Ctx* c, const T* a, size_t n, T* d, T* e) {
    if (!d && !e) return 0;
    extract_bidiagonal_kernel<T><<<dim3((unsigned)((n + 255) / 256), 1), 256, 0, c->stream>>>(a, (int)n, d, e);
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    return 0;
}
template int extract_bidiagonal<float>(Ctx*, const float*, size_t, float*, float*);
template int extract_bidiagonal<double>(Ctx*, const double*, size_t, double*, double*);

template int stage2_chase_batched<float>(Ctx*, float*, size_t, size_t, float*, float*, int);
template int stage2_chase_batched<double>(Ctx*, double*, size_t, size_t, double*, double*, int);
template int stage2_chase<float>(Ctx*, float*, size_t, size_t, float*, float*);
template int stage2_chase<double>(Ctx*, double*, size_t, size_t, double*, double*);

}  // namespace svdb200

// C ABI of libsvdb200.so (declared in include/svdb200.h).  Thin: argument checks, workspace
// ownership, host<->device staging and CUDA-event timing; all arithmetic lives in the kernels.
// Every dense single-matrix call runs run_chain on the device; every single-matrix host-pointer
// call is one host_call (copies in, device work, copies out, one synchronise, stage timings).
#include <algorithm>
#include <initializer_list>
#include <new>
#include "common.cuh"

using namespace svdb200;

namespace svdb200 {
template <typename T, bool kTrans> int launch_panel_public(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream);
namespace {

// ---- small utility kernels ------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
// element i = lo + (hi-lo) * (splitmix64(seed+i) >> 11) * 2^-53, evaluated in double, rounded to T
// (svdsolver_b200/synth.py is the host mirror).  No FMA contraction so host and device agree bitwise.
template <typename T>
__global__ void fill_uniform_kernel(T* __restrict__ a, size_t count, unsigned long long seed, double lo, double hi) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t stride = (size_t)gridDim.x * blockDim.x;
    const double span = __dsub_rn(hi, lo);
    for (; i < count; i += stride) {
        double u = __dmul_rn((double)(splitmix64(seed + i) >> 11), 1.0 / 9007199254740992.0);
        a[i] = (T)__dadd_rn(lo, __dmul_rn(span, u));
    }
}

// gpu::Matrix<T>::mse (matrix_gpu.h:438-453): sum over i, j in [i, min(i+band, n)) of | |a|-|b| |,
// divided by band*nrows.  (The reference accumulates in float in row order; this is a reported
// metric, not a parity target, so a tree reduction in double is used.)
template <typename T>
__global__ void mse_kernel(const T* __restrict__ a, const T* __restrict__ b, int n, int band, double* __restrict__ out) {
    __shared__ double sh[256];
    double acc = 0.0;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < (size_t)n * band; e += (size_t)gridDim.x * blockDim.x) {
        int i = (int)(e / band), j = i + (int)(e % band);
        if (j < n) acc += fabs(fabs((double)a[(size_t)i * n + j]) - fabs((double)b[(size_t)i * n + j]));
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) atomicAdd(out, sh[0]);
}

// ---- register-resident peak probes (roofline denominators) -----------------------------------------
template <int KIND>
__global__ void __launch_bounds__(256) peak_kernel(double* sink, int iters) {
    const int lane = threadIdx.x & 31;
    if (KIND == 0) {                       // DFMA: 8 independent chains
        double a = 1.0 + lane * 1e-9, b = 0.999999, c[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) c[i] = i;
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < 8; ++i) c[i] = fma(a, b, c[i]);
#pragma unroll
            for (int i = 0; i < 8; ++i) c[i] = fma(c[i], b, a);
        }
        double s = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += c[i];
        if (s == 123.456) sink[0] = s;
    } else if (KIND == 1) {                // DMMA m8n8k4: 8 independent accumulator tiles
        double a = 1.0 + lane * 1e-9, b = 0.5, c[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) c[i] = 0;
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
                asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                             : "+d"(c[2 * i]), "+d"(c[2 * i + 1]) : "d"(a), "d"(b));
        }
        double s = 0;
#pragma unroll
        for (int i = 0; i < 16; ++i) s += c[i];
        if (s == 123.456) sink[0] = s;
    } else if (KIND == 2) {                // FFMA
        float a = 1.0f + lane * 1e-6f, b = 0.99999f, c[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) c[i] = (float)i;
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < 8; ++i) c[i] = fmaf(a, b, c[i]);
#pragma unroll
            for (int i = 0; i < 8; ++i) c[i] = fmaf(c[i], b, a);
        }
        float s = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i) s += c[i];
        if (s == 123.456f) sink[0] = s;
    } else {                               // TF32 mma.sync m16n8k8
        uint32_t a[4] = {0x3f800000u, 0x3f800000u, 0x3f800000u, 0x3f800000u}, b[2] = {0x3f000000u, 0x3f000000u};
        float c[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) c[i] = 0.f;
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
                asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                             : "+f"(c[4 * i]), "+f"(c[4 * i + 1]), "+f"(c[4 * i + 2]), "+f"(c[4 * i + 3])
                             : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
        }
        float s = 0;
#pragma unroll
        for (int i = 0; i < 32; ++i) s += c[i];
        if (s == 123.456f) sink[0] = s;
    }
}

}  // namespace

template <typename T>
int fill_uniform(Ctx* c, T* a, size_t count, unsigned long long seed, double lo, double hi) {
    if (count == 0) return 0;
    unsigned blocks = (unsigned)((count + 255) / 256);
    if (blocks > 148u * 16u) blocks = 148u * 16u;
    fill_uniform_kernel<T><<<blocks, 256, 0, c->stream>>>(a, count, seed, lo, hi);
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    return 0;
}
template int fill_uniform<float>(Ctx*, float*, size_t, unsigned long long, double, double);
template int fill_uniform<double>(Ctx*, double*, size_t, unsigned long long, double, double);

template <typename T>
int mse_metric(Ctx* c, const T* a, const T* b, size_t n, size_t band, T* out_host) {
    double* acc = reinterpret_cast<double*>(c->qr_info + 4);
    SVDB_CHECK(c, cudaMemsetAsync(acc, 0, sizeof(double), c->stream));
    mse_kernel<T><<<148, 256, 0, c->stream>>>(a, b, (int)n, (int)band, acc);
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    double h = 0;
    SVDB_CHECK(c, cudaMemcpyAsync(&h, acc, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    SVDB_CHECK(c, cudaStreamSynchronize(c->stream));
    *out_host = (T)(h / ((double)band * (double)n));
    return 0;
}
template int mse_metric<float>(Ctx*, const float*, const float*, size_t, size_t, float*);
template int mse_metric<double>(Ctx*, const double*, const double*, size_t, size_t, double*);

int probe_peak(Ctx* c, int kind, double* tflops) {
    if (kind < 0 || kind > 3 || !tflops) return SVDB200_E_ARG;
    double* sink = reinterpret_cast<double*>(c->qr_info + 4);
    const int iters = 20000, blocks = c->num_sms * 8, threads = 256;
    cudaEvent_t e0 = c->ev[6], e1 = c->ev[7];
    double best = 0;
    for (int rep = 0; rep < 3; ++rep) {
        SVDB_CHECK(c, cudaEventRecord(e0, c->stream));
        switch (kind) {
            case 0: peak_kernel<0><<<blocks, threads, 0, c->stream>>>(sink, iters); break;
            case 1: peak_kernel<1><<<blocks, threads, 0, c->stream>>>(sink, iters); break;
            case 2: peak_kernel<2><<<blocks, threads, 0, c->stream>>>(sink, iters); break;
            default: peak_kernel<3><<<blocks, threads, 0, c->stream>>>(sink, iters); break;
        }
        SVDB_CHECK(c, cudaGetLastError());
        c->launches++;
        SVDB_CHECK(c, cudaEventRecord(e1, c->stream));
        SVDB_CHECK(c, cudaEventSynchronize(e1));
        float ms = 0;
        SVDB_CHECK(c, cudaEventElapsedTime(&ms, e0, e1));
        double flops;
        if (kind == 0 || kind == 2) flops = (double)blocks * threads * iters * 16.0 * 2.0;
        else if (kind == 1) flops = (double)blocks * (threads / 32) * iters * 8.0 * (8.0 * 8.0 * 4.0 * 2.0);
        else flops = (double)blocks * (threads / 32) * iters * 8.0 * (16.0 * 8.0 * 8.0 * 2.0);
        double tf = flops / (ms * 1e-3) * 1e-12;
        if (tf > best) best = tf;
    }
    *tflops = best;
    return 0;
}

// Batched driver (BASELINE config 5): the matrices are independent, so they are spread round-robin
// over a pool of sub-handles, each with its own stream and workspace; the small kernels of
// different matrices overlap on the GPU (a 256 x 256 reduction cannot fill 148 SMs on its own).
// Shards by matrix across GPUs at the caller's level (one handle per GPU), no collective.
constexpr int kBatchPool = 16;

// Sub-handles (batch pool, stage-1 chains of the pipelined driver) follow the parent's settings on every call,
// not only those set after the sub-handle was created.
static void inherit_settings(const Ctx* c, Ctx* s) { s->cfg = c->cfg; }

// Small matrices (min(m, n) <= 1024, band <= 64): every kernel of the path runs ONCE PER STEP FOR THE WHOLE BATCH -- a
// thread-block cluster per matrix for the panels (panel resident in cluster shared memory), one grid slice per
// matrix for the three update GEMMs, groups of CTAs that pipeline the sweeps of one matrix each for stage 2, one
// thread per singular value for the bisection -- instead of ~80 launches per matrix.  The matrices of a chunk stay
// L2 / HBM resident.  `a` holds count m x n matrices back to back; with k = min(m, n), the rows of d, e and sigma have
// length k.  Tall (m >= n): the QR panels of step j span rows j .. m-1 (as in stage1_panel_order), and stage 2 and sigma
// run on the top k x k block, which is upper band.  Wide (m < n): each A^T is reduced as tall in the chunk's workspace and
// transposed back, so `a` ends in gebrd's lower form (as in run_chain).  Workspace per matrix of a chunk: 5 max(m, n) b
// + 2 k elements, plus m n for A^T when m < n.
static bool batched_in_range(const Ctx* c, size_t m, size_t n, size_t band) {
    const size_t k = std::min(m, n);
    return k >= 2 && k <= 1024 && band <= 64 && c->cluster_ok >= 8 && panel_batched_fits((int)std::max(m, n), (int)band, c->esz);
}

template <typename T>
int batched_small(Ctx* c, T* a, size_t count, size_t m, size_t n, size_t band, T* sigma, int what = 7, T* d_out = nullptr,
                  T* e_out = nullptr) {
    if ((what & 4) && !(what & 2) && (!d_out || !e_out)) return SVDB200_E_ARG;
    const int b = (int)band;
    const bool wide = m < n && (what & 3);
    const size_t N = std::min(m, n), M = std::max(m, n);       // the tall matrices reduced: M x N, ld = N
    const size_t sA = m * n, sV = M * band;
    const size_t per_mat = 5 * sV + 2 * N + (wide ? sA : 0);
    size_t chunk = std::min<size_t>(count, 8192);
    while (chunk > 1 && chunk * per_mat * sizeof(T) > ((size_t)2 << 30)) chunk = (chunk + 1) / 2;
    SVDB_TRY(reserve(c, c->batch_ws, chunk * per_mat * sizeof(T)));
    T* Vq = reinterpret_cast<T*>(c->batch_ws.p);
    T* V2q = Vq + chunk * sV;
    T* Vl = V2q + chunk * sV;
    T* V2l = Vl + chunk * sV;
    T* W = V2l + chunk * sV;
    T* dall = W + chunk * sV;
    T* eall = dall + chunk * N;
    T* xt = eall + chunk * N;                                  // wide: the chunk's A^T
    for (size_t z0 = 0; z0 < count; z0 += chunk) {
        const int cnt = (int)std::min(chunk, count - z0);
        T* x0 = a + z0 * sA;
        if (wide) {
            SVDB_TRY(transpose_batched<T>(c, x0, sA, m, n, xt, sA, cnt));
            x0 = xt;
        }
        for (size_t j = 0; (what & 1) && j < N; j += band) {   // same panel sequence as stage1_panel_order (svd_cpu.h:382-423)
            const int mh = (int)(M - j), nc = (int)(N - j - band);
            const bool has_lq = (j + band < N - 1);
            SVDB_TRY((panel_batched<T, false>(c, x0 + j * N + j, N, sA, mh, b, Vq, V2q, sV, cnt)));
            if (nc > 0) {
                T* A2 = x0 + j * N + j + band;
                SVDB_TRY(gemm_tn_batched<T>(c, Vq, sV, A2, N, sA, mh, nc, b, W, sV, cnt));                    // W = V^T A2
                SVDB_TRY(rank_update_batched<T>(c, A2, N, sA, mh, nc, b, V2q, sV, W, (size_t)nc, sV, cnt));    // A2 += (V S^T) W
                if (has_lq) {
                    SVDB_TRY((panel_batched<T, true>(c, A2, N, sA, nc, b, Vl, V2l, sV, cnt)));               // LQ of the row panel
                    const int mr = mh - b;
                    if (mr > 0) {
                        T* A3 = x0 + (j + band) * N + j + band;
                        SVDB_TRY(gemm_nn_batched<T>(c, A3, N, sA, mr, nc, b, Vl, sV, W, sV, cnt));            // W = A3 U^T
                        SVDB_TRY(rank_update_batched<T>(c, A3, N, sA, mr, nc, b, W, sV, V2l, (size_t)nc, sV, cnt));
                    }
                }
            }
        }
        if (what & 2) {
            SVDB_TRY(stage2_chase_batched<T>(c, x0, sA, N, band, dall, eall, cnt));
            if (d_out) SVDB_CHECK(c, cudaMemcpyAsync(d_out + z0 * N, dall, sizeof(T) * N * cnt, cudaMemcpyDeviceToDevice, c->stream));
            if (e_out) SVDB_CHECK(c, cudaMemcpyAsync(e_out + z0 * N, eall, sizeof(T) * N * cnt, cudaMemcpyDeviceToDevice, c->stream));
        }
        if (wide) SVDB_TRY(transpose_batched<T>(c, xt, sA, n, m, a + z0 * sA, sA, cnt));
        if (!(what & 4)) continue;
        if (!(what & 2)) {                                // sigma of caller-provided bidiagonals
            SVDB_CHECK(c, cudaMemcpyAsync(dall, d_out + z0 * N, sizeof(T) * N * cnt, cudaMemcpyDeviceToDevice, c->stream));
            SVDB_CHECK(c, cudaMemcpyAsync(eall, e_out + z0 * N, sizeof(T) * N * cnt, cudaMemcpyDeviceToDevice, c->stream));
        }
        if (c->cfg.qr_method == 1) {                      // the reference's zero-shift QR sweeps, one CTA per matrix
            for (int i = 0; i < cnt; ++i) SVDB_TRY(bidiag_qr<T>(c, dall + (size_t)i * N, eall + (size_t)i * N, N, sigma + (z0 + i) * N));
        } else {
            for (int i0 = 0; i0 < cnt; i0 += 32768) {
                const int ic = std::min(32768, cnt - i0);
                SVDB_TRY(bidiag_bisect_batched<T>(c, dall + (size_t)i0 * N, eall + (size_t)i0 * N, N, sigma + (z0 + i0) * N, ic));
            }
        }
    }
    return 0;
}

template <typename T>
int batched_svdvals(Ctx* c, T* a, size_t count, size_t n, size_t band, T* sigma) {
    if (count == 0) return 0;
    if (batched_in_range(c, n, n, band)) return batched_small<T>(c, a, count, n, n, band, sigma);
    if (c->pool_n != n || c->pool_band != band) {
        for (auto& h : c->pool) if (h) { svdb200_destroy(reinterpret_cast<svdb200_handle>(h)); h = nullptr; }
        c->pool.clear();
        for (int i = 0; i < kBatchPool; ++i) {
            svdb200_handle h = nullptr;
            int st = svdb200_create(&h, c->device, n, band, c->dtype);
            if (st != 0) return st;
            c->pool.push_back(reinterpret_cast<Ctx*>(h));
        }
        c->pool_n = n; c->pool_band = band;
    }
    // Several matrices in flight: stage 1 may then only use kernels without cross-cluster / grid-wide spin waits (their
    // CTAs must all be co-resident, which the neighbours' panels and cooperative stage-2 grids could prevent:
    // stage1_panel_reg.cu).  Matrices whose panels need those kernels (n > kOverlapMaxN) go one after the other instead.
    const bool concurrent = n <= 4096;
    const int K = concurrent ? (int)std::min<size_t>(c->pool.size(), count) : 1;
    SVDB_CHECK(c, cudaEventRecord(c->lev[0], c->stream));            // inputs are ready on the caller's stream
    for (int i = 0; i < K; ++i) SVDB_CHECK(c, cudaStreamWaitEvent(c->pool[i]->stream, c->lev[0], 0));
    for (size_t i = 0; i < count; ++i) {
        Ctx* s = c->pool[i % K];
        inherit_settings(c, s);
        T* ai = a + i * n * n;
        T* d = reinterpret_cast<T*>(s->d);
        T* e = reinterpret_cast<T*>(s->e);
        const long long before = s->launches;
        s->overlap_safe = (concurrent && K > 1) ? 1 : 0;
        const int st1 = stage1_panel_order<T>(s, ai, n, n, band);
        s->overlap_safe = 0;
        if (st1 != 0) { c->last_error = s->last_error; return st1; }
        SVDB_TRY(stage2_chase<T>(s, ai, n, band, d, e));
        SVDB_TRY(bidiag_qr<T>(s, d, e, n, sigma + i * n));
        c->launches += s->launches - before;
    }
    for (int i = 0; i < K; ++i) {                                    // join
        SVDB_CHECK(c, cudaEventRecord(c->pool[i]->lev[0], c->pool[i]->stream));
        SVDB_CHECK(c, cudaStreamWaitEvent(c->stream, c->pool[i]->lev[0], 0));
    }
    return 0;
}
// The stages of the batched path (m x n matrices, m == n for the square call); outside the range of its kernels there is
// no other batched path: SVDB200_E_CAPACITY, with nothing enqueued
template <typename T>
int batched_chain(Ctx* c, T* a, size_t count, size_t m, size_t n, size_t band, int what, T* d, T* e, T* sigma) {
    if (count == 0) return 0;
    if (!batched_in_range(c, m, n, band)) return SVDB200_E_CAPACITY;
    return batched_small<T>(c, a, count, m, n, band, sigma, what, d, e);
}
template int batched_chain<float>(Ctx*, float*, size_t, size_t, size_t, size_t, int, float*, float*, float*);
template int batched_chain<double>(Ctx*, double*, size_t, size_t, size_t, size_t, int, double*, double*, double*);
template int batched_svdvals<float>(Ctx*, float*, size_t, size_t, size_t, float*);
template int batched_svdvals<double>(Ctx*, double*, size_t, size_t, size_t, double*);

// Pipelined driver for a list of independent matrices (different sizes allowed): stage 2 of matrix i runs on its own
// stream beside stage 1 of matrix i+1 -- and beside stage 2 of matrix i-1: up to Ctx::kLanes sweep pipelines are in
// flight.  Both stages are latency-bound at moderate n (a bulge-chasing sweep pipeline uses n/(2b)+2 CTAs, a panel
// factorisation one cluster), so together they fill a B200 much better than one after the other.
// Stage 1 is restricted to kernels without cross-cluster / grid-wide waits while a stage-2 kernel may be resident
// (Ctx::overlap_safe): such kernels need all their CTAs co-resident, which the cooperative stage-2 grids could prevent.
// The stage-2 grids themselves always fit together (kLanes x (n/(2b)+2) CTAs <= 148 for n <= kOverlapMaxN at band >= 32;
// for narrower bands the second lane is not used).  Matrices larger than kOverlapMaxN are processed without overlap.
constexpr size_t kOverlapMaxN = 4096;

static void release_s2(Ctx* c) {
    for (int l = 0; l < Ctx::kLanes; ++l) {
        if (c->s1ctx[l]) { svdb200_destroy(reinterpret_cast<svdb200_handle>(c->s1ctx[l])); c->s1ctx[l] = nullptr; }
        if (l > 0 && c->s2_prog[l]) cudaFree(c->s2_prog[l]);
        c->s2_prog[l] = nullptr;
        if (c->s2_stream[l]) { cudaStreamDestroy(c->s2_stream[l]); c->s2_stream[l] = nullptr; }
    }
    for (auto& e : c->s2ev) if (e) { cudaEventDestroy(e); e = nullptr; }
    c->s2_ready = 0;
}

static int ensure_s2_impl(Ctx* c) {
    for (int l = 0; l < Ctx::kLanes; ++l) {
        SVDB_CHECK(c, cudaStreamCreateWithFlags(&c->s2_stream[l], cudaStreamNonBlocking));
        if (l == 0) c->s2_prog[l] = c->prog;
        else SVDB_CHECK(c, cudaMalloc(&c->s2_prog[l], sizeof(int) * (c->max_n + 8)));
        svdb200_handle h = nullptr;                                   // stage-1 sub-handle: own reflector / W workspace and streams
        int st = svdb200_create(&h, c->device, c->max_n, c->band, c->dtype);
        if (st != 0) return st;
        c->s1ctx[l] = reinterpret_cast<Ctx*>(h);
    }
    for (auto& e : c->s2ev) SVDB_CHECK(c, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return 0;
}

// the pipeline's streams, counters, events and stage-1 sub-handles: all or nothing (a failure half-way is rolled back,
// so a later call starts from scratch instead of dereferencing what was never created)
static int ensure_s2(Ctx* c) {
    if (c->s2_ready) return 0;
    const int st = ensure_s2_impl(c);
    if (st != 0) { release_s2(c); return st; }
    c->s2_ready = 1;
    return 0;
}

// chains usable for this matrix: their sweep pipelines must be co-resident beside each other
static int lanes_for(Ctx* c, size_t n, size_t band) {
    const size_t ctas = n / band / 2 + 2;                             // CTAs of one sweep pipeline, all of which must be resident
    const size_t cap = (size_t)c->num_sms - 8;                        // the 153-register stage-2 variant: one CTA per SM
    return ((size_t)Ctx::kLanes * ctas <= cap) ? Ctx::kLanes : 1;
}

template <typename T>
static int run_stage2_on_lane(Ctx* c, int lane, T* a, size_t n, size_t band, T* d, T* e) {
    cudaStream_t s0 = c->stream;
    int* p0 = c->prog;
    c->stream = c->s2_stream[lane];
    c->prog = c->s2_prog[lane];
    const int st = stage2_chase<T>(c, a, n, band, d, e);
    c->stream = s0;
    c->prog = p0;
    return st;
}

// every stream of the pipeline has finished what was enqueued so far, as seen from `into`
static int drain_into(Ctx* c, cudaStream_t into) {
    for (int l = 0; l < Ctx::kLanes; ++l) {
        SVDB_CHECK(c, cudaEventRecord(c->s2ev[4 + l], c->s2_stream[l]));
        SVDB_CHECK(c, cudaStreamWaitEvent(into, c->s2ev[4 + l], 0));
        SVDB_CHECK(c, cudaEventRecord(c->s1ctx[l]->lev[0], c->s1ctx[l]->stream));
        SVDB_CHECK(c, cudaStreamWaitEvent(into, c->s1ctx[l]->lev[0], 0));
    }
    return 0;
}

// One matrix through the pipeline.  Chain k (chosen by plan_list): stage 1 on sub-handle k's streams, stage 2 on lane k -- so kLanes
// stage-1 factorizations and kLanes sweep pipelines are in flight; within a chain stage 1 of the next matrix starts as soon
// as the previous stage 1 is done, beside that matrix's stage 2.  `h2d` (host variant): copy issued on the chain's stream.
template <typename T>
static int pipeline_one(Ctx* c, size_t i, T* a_dev, const T* a_host, size_t n, size_t band, int order, T* d, T* e, cudaStream_t* lane_out,
                        int k) {
    const bool overlap = order == SVDB200_ORDER_PANEL && n <= kOverlapMaxN && !c->profile;
    const int nl = overlap ? lanes_for(c, n, band) : 1;
    if (!overlap || nl == 1) {
        // no overlap: wait for everything, run on the parent handle, and hold the pipeline back until it is done
        SVDB_TRY(drain_into(c, c->stream));
        if (a_host) SVDB_CHECK(c, cudaMemcpyAsync(a_dev, a_host, sizeof(T) * n * n, cudaMemcpyHostToDevice, c->stream));
        SVDB_TRY(order == SVDB200_ORDER_PANEL ? stage1_panel_order<T>(c, a_dev, n, n, band) : stage1_tile_order<T>(c, a_dev, n, band));
        if (i < c->band_capture.size() && c->band_capture[i])
            SVDB_CHECK(c, cudaMemcpyAsync(c->band_capture[i], a_dev, sizeof(T) * n * n, cudaMemcpyDeviceToDevice, c->stream));
        SVDB_TRY(stage2_chase<T>(c, a_dev, n, band, d, e));
        SVDB_CHECK(c, cudaEventRecord(c->s2ev[1], c->stream));
        for (int l = 0; l < Ctx::kLanes; ++l) {
            SVDB_CHECK(c, cudaStreamWaitEvent(c->s2_stream[l], c->s2ev[1], 0));
            SVDB_CHECK(c, cudaStreamWaitEvent(c->s1ctx[l]->stream, c->s2ev[1], 0));
        }
        *lane_out = c->stream;
        return 0;
    }
    Ctx* s = c->s1ctx[k];
    inherit_settings(c, s);
    if (a_host) SVDB_CHECK(c, cudaMemcpyAsync(a_dev, a_host, sizeof(T) * n * n, cudaMemcpyHostToDevice, s->stream));
    s->overlap_safe = 1;
    int st = stage1_panel_order<T>(s, a_dev, n, n, band);
    s->overlap_safe = 0;
    c->launches += s->launches; s->launches = 0;
    if (st != 0) { c->last_error = s->last_error; return st; }
    if (i < c->band_capture.size() && c->band_capture[i])            // test hook: the band this matrix enters stage 2 with
        SVDB_CHECK(c, cudaMemcpyAsync(c->band_capture[i], a_dev, sizeof(T) * n * n, cudaMemcpyDeviceToDevice, s->stream));
    SVDB_CHECK(c, cudaEventRecord(s->lev[0], s->stream));
    SVDB_CHECK(c, cudaStreamWaitEvent(c->s2_stream[k], s->lev[0], 0));
    SVDB_TRY(run_stage2_on_lane<T>(c, k, a_dev, n, band, d, e));
    *lane_out = c->s2_stream[k];
    return 0;
}

// Which chain works on which matrix, and in which order the matrices are issued.  The chains are bound by their stage-2 lanes
// (stage-2 time ~ n), so the matrices are partitioned by longest-processing-time-first over the chains; inside a chain they
// run in ascending size, and the issue order alternates between the chains.  (The reference's benchmark list is ascending:
// dealing it out i % lanes leaves the last chain 8 % longer than the first.  Odd chains running large-to-small -- so that
// the large pipelines of two chains do not coincide -- measured slower: 2718 vs 3011 GFLOP/s.)  Results do not depend on
// the order.
struct ListPlan { std::vector<size_t> order; std::vector<int> chain; };
static ListPlan plan_list(int lanes, size_t count, const size_t* n) {
    ListPlan pl;
    const int L = lanes < 1 ? 1 : lanes;
    pl.order.reserve(count); pl.chain.reserve(count);
    if (L == 1 || count <= (size_t)L) {
        for (size_t i = 0; i < count; ++i) { pl.order.push_back(i); pl.chain.push_back((int)(i % (size_t)L)); }
        return pl;
    }
    std::vector<size_t> idx(count);
    for (size_t i = 0; i < count; ++i) idx[i] = i;
    std::stable_sort(idx.begin(), idx.end(), [&](size_t x, size_t y) { return n[x] > n[y]; });
    std::vector<std::vector<size_t>> items(L);
    std::vector<size_t> load(L, 0);
    for (size_t i : idx) {
        int best = 0;
        for (int l = 1; l < L; ++l) if (load[l] < load[best]) best = l;
        items[best].push_back(i);
        load[best] += n[i];
    }
    for (auto& v : items) std::stable_sort(v.begin(), v.end(), [&](size_t x, size_t y) { return n[x] != n[y] ? n[x] < n[y] : x < y; });
    for (size_t t = 0; pl.order.size() < count; ++t)
        for (int l = 0; l < L; ++l)
            if (t < items[l].size()) { pl.order.push_back(items[l][t]); pl.chain.push_back(l); }
    return pl;
}

template <typename T>
int bidiagonalize_many_dev(Ctx* c, size_t count, T* const* a, const size_t* n, size_t band, int order, T* const* d, T* const* e) {
    if (count == 0) return 0;
    SVDB_TRY(ensure_s2(c));
    cudaStream_t s0 = c->stream;
    SVDB_CHECK(c, cudaEventRecord(c->s2ev[0], s0));                  // the pipeline sees everything enqueued on the caller's stream
    for (int l = 0; l < Ctx::kLanes; ++l) {
        SVDB_CHECK(c, cudaStreamWaitEvent(c->s2_stream[l], c->s2ev[0], 0));
        SVDB_CHECK(c, cudaStreamWaitEvent(c->s1ctx[l]->stream, c->s2ev[0], 0));
    }
    const ListPlan pl = plan_list(Ctx::kLanes, count, n);
    for (size_t j = 0; j < count; ++j) {
        const size_t i = pl.order[j];
        cudaStream_t lane;
        SVDB_TRY(pipeline_one<T>(c, i, a[i], (const T*)nullptr, n[i], band, order, d ? d[i] : nullptr, e ? e[i] : nullptr, &lane, pl.chain[j]));
    }
    const int sj = drain_into(c, s0);                                 // join
    c->band_capture.clear();
    return sj;
}
template int bidiagonalize_many_dev<float>(Ctx*, size_t, float* const*, const size_t*, size_t, int, float* const*, float* const*);
template int bidiagonalize_many_dev<double>(Ctx*, size_t, double* const*, const size_t*, size_t, int, double* const*, double* const*);

// Host-pointer variant: 2 * kLanes staging buffers (two per chain), so the H2D copy of a chain's next matrix and the D2H
// copy of its previous one overlap the kernels as well.  a[i] is overwritten by the bidiagonalised matrix, d[i] / e[i]
// receive the bidiagonal.  Pinned (or registered) host buffers get fully asynchronous copies.  A copy INTO pageable memory
// blocks the calling thread until the stream reaches it, which would serialise the pipeline if it were issued right behind
// the matrix's stage 2 -- for pageable destinations the copies are therefore issued only when the staging buffer is needed
// again (NB matrices later) or at the end, while the matrices in between keep the device busy.
static bool is_pageable(const void* p) {
    if (!p) return false;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}

template <typename T>
int bidiagonalize_many_host(Ctx* c, size_t count, T* const* a, const size_t* n, size_t band, int order, T* const* d, T* const* e) {
    if (count == 0) return 0;
    SVDB_TRY(ensure_s2(c));
    constexpr int NB = 2 * Ctx::kLanes;
    SVDB_TRY(reserve(c, c->a_dev, c->esz * c->max_n * c->max_n));
    c->a_stage[0] = c->a_dev.p;
    for (int k = 1; k < NB; ++k)
        if (!c->a_stage[k]) SVDB_CHECK(c, cudaMalloc(&c->a_stage[k], c->esz * c->max_n * c->max_n));
    if (!c->de2) SVDB_CHECK(c, cudaMalloc(&c->de2, c->esz * 2 * NB * (c->max_n + 8)));
    cudaStream_t s0 = c->stream;
    SVDB_CHECK(c, cudaEventRecord(c->s2ev[0], s0));
    for (int l = 0; l < Ctx::kLanes; ++l) {
        SVDB_CHECK(c, cudaStreamWaitEvent(c->s2_stream[l], c->s2ev[0], 0));
        SVDB_CHECK(c, cudaStreamWaitEvent(c->s1ctx[l]->stream, c->s2ev[0], 0));
    }
    struct EvSet {                                                       // buffer k is free again (its D2H copies have finished)
        cudaEvent_t ev[NB] = {};
        ~EvSet() { for (auto& x : ev) if (x) cudaEventDestroy(x); }
    } evs;
    cudaEvent_t* ev_free = evs.ev;
    for (auto& ev : evs.ev) SVDB_CHECK(c, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    struct Result { T *a, *d, *e; size_t n; cudaStream_t lane; bool live; } res[NB] = {};
    auto copy_back = [&](int k) -> int {                              // results of the matrix in staging buffer k -> host
        Result& r = res[k];
        if (!r.live) return 0;
        r.live = false;
        T* buf = reinterpret_cast<T*>(c->a_stage[k]);
        T* dd = reinterpret_cast<T*>(c->de2) + (size_t)2 * k * (c->max_n + 8);
        T* ee = dd + (c->max_n + 8);
        SVDB_CHECK(c, cudaMemcpyAsync(r.a, buf, sizeof(T) * r.n * r.n, cudaMemcpyDeviceToHost, r.lane));
        if (r.d) SVDB_CHECK(c, cudaMemcpyAsync(r.d, dd, sizeof(T) * r.n, cudaMemcpyDeviceToHost, r.lane));
        if (r.e) SVDB_CHECK(c, cudaMemcpyAsync(r.e, ee, sizeof(T) * (r.n - 1), cudaMemcpyDeviceToHost, r.lane));
        SVDB_CHECK(c, cudaEventRecord(ev_free[k], r.lane));
        return 0;
    };
    int st = 0;
    const ListPlan pl = plan_list(Ctx::kLanes, count, n);
    size_t per_chain[Ctx::kLanes] = {};
    bool used[NB] = {};
    for (size_t j = 0; j < count && st == 0; ++j) {
        const size_t i = pl.order[j];
        const int ch = pl.chain[j];
        const int k = ch + Ctx::kLanes * (int)(per_chain[ch]++ % 2);  // a chain alternates between its two staging buffers
        const size_t ni = n[i];
        T* buf = reinterpret_cast<T*>(c->a_stage[k]);
        T* dd = reinterpret_cast<T*>(c->de2) + (size_t)2 * k * (c->max_n + 8);
        T* ee = dd + (c->max_n + 8);
        if ((st = copy_back(k)) != 0) break;                          // a deferred (pageable) result still sitting in this buffer
        if (used[k]) {                                                // the copy into the buffer is issued on the chain's stage-1 stream
            cudaError_t we = cudaStreamWaitEvent(c->s1ctx[ch]->stream, ev_free[k], 0);
            if (we == cudaSuccess) we = cudaStreamWaitEvent(s0, ev_free[k], 0);
            if (we != cudaSuccess) { st = cuda_status(c, we, "cudaStreamWaitEvent"); break; }
        }
        used[k] = true;
        cudaStream_t lane = s0;
        st = pipeline_one<T>(c, i, buf, a[i], ni, band, order, dd, ee, &lane, ch);
        if (st != 0) break;
        res[k] = Result{a[i], d ? d[i] : nullptr, e ? e[i] : nullptr, ni, lane, true};
        const bool defer = is_pageable(a[i]) || is_pageable(res[k].d) || is_pageable(res[k].e);
        if (!defer && (st = copy_back(k)) != 0) break;
    }
    for (int j = 0; j < NB && st == 0; ++j) st = copy_back(j);       // whatever is still deferred
    int sj = drain_into(c, s0);
    c->band_capture.clear();
    cudaError_t es = cudaStreamSynchronize(s0);                       // host buffers are valid on return
    if (st == 0 && sj != 0) return sj;
    if (st == 0 && es != cudaSuccess) return cuda_status(c, es, "cudaStreamSynchronize");
    return st;
}
template int bidiagonalize_many_host<float>(Ctx*, size_t, float* const*, const size_t*, size_t, int, float* const*, float* const*);
template int bidiagonalize_many_host<double>(Ctx*, size_t, double* const*, const size_t*, size_t, int, double* const*, double* const*);

}  // namespace svdb200

// ======================================================================================================
namespace {

template <typename T> constexpr int dtype_of();
template <> constexpr int dtype_of<float>() { return SVDB200_F32; }
template <> constexpr int dtype_of<double>() { return SVDB200_F64; }

int check_square(Ctx* c, size_t m, size_t n, size_t band, int dtype) {
    if (!c) return SVDB200_E_ARG;
    if (c->dtype != dtype) return SVDB200_E_ARG;
    if (m != n || band == 0 || n == 0 || n % band != 0) return SVDB200_E_SHAPE;
    if (n > c->max_n || band > c->band) return SVDB200_E_CAPACITY;
    return 0;
}

float elapsed(cudaEvent_t a, cudaEvent_t b) {
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    return ms;
}

// marks[k] recorded on the handle's stream (marks == nullptr: nothing recorded)
int mark(Ctx* c, cudaEvent_t* marks, int k) {
    if (marks) SVDB_CHECK(c, cudaEventRecord(marks[k], c->stream));
    return 0;
}

// The device chain of the dense single-matrix calls, square and m x n.  what: 1 = stage 1 (a -> band), 2 = stage 2 (band ->
// d, e: min(m, n) and min(m, n) - 1 entries), 4 = singular values of d, e into sigma; each bit runs its own stage only.
// Tall (m >= n): stage 1 runs in place on the m x n array; the top n x n block is then upper band, the rows below it zero,
// and stage 2 / the singular values run on that block (contiguous, ld = n) exactly as for a square matrix.  Wide (m < n):
// sigma(A) = sigma(A^T), so A is transposed into the handle's scratch, reduced there as tall and transposed back; `a` then
// holds a LOWER band / bidiagonal matrix in its left m x m block (LAPACK gebrd's convention) and e is the sub-diagonal.
// The tile order takes square matrices only.  marks (4 events, optional) are recorded after stage 1 (forward transpose
// included), after stage 2, after the singular values and after the transpose back.  Shapes are checked by the caller.
template <typename T>
int run_chain(Ctx* c, T* a, size_t m, size_t n, size_t band, int order, int what, T* d, T* e, T* sigma, cudaEvent_t* marks) {
    const bool wide = m < n;
    const size_t k = std::min(m, n);
    T* x = a;
    if (wide) {
        SVDB_TRY(reserve(c, c->rect_ws, sizeof(T) * m * n));   // grown (never shrunk) when a larger wide matrix arrives
        x = reinterpret_cast<T*>(c->rect_ws.p);
        SVDB_TRY(transpose<T>(c, a, m, n, x));                 // x = A^T: n x m, tall
    }
    if (what & 1) {
        if (order == SVDB200_ORDER_PANEL) SVDB_TRY(stage1_panel_order<T>(c, x, std::max(m, n), k, band));
        else if (order == SVDB200_ORDER_TILE && m == n) SVDB_TRY(stage1_tile_order<T>(c, x, n, band));
        else return SVDB200_E_ARG;
    }
    SVDB_TRY(mark(c, marks, 0));
    if (what & 2) SVDB_TRY(stage2_chase<T>(c, x, k, band, d, e));
    SVDB_TRY(mark(c, marks, 1));
    if (what & 4) SVDB_TRY(bidiag_qr<T>(c, d, e, k, sigma));
    SVDB_TRY(mark(c, marks, 2));
    if (wide) SVDB_TRY(transpose<T>(c, x, n, m, a));
    return mark(c, marks, 3);
}

// Singular values of count m x n matrices (back to back; sigma count x min(m, n)): the batched kernels where they apply,
// otherwise one run_chain per matrix on the handle -- the bytes of svdb200_svdvals_mn_dev_* with the handle's settings
template <typename T>
int batched_svdvals_mn(Ctx* c, T* a, size_t count, size_t m, size_t n, size_t band, T* sigma) {
    if (count == 0) return 0;
    if (batched_in_range(c, m, n, band)) return batched_small<T>(c, a, count, m, n, band, sigma);
    const size_t k = std::min(m, n);
    T* d = reinterpret_cast<T*>(c->d);
    T* e = reinterpret_cast<T*>(c->e);
    for (size_t i = 0; i < count; ++i)
        SVDB_TRY(run_chain<T>(c, a + i * m * n, m, n, band, SVDB200_ORDER_PANEL, 7, d, e, sigma + i * k, nullptr));
    return 0;
}

// One-stage Golub-Kahan bidiagonalisation: the stage-1 panel driver with band 1 in the one-stage order, then d, e (optional)
// read off the result.  All four marks (as run_chain's) follow the reduction: it is all stage 1.
template <typename T>
int onestage_chain(Ctx* c, T* a, size_t n, T* d, T* e, cudaEvent_t* marks) {
    c->onestage = 1;
    const int st = stage1_panel_order<T>(c, a, n, n, 1);
    c->onestage = 0;
    if (st != 0) return st;
    SVDB_TRY(extract_bidiagonal<T>(c, a, n, d, e));
    for (int k = 0; k < 4; ++k) SVDB_TRY(mark(c, marks, k));
    return 0;
}

// Stage 2 from LAPACK upper band storage and, when sigma is given, the singular values of d, e; marks as run_chain's
// (there is no stage 1)
template <typename T>
int packed_chain(Ctx* c, const T* ab, size_t n, size_t band, T* d, T* e, T* sigma, cudaEvent_t* marks) {
    SVDB_TRY(mark(c, marks, 0));
    SVDB_TRY(stage2_chase_packed<T>(c, ab, n, band, d, e));
    SVDB_TRY(mark(c, marks, 1));
    if (sigma) SVDB_TRY(bidiag_qr<T>(c, d, e, n, sigma));
    SVDB_TRY(mark(c, marks, 2));
    return mark(c, marks, 3);
}

// One copy of a host-pointer call; skipped when dst is null (an optional output) or bytes is 0
struct Copy { void* dst; const void* src; size_t bytes; };

// Every single-matrix host-pointer call: the input copies (host -> device), run(marks), which enqueues the device work and
// records the four marks of run_chain, and the output copies (device -> host).  The stream is synchronised once before
// returning, on success and on error, so that no copy from or to the caller's buffers is in flight after the call; a
// failed stage's status wins over a later CUDA error.  The device buffers are the caller's.  svdb200_last_timings gets
// h2d, d2h and the time of every stage whose `what` bit is set (1 stage 1 with the transpose back of a wide matrix,
// 2 stage 2, 4 singular values); a stage whose bit is clear reports 0.  With bit 4 the status of the singular values is
// read back: non-convergence returns SVDB200_E_NOCONV, and the sweep count goes to *sweeps.
template <typename Run>
int host_call(Ctx* c, std::initializer_list<Copy> in, Run&& run, std::initializer_list<Copy> out, int what,
              long long* sweeps = nullptr) {
    cudaStream_t s = c->stream;
    cudaEvent_t* ev = c->ev;
    long long info[3] = {0, 0, 0};
    c->ms_stage1 = c->ms_stage2 = c->ms_qr = c->ms_h2d = c->ms_d2h = 0;
    auto enqueue = [&]() -> int {
        SVDB_CHECK(c, cudaEventRecord(ev[0], s));
        for (const Copy& x : in)
            if (x.dst && x.bytes) SVDB_CHECK(c, cudaMemcpyAsync(x.dst, x.src, x.bytes, cudaMemcpyHostToDevice, s));
        SVDB_CHECK(c, cudaEventRecord(ev[1], s));
        SVDB_TRY(run(ev + 2));                                    // ev[2..5]
        for (const Copy& x : out)
            if (x.dst && x.bytes) SVDB_CHECK(c, cudaMemcpyAsync(x.dst, x.src, x.bytes, cudaMemcpyDeviceToHost, s));
        if (what & 4) SVDB_CHECK(c, cudaMemcpyAsync(info, c->qr_info, sizeof(info), cudaMemcpyDeviceToHost, s));
        SVDB_CHECK(c, cudaEventRecord(ev[6], s));
        return 0;
    };
    const int st = enqueue();
    const cudaError_t se = cudaStreamSynchronize(s);
    if (st != 0) return st;
    if (se != cudaSuccess) return cuda_status(c, se, "cudaStreamSynchronize");
    c->ms_h2d = elapsed(ev[0], ev[1]);
    if (what & 1) c->ms_stage1 = elapsed(ev[1], ev[2]) + elapsed(ev[4], ev[5]);
    if (what & 2) c->ms_stage2 = elapsed(ev[2], ev[3]);
    if (what & 4) c->ms_qr = elapsed(ev[3], ev[4]);
    c->ms_d2h = elapsed(ev[5], ev[6]);
    if (what & 4) {
        if (sweeps) *sweeps = info[0];
        if (info[1] != 0) return SVDB200_E_NOCONV;
    }
    return 0;
}

// Host-pointer dense call (square or m x n) through run_chain, staged through the handle's max_n^2 buffer; d, e, sigma
// (host, each optional) receive min(m, n), min(m, n) - 1 and min(m, n) entries
template <typename T>
int dense_host(Ctx* c, T* a, size_t m, size_t n, size_t band, int order, int what, T* d, T* e, T* sigma) {
    SVDB_TRY(reserve(c, c->a_dev, c->esz * c->max_n * c->max_n));
    T* ad = reinterpret_cast<T*>(c->a_dev.p);
    T* dd = reinterpret_cast<T*>(c->d);
    T* ed = reinterpret_cast<T*>(c->e);
    T* sd = reinterpret_cast<T*>(c->sigma);
    const size_t k = std::min(m, n), bytes = sizeof(T) * m * n;
    return host_call(
        c, {{ad, a, bytes}}, [&](cudaEvent_t* marks) { return run_chain<T>(c, ad, m, n, band, order, what, dd, ed, sd, marks); },
        {{a, ad, bytes}, {d, dd, sizeof(T) * k}, {e, ed, sizeof(T) * (k - 1)}, {sigma, sd, sizeof(T) * k}}, what);
}

// Shape rules of the m x n calls: any orientation, band | min(m, n) (the panel order needs whole panels along the
// shorter side; the longer side is arbitrary)
int check_mn(Ctx* c, size_t m, size_t n, size_t band) {
    const size_t k = std::min(m, n);
    if (k < 2 || band == 0 || k % band != 0) return SVDB200_E_SHAPE;
    if (std::max(m, n) > c->max_n || band > c->band) return SVDB200_E_CAPACITY;
    return 0;
}

size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Shape rules of stage 2 from band storage: those of svdb200_band_to_bidiag_dev_* (no m, band need not divide n)
int check_packed(Ctx* c, size_t n, size_t band) {
    if (n < 2) return SVDB200_E_SHAPE;
    if (band == 0 || band > c->band || n > c->max_n) return SVDB200_E_CAPACITY;
    return 0;
}

}  // namespace

extern "C" {

int svdb200_version(void) { return 100; }

const char* svdb200_strerror(int s) {
    switch (s) {
        case SVDB200_OK: return "ok";
        case SVDB200_E_ARG: return "invalid argument";
        case SVDB200_E_SHAPE: return "shape error: need square n x n with band | n (m x n calls: band | min(m, n) >= 2)";
        case SVDB200_E_CAPACITY: return "exceeds handle capacity or kernel limits";
        case SVDB200_E_NODEVICE: return "no usable CUDA device (there is no CPU fallback)";
        case SVDB200_E_NOCONV: return "QR diagonalisation reached max_iter";
        case SVDB200_E_STATE: return "invalid state";
        default: break;
    }
    if (s >= SVDB200_NCCL_ERR) return "NCCL error";
    if (s >= SVDB200_CUDA_ERR) return cudaGetErrorString((cudaError_t)(s - SVDB200_CUDA_ERR));
    return "unknown status";
}

const char* svdb200_last_error(svdb200_handle h) {
    return h ? reinterpret_cast<Ctx*>(h)->last_error.c_str() : "";
}

int svdb200_create(svdb200_handle* out, int device, size_t max_n, size_t band, int dtype) {
    if (!out || (dtype != SVDB200_F32 && dtype != SVDB200_F64)) return SVDB200_E_ARG;
    if (max_n == 0 || band == 0 || band > (size_t)kMaxBand) return SVDB200_E_SHAPE;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device < 0 || device >= ndev) {
        cudaGetLastError();
        return SVDB200_E_NODEVICE;
    }
    Ctx* c = new (std::nothrow) Ctx();
    if (!c) return SVDB200_E_STATE;
    c->device = device; c->dtype = dtype; c->max_n = max_n; c->band = band;
    c->esz = dtype == SVDB200_F32 ? 4 : 8;
#define SVDB_CREATE_CHECK(expr)                                         \
    do {                                                                \
        cudaError_t _e = (expr);                                        \
        if (_e != cudaSuccess) {                                        \
            int _s = cuda_status(c, _e, #expr);                         \
            svdb200_destroy(reinterpret_cast<svdb200_handle>(c));       \
            return _s;                                                  \
        }                                                               \
    } while (0)
    SVDB_CREATE_CHECK(cudaSetDevice(device));
    cudaDeviceProp prop;
    SVDB_CREATE_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) { delete c; return SVDB200_E_NODEVICE; }   // sm_100a code only
    c->num_sms = prop.multiProcessorCount;
    c->coop_supported = prop.cooperativeLaunch;
    SVDB_CREATE_CHECK(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    for (auto& e : c->ev) SVDB_CREATE_CHECK(cudaEventCreate(&e));
    for (auto& e : c->pev) SVDB_CREATE_CHECK(cudaEventCreate(&e));
    const size_t es = c->esz, nb = round_up(max_n, 128) + 128;
    // a_dev (max_n^2 staging for the host-pointer entry points) is allocated on first use
    SVDB_CREATE_CHECK(cudaMalloc(&c->v, es * nb * band));
    SVDB_CREATE_CHECK(cudaMalloc(&c->v2, es * nb * band));
    SVDB_CREATE_CHECK(cudaMalloc(&c->vb, es * nb * band));
    SVDB_CREATE_CHECK(cudaMalloc(&c->v2b, es * nb * band));
    {
        int lo = 0, hi = 0;
        SVDB_CREATE_CHECK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        SVDB_CREATE_CHECK(cudaStreamCreateWithPriority(&c->aux_stream, cudaStreamNonBlocking, hi));
        for (auto& e : c->lev) SVDB_CREATE_CHECK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    SVDB_CREATE_CHECK(cudaMalloc(&c->w, es * nb * band));
    c->wpart_elems = 16 * nb * band;
    if (c->wpart_elems < 4 * nb) c->wpart_elems = 4 * nb;
    SVDB_CREATE_CHECK(cudaMalloc(&c->wpart, es * c->wpart_elems));
    SVDB_CREATE_CHECK(cudaMalloc(&c->s, es * band * band));
    SVDB_CREATE_CHECK(cudaMalloc(&c->tau, es * band));
    SVDB_CREATE_CHECK(cudaMalloc(&c->red, es * 2 * (kMaxPanelCtas + 1) * (2 * band + 8)));
    SVDB_CREATE_CHECK(cudaMemset(c->red, 0, es * 2 * (kMaxPanelCtas + 1) * (2 * band + 8)));   // flag-stamped words start unset
    SVDB_CREATE_CHECK(cudaMalloc(&c->red2, 512 * 1024));
    SVDB_CREATE_CHECK(cudaMemset(c->red2, 0, 512 * 1024));
    SVDB_CREATE_CHECK(cudaMalloc(&c->chol_ws, 1 << 20));
    SVDB_CREATE_CHECK(cudaMemset(c->chol_ws, 0, 1 << 20));
    SVDB_CREATE_CHECK(cudaMalloc(&c->bar, 64));
    SVDB_CREATE_CHECK(cudaMemset(c->bar, 0, 64));
    SVDB_CREATE_CHECK(cudaMalloc(&c->prog, sizeof(int) * (max_n + 8)));
    SVDB_CREATE_CHECK(cudaMalloc(&c->d, es * (max_n + 8)));
    SVDB_CREATE_CHECK(cudaMalloc(&c->e, es * (max_n + 8)));
    SVDB_CREATE_CHECK(cudaMalloc(&c->sigma, es * (max_n + 8)));
    SVDB_CREATE_CHECK(cudaMalloc(&c->qr_info, 64));
    SVDB_CREATE_CHECK(cudaMemset(c->qr_info, 0, 64));
    SVDB_CREATE_CHECK(cudaMalloc(&c->tileq, es * (max_n / band + 2) * 4 * band * band));
    SVDB_CREATE_CHECK(cudaMalloc(&c->tilestate, es * (4 * band * band + 64)));
#undef SVDB_CREATE_CHECK
    *out = reinterpret_cast<svdb200_handle>(c);
    return 0;
}

int svdb200_destroy(svdb200_handle h) {
    if (!h) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    cudaSetDevice(c->device);
    if (c->own_stream) cudaStreamSynchronize(c->own_stream);
    for (auto& ph : c->pool) if (ph) svdb200_destroy(reinterpret_cast<svdb200_handle>(ph));
    c->pool.clear();
    void* ptrs[] = {c->v, c->v2, c->vb, c->v2b, c->w, c->wpart, c->s, c->tau, c->red, c->red2, c->chol_ws, c->bar, c->prog,
                    c->d, c->e, c->sigma, c->qr_info, c->tileq, c->tilestate, c->de2};   // the DevBuf members free themselves with c
    for (int k = 1; k < 2 * Ctx::kLanes; ++k) if (c->a_stage[k]) cudaFree(c->a_stage[k]);
    for (int l = 0; l < Ctx::kLanes; ++l) if (c->s1ctx[l]) svdb200_destroy(reinterpret_cast<svdb200_handle>(c->s1ctx[l]));
    for (int l = 1; l < Ctx::kLanes; ++l) if (c->s2_prog[l]) cudaFree(c->s2_prog[l]);
    for (void* p : ptrs) if (p) cudaFree(p);
    for (auto& e : c->ev) if (e) cudaEventDestroy(e);
    for (auto& e : c->pev) if (e) cudaEventDestroy(e);
    for (auto& e : c->lev) if (e) cudaEventDestroy(e);
    for (auto& e : c->s2ev) if (e) cudaEventDestroy(e);
    for (auto& st2 : c->s2_stream) if (st2) cudaStreamDestroy(st2);
    if (c->aux_stream) cudaStreamDestroy(c->aux_stream);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return 0;
}

int svdb200_set_stream(svdb200_handle h, void* stream) {
    if (!h) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    c->stream = stream ? reinterpret_cast<cudaStream_t>(stream) : c->own_stream;
    return 0;
}

int svdb200_synchronize(svdb200_handle h) {
    if (!h) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    SVDB_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

#define SVDB_ENTER(T)                                    \
    Ctx* c = reinterpret_cast<Ctx*>(h);                  \
    if (!c) return SVDB200_E_ARG;                        \
    if (c->dtype != dtype_of<T>()) return SVDB200_E_ARG; \
    SVDB_CHECK(c, cudaSetDevice(c->device));

#define SVDB_DEFINE_TYPED(T, S)                                                                                          \
    int svdb200_dense_to_band_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, int order) {                  \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_square(c, m, n, band, dtype_of<T>()));                                                            \
        return dense_host<T>(c, a, n, n, band, order, 1, nullptr, nullptr, nullptr);                                     \
    }                                                                                                                    \
    int svdb200_dense_to_band_dev_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, int order) {              \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_square(c, m, n, band, dtype_of<T>()));                                                            \
        return run_chain<T>(c, a, n, n, band, order, 1, nullptr, nullptr, nullptr, nullptr);                             \
    }                                                                                                                    \
    int svdb200_band_to_bidiag_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, T* d, T* e) {                \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_square(c, m, n, 1, dtype_of<T>()));                                                               \
        if (band == 0 || band > c->band) return SVDB200_E_CAPACITY;                                                      \
        return dense_host<T>(c, a, n, n, band, SVDB200_ORDER_PANEL, 2, d, e, nullptr);                                   \
    }                                                                                                                    \
    int svdb200_band_to_bidiag_dev_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, T* d, T* e) {            \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_square(c, m, n, 1, dtype_of<T>()));                                                               \
        if (band == 0 || band > c->band) return SVDB200_E_CAPACITY;                                                      \
        return run_chain<T>(c, a, n, n, band, SVDB200_ORDER_PANEL, 2, d, e, nullptr, nullptr);                           \
    }                                                                                                                    \
    int svdb200_band_to_bidiag_packed_##S(svdb200_handle h, const T* ab, size_t n, size_t band, T* d, T* e) {            \
        SVDB_ENTER(T)                                                                                                    \
        if (!ab) return SVDB200_E_ARG;                                                                                   \
        SVDB_TRY(check_packed(c, n, band));                                                                              \
        DevBuf abd;                                        /* per call: the handle does not keep n (band + 1) elements */ \
        SVDB_TRY(reserve(c, abd, sizeof(T) * n * (band + 1)));                                                           \
        T* dd = reinterpret_cast<T*>(c->d);                                                                              \
        T* ed = reinterpret_cast<T*>(c->e);                                                                              \
        return host_call(c, {{abd.p, ab, abd.bytes}},                                                                    \
                         [&](cudaEvent_t* mk) { return packed_chain<T>(c, (const T*)abd.p, n, band, dd, ed, nullptr, mk); }, \
                         {{d, dd, sizeof(T) * n}, {e, ed, sizeof(T) * (n - 1)}}, 2);                                     \
    }                                                                                                                    \
    int svdb200_band_to_bidiag_packed_dev_##S(svdb200_handle h, const T* ab, size_t n, size_t band, T* d, T* e) {        \
        SVDB_ENTER(T)                                                                                                    \
        if (!ab) return SVDB200_E_ARG;                                                                                   \
        SVDB_TRY(check_packed(c, n, band));                                                                              \
        return stage2_chase_packed<T>(c, ab, n, band, d, e);                                                             \
    }                                                                                                                    \
    int svdb200_band_svdvals_packed_##S(svdb200_handle h, const T* ab, size_t n, size_t band, T* sigma) {                \
        SVDB_ENTER(T)                                                                                                    \
        if (!ab || !sigma) return SVDB200_E_ARG;                                                                         \
        SVDB_TRY(check_packed(c, n, band));                                                                              \
        DevBuf abd;                                                                                                      \
        SVDB_TRY(reserve(c, abd, sizeof(T) * n * (band + 1)));                                                           \
        T* dd = reinterpret_cast<T*>(c->d);                                                                              \
        T* ed = reinterpret_cast<T*>(c->e);                                                                              \
        T* sd = reinterpret_cast<T*>(c->sigma);                                                                          \
        return host_call(c, {{abd.p, ab, abd.bytes}},                                                                    \
                         [&](cudaEvent_t* mk) { return packed_chain<T>(c, (const T*)abd.p, n, band, dd, ed, sd, mk); },  \
                         {{sigma, sd, sizeof(T) * n}}, 6);                                                               \
    }                                                                                                                    \
    int svdb200_band_svdvals_packed_dev_##S(svdb200_handle h, const T* ab, size_t n, size_t band, T* sigma) {            \
        SVDB_ENTER(T)                                                                                                    \
        if (!ab || !sigma) return SVDB200_E_ARG;                                                                         \
        SVDB_TRY(check_packed(c, n, band));                                                                              \
        return packed_chain<T>(c, ab, n, band, reinterpret_cast<T*>(c->d), reinterpret_cast<T*>(c->e), sigma, nullptr);  \
    }                                                                                                                    \
    int svdb200_bidiag_qr_##S(svdb200_handle h, const T* d, const T* e, size_t n, T* sigma, long long* sweeps) {         \
        SVDB_ENTER(T)                                                                                                    \
        if (!d || !e || !sigma) return SVDB200_E_ARG;                                                                    \
        if (n < 2) return SVDB200_E_SHAPE;                                                                               \
        if (n > c->max_n) return SVDB200_E_CAPACITY;                                                                     \
        T* dd = reinterpret_cast<T*>(c->d);                                                                              \
        T* ed = reinterpret_cast<T*>(c->e);                                                                              \
        T* sd = reinterpret_cast<T*>(c->sigma);                                                                          \
        return host_call(c, {{dd, d, sizeof(T) * n}, {ed, e, sizeof(T) * (n - 1)}},                                      \
                         [&](cudaEvent_t* mk) { return run_chain<T>(c, (T*)nullptr, n, n, 1, SVDB200_ORDER_PANEL, 4, dd, ed, sd, mk); }, \
                         {{sigma, sd, sizeof(T) * n}}, 4, sweeps);                                                       \
    }                                                                                                                    \
    int svdb200_bidiag_qr_dev_##S(svdb200_handle h, T* d, T* e, size_t n, T* sigma) {                                    \
        SVDB_ENTER(T)                                                                                                    \
        if (!d || !e || !sigma) return SVDB200_E_ARG;                                                                    \
        if (n < 2) return SVDB200_E_SHAPE;                                                                               \
        return bidiag_qr<T>(c, d, e, n, sigma);                                                                          \
    }                                                                                                                    \
    int svdb200_bidiagonalize_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, int order, T* d, T* e) {      \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_square(c, m, n, band, dtype_of<T>()));                                                            \
        return dense_host<T>(c, a, n, n, band, order, 3, d, e, nullptr);                                                 \
    }                                                                                                                    \
    int svdb200_bidiagonalize_dev_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, int order, T* d, T* e) {  \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_square(c, m, n, band, dtype_of<T>()));                                                            \
        return run_chain<T>(c, a, n, n, band, order, 3, d, e, nullptr, nullptr);                                         \
    }                                                                                                                    \
    int svdb200_bidiagonalize_onestage_dev_##S(svdb200_handle h, T* a, size_t m, size_t n, T* d, T* e) {                 \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_square(c, m, n, 1, dtype_of<T>()));                                                               \
        return onestage_chain<T>(c, a, n, d, e, nullptr);                                                                \
    }                                                                                                                    \
    int svdb200_bidiagonalize_onestage_##S(svdb200_handle h, T* a, size_t m, size_t n, T* d, T* e) {                     \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_square(c, m, n, 1, dtype_of<T>()));                                                               \
        SVDB_TRY(reserve(c, c->a_dev, c->esz * c->max_n * c->max_n));                                                    \
        T* ad = reinterpret_cast<T*>(c->a_dev.p);                                                                        \
        T* dd = reinterpret_cast<T*>(c->d);                                                                              \
        T* ed = reinterpret_cast<T*>(c->e);                                                                              \
        return host_call(c, {{ad, a, sizeof(T) * n * n}}, [&](cudaEvent_t* mk) { return onestage_chain<T>(c, ad, n, dd, ed, mk); }, \
                         {{a, ad, sizeof(T) * n * n}, {d, dd, sizeof(T) * n}, {e, ed, sizeof(T) * (n - 1)}}, 1);         \
    }                                                                                                                    \
    int svdb200_bidiagonalize_many_dev_##S(svdb200_handle h, size_t count, T* const* a, const size_t* n, size_t band,    \
                                           int order, T* const* d, T* const* e) {                                        \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !n) return SVDB200_E_ARG;                                                                              \
        for (size_t i = 0; i < count; ++i) {                                                                             \
            if (!a[i]) return SVDB200_E_ARG;                                                                             \
            SVDB_TRY(check_square(c, n[i], n[i], band, dtype_of<T>()));                                                  \
        }                                                                                                                \
        return bidiagonalize_many_dev<T>(c, count, a, n, band, order, d, e);                                             \
    }                                                                                                                    \
    int svdb200_bidiagonalize_many_##S(svdb200_handle h, size_t count, T* const* a, const size_t* n, size_t band,        \
                                       int order, T* const* d, T* const* e) {                                            \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !n) return SVDB200_E_ARG;                                                                              \
        for (size_t i = 0; i < count; ++i) {                                                                             \
            if (!a[i]) return SVDB200_E_ARG;                                                                             \
            SVDB_TRY(check_square(c, n[i], n[i], band, dtype_of<T>()));                                                  \
        }                                                                                                                \
        return bidiagonalize_many_host<T>(c, count, a, n, band, order, d, e);                                            \
    }                                                                                                                    \
    int svdb200_svdvals_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, int order, T* sigma) {              \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !sigma) return SVDB200_E_ARG;                                                                          \
        SVDB_TRY(check_square(c, m, n, band, dtype_of<T>()));                                                            \
        return dense_host<T>(c, a, n, n, band, order, 7, nullptr, nullptr, sigma);                                       \
    }                                                                                                                    \
    int svdb200_svdvals_dev_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, int order, T* sigma) {          \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !sigma) return SVDB200_E_ARG;                                                                          \
        SVDB_TRY(check_square(c, m, n, band, dtype_of<T>()));                                                            \
        return run_chain<T>(c, a, n, n, band, order, 7, reinterpret_cast<T*>(c->d), reinterpret_cast<T*>(c->e), sigma, nullptr); \
    }                                                                                                                    \
    int svdb200_dense_to_band_mn_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band) {                          \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        return dense_host<T>(c, a, m, n, band, SVDB200_ORDER_PANEL, 1, nullptr, nullptr, nullptr);                       \
    }                                                                                                                    \
    int svdb200_dense_to_band_mn_dev_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band) {                      \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        return run_chain<T>(c, a, m, n, band, SVDB200_ORDER_PANEL, 1, nullptr, nullptr, nullptr, nullptr);               \
    }                                                                                                                    \
    int svdb200_bidiagonalize_mn_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, T* d, T* e) {              \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !d || !e) return SVDB200_E_ARG;                                                                        \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        return dense_host<T>(c, a, m, n, band, SVDB200_ORDER_PANEL, 3, d, e, nullptr);                                   \
    }                                                                                                                    \
    int svdb200_bidiagonalize_mn_dev_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, T* d, T* e) {          \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !d || !e) return SVDB200_E_ARG;                                                                        \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        return run_chain<T>(c, a, m, n, band, SVDB200_ORDER_PANEL, 3, d, e, nullptr, nullptr);                           \
    }                                                                                                                    \
    int svdb200_svdvals_mn_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, T* sigma) {                      \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !sigma) return SVDB200_E_ARG;                                                                          \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        return dense_host<T>(c, a, m, n, band, SVDB200_ORDER_PANEL, 7, nullptr, nullptr, sigma);                         \
    }                                                                                                                    \
    int svdb200_svdvals_mn_dev_##S(svdb200_handle h, T* a, size_t m, size_t n, size_t band, T* sigma) {                  \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !sigma) return SVDB200_E_ARG;                                                                          \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        return run_chain<T>(c, a, m, n, band, SVDB200_ORDER_PANEL, 7, reinterpret_cast<T*>(c->d), reinterpret_cast<T*>(c->e), sigma, nullptr); \
    }                                                                                                                    \
    int svdb200_svdvals_batched_dev_##S(svdb200_handle h, T* a, size_t count, size_t n, size_t band, T* sigma) {         \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !sigma) return SVDB200_E_ARG;                                                                          \
        SVDB_TRY(check_square(c, n, n, band, dtype_of<T>()));                                                            \
        return batched_svdvals<T>(c, a, count, n, band, sigma);                                                          \
    }                                                                                                                    \
    int svdb200_svdvals_batched_##S(svdb200_handle h, T* a, size_t count, size_t n, size_t band, T* sigma) {             \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !sigma) return SVDB200_E_ARG;                                                                          \
        SVDB_TRY(check_square(c, n, n, band, dtype_of<T>()));                                                            \
        DevBuf ad, sd;                                     /* per call: the handle does not keep count n^2 elements */   \
        SVDB_TRY(reserve(c, ad, sizeof(T) * count * n * n));                                                             \
        SVDB_TRY(reserve(c, sd, sizeof(T) * count * n));                                                                 \
        /* the driver interleaves the stages of different matrices: what = 0, only the copies are timed */               \
        return host_call(c, {{ad.p, a, ad.bytes}},                                                                       \
                         [&](cudaEvent_t* mk) {                                                                          \
                             SVDB_TRY(batched_svdvals<T>(c, (T*)ad.p, count, n, band, (T*)sd.p));                        \
                             for (int k = 0; k < 4; ++k) SVDB_TRY(mark(c, mk, k));                                       \
                             return 0;                                                                                   \
                         },                                                                                              \
                         {{sigma, sd.p, sd.bytes}, {a, ad.p, ad.bytes}}, 0);                                             \
    }                                                                                                                    \
    int svdb200_chain_batched_dev_##S(svdb200_handle h, T* a, size_t count, size_t n, size_t band, int what, T* d, T* e, T* sigma) { \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || what <= 0 || what > 7 || ((what & 4) && !sigma)) return SVDB200_E_ARG;                                 \
        SVDB_TRY(check_square(c, n, n, band, dtype_of<T>()));                                                            \
        return batched_chain<T>(c, a, count, n, n, band, what, d, e, sigma);                                             \
    }                                                                                                                    \
    int svdb200_svdvals_batched_mn_dev_##S(svdb200_handle h, T* a, size_t count, size_t m, size_t n, size_t band, T* sigma) { \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !sigma) return SVDB200_E_ARG;                                                                          \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        return batched_svdvals_mn<T>(c, a, count, m, n, band, sigma);                                                    \
    }                                                                                                                    \
    int svdb200_svdvals_batched_mn_##S(svdb200_handle h, T* a, size_t count, size_t m, size_t n, size_t band, T* sigma) { \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !sigma) return SVDB200_E_ARG;                                                                          \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        DevBuf ad, sd;                                     /* per call, as svdb200_svdvals_batched_* */                  \
        SVDB_TRY(reserve(c, ad, sizeof(T) * count * m * n));                                                             \
        SVDB_TRY(reserve(c, sd, sizeof(T) * count * std::min(m, n)));                                                    \
        return host_call(c, {{ad.p, a, ad.bytes}},                                                                       \
                         [&](cudaEvent_t* mk) {                                                                          \
                             SVDB_TRY(batched_svdvals_mn<T>(c, (T*)ad.p, count, m, n, band, (T*)sd.p));                  \
                             for (int k = 0; k < 4; ++k) SVDB_TRY(mark(c, mk, k));                                       \
                             return 0;                                                                                   \
                         },                                                                                              \
                         {{sigma, sd.p, sd.bytes}, {a, ad.p, ad.bytes}}, 0);                                             \
    }                                                                                                                    \
    int svdb200_chain_batched_mn_dev_##S(svdb200_handle h, T* a, size_t count, size_t m, size_t n, size_t band, int what, \
                                         T* d, T* e, T* sigma) {                                                         \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || what <= 0 || what > 7 || ((what & 4) && !sigma)) return SVDB200_E_ARG;                                 \
        SVDB_TRY(check_mn(c, m, n, band));                                                                               \
        return batched_chain<T>(c, a, count, m, n, band, what, d, e, sigma);                                             \
    }                                                                                                                    \
    int svdb200_panel_factor_dev_##S(svdb200_handle h, T* a, size_t lda, size_t m, size_t b, int trans, T* v, T* v2) {   \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !v || !v2 || m == 0 || b == 0 || b > c->band || m > c->max_n) return SVDB200_E_ARG;                    \
        return trans ? launch_panel_public<T, true>(c, a, lda, (int)m, (int)b, v, v2, c->stream)                         \
                     : launch_panel_public<T, false>(c, a, lda, (int)m, (int)b, v, v2, c->stream);                       \
    }                                                                                                                    \
    int svdb200_mse_##S(svdb200_handle h, const T* a, const T* b, size_t n, size_t band, T* out) {                       \
        SVDB_ENTER(T)                                                                                                    \
        if (!a || !b || !out || n == 0 || band == 0) return SVDB200_E_ARG;                                               \
        if (n > c->max_n) return SVDB200_E_CAPACITY;                                                                     \
        SVDB_TRY(reserve(c, c->a_dev, c->esz * c->max_n * c->max_n));                                                    \
        T* ad = reinterpret_cast<T*>(c->a_dev.p);                                                                        \
        DevBuf bd;                                                                                                       \
        SVDB_TRY(reserve(c, bd, sizeof(T) * n * n));                                                                     \
        SVDB_CHECK(c, cudaMemcpyAsync(ad, a, sizeof(T) * n * n, cudaMemcpyHostToDevice, c->stream));                     \
        SVDB_CHECK(c, cudaMemcpyAsync(bd.p, b, sizeof(T) * n * n, cudaMemcpyHostToDevice, c->stream));                   \
        return mse_metric<T>(c, ad, (const T*)bd.p, n, band, out);                                                       \
    }                                                                                                                    \
    int svdb200_fill_uniform_dev_##S(svdb200_handle h, T* a, size_t count, unsigned long long seed, double lo, double hi) { \
        SVDB_ENTER(T)                                                                                                    \
        if (!a) return SVDB200_E_ARG;                                                                                    \
        return fill_uniform<T>(c, a, count, seed, lo, hi);                                                               \
    }                                                                                                                    \
    int svdb200_gemm_tn_dev_##S(svdb200_handle h, const T* v, const T* cm, size_t ldc, size_t mrows, size_t ncols, size_t b, T* w) { \
        SVDB_ENTER(T)                                                                                                    \
        if (!v || !cm || !w) return SVDB200_E_ARG;                                                                       \
        return gemm_tn<T>(c, v, cm, ldc, mrows, ncols, b, w);                                                            \
    }                                                                                                                    \
    int svdb200_rank_update_dev_##S(svdb200_handle h, T* cm, size_t ldc, size_t mrows, size_t ncols, size_t b, const T* p, const T* q, size_t ldq) { \
        SVDB_ENTER(T)                                                                                                    \
        if (!cm || !p || !q) return SVDB200_E_ARG;                                                                       \
        return rank_update<T>(c, cm, ldc, mrows, ncols, b, p, q, ldq);                                                   \
    }                                                                                                                    \
    int svdb200_gemm_nn_dev_##S(svdb200_handle h, const T* cm, size_t ldc, size_t mrows, size_t ncols, size_t b, const T* ut, T* w) { \
        SVDB_ENTER(T)                                                                                                    \
        if (!cm || !ut || !w) return SVDB200_E_ARG;                                                                      \
        return gemm_nn<T>(c, cm, ldc, mrows, ncols, b, ut, w);                                                           \
    }

SVDB_DEFINE_TYPED(float, f32)
SVDB_DEFINE_TYPED(double, f64)

int svdb200_last_timings(svdb200_handle h, double* s1, double* s2, double* qr, double* h2d, double* d2h) {
    if (!h) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    if (s1) *s1 = c->ms_stage1;
    if (s2) *s2 = c->ms_stage2;
    if (qr) *qr = c->ms_qr;
    if (h2d) *h2d = c->ms_h2d;
    if (d2h) *d2h = c->ms_d2h;
    return 0;
}

int svdb200_set_band_capture(svdb200_handle h, void* const* dev_bufs, size_t count) {
    if (!h || (count && !dev_bufs)) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    c->band_capture.assign(dev_bufs, dev_bufs + count);
    return 0;
}

int svdb200_set_profile(svdb200_handle h, int on) {
    if (!h) return SVDB200_E_ARG;
    reinterpret_cast<Ctx*>(h)->profile = on ? 1 : 0;
    return 0;
}
int svdb200_reset_profile(svdb200_handle h) {
    if (!h) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    for (int i = 0; i < SVDB200_PROFILE_CLASSES; ++i) { c->prof_ms[i] = 0; c->prof_work[i] = 0; c->prof_launches[i] = 0; }
    return 0;
}
int svdb200_get_profile(svdb200_handle h, double* ms, double* work, long long* launches) {
    if (!h) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    for (int i = 0; i < SVDB200_PROFILE_CLASSES; ++i) {
        if (ms) ms[i] = c->prof_ms[i];
        if (work) work[i] = c->prof_work[i];
        if (launches) launches[i] = c->prof_launches[i];
    }
    return 0;
}

long long svdb200_launch_count(svdb200_handle h) { return h ? reinterpret_cast<Ctx*>(h)->launches : -1; }

int svdb200_probe_peak(svdb200_handle h, int kind, double* tflops) {
    if (!h || !tflops) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    SVDB_CHECK(c, cudaSetDevice(c->device));
    if (kind == 4) return probe_tc05_tf32(c, tflops);
    return probe_peak(c, kind, tflops);
}

int svdb200_debug_stage2_timing(long long* out16) { return out16 ? stage2_debug_read(out16) : SVDB200_E_ARG; }
int svdb200_debug_stage2_fast_timing(long long* out24) { return out24 ? stage2_fast_debug_read(out24) : SVDB200_E_ARG; }
int svdb200_debug_panel_timing(long long* out16) { return out16 ? panel_reg_debug_read(out16) : SVDB200_E_ARG; }
int svdb200_debug_panel_blk_timing(long long* out16) { return out16 ? panel_blk_debug_read(out16) : SVDB200_E_ARG; }
int svdb200_list_plan(int lanes, size_t count, const size_t* n, size_t* order_out, int* chain_out) {
    constexpr int kMaxPlanLanes = 4;                                  // plans for more chains than the pipeline runs (Ctx::kLanes)
    if (lanes < 1 || lanes > kMaxPlanLanes || (count > 0 && (!n || !order_out || !chain_out))) return SVDB200_E_ARG;
    const ListPlan pl = plan_list(lanes, count, n);
    for (size_t j = 0; j < count; ++j) { order_out[j] = pl.order[j]; chain_out[j] = pl.chain[j]; }
    return 0;
}
int svdb200_debug_panel_chol_timing(long long* out16) { return out16 ? panel_chol_debug_read(out16) : SVDB200_E_ARG; }
int svdb200_set_panel_kernel(svdb200_handle h, int blocked) {
    if (!h || blocked < 0 || blocked > 2) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    c->cfg.panel_blk = blocked >= 1;
    c->cfg.panel_chol = blocked == 2;
    return 0;
}
int svdb200_set_chol_guard(svdb200_handle h, double guard) {
    if (!h || !(guard >= 0.0)) return SVDB200_E_ARG;
    reinterpret_cast<Ctx*>(h)->cfg.chol_guard = guard;
    return 0;
}
int svdb200_chol_fallback_count(svdb200_handle h, long long* count) {
    if (!h || !count) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    SVDB_CHECK(c, cudaSetDevice(c->device));
    SVDB_CHECK(c, cudaStreamSynchronize(c->stream));
    if (c->aux_stream) SVDB_CHECK(c, cudaStreamSynchronize(c->aux_stream));
    int st[2] = {0, 0};
    SVDB_CHECK(c, cudaMemcpy(st, c->chol_ws, sizeof(st), cudaMemcpyDeviceToHost));
    *count = st[1];
    return 0;
}

int svdb200_set_stage2_schedule(svdb200_handle h, int mode) {
    if (!h || mode < 0 || mode > 1) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    c->cfg.stage2_complete = mode;
    return 0;
}

int svdb200_set_qr_method(svdb200_handle h, int method, size_t auto_limit) {
    if (!h || method < 0 || method > 3) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    c->cfg.qr_method = method;
    if (auto_limit > 0) c->cfg.qr_auto_limit = auto_limit;
    return 0;
}

int svdb200_tc05_selftest(svdb200_handle h, int a_mn, int b_mn, const float* a, const float* b, float* out, float* dump) {
    if (!h || !a || !b || !out || !dump) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    SVDB_CHECK(c, cudaSetDevice(c->device));
    return tc05_selftest(c, a_mn, b_mn, a, b, out, dump);
}

int svdb200_set_tc05(svdb200_handle h, int mode, long long min_elems) {
    if (!h || mode < 0 || mode > 2) return SVDB200_E_ARG;
    Ctx* c = reinterpret_cast<Ctx*>(h);
    c->cfg.use_tc05 = mode;
    if (min_elems > 0) c->cfg.tc05_min_elems = min_elems;
    return 0;
}

}  // extern "C"

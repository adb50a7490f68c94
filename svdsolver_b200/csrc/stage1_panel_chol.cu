// Stage-1 panel factorisation WITHOUT a per-column (or per-sub-panel) exchange: Cholesky-QR with reconstructed Householder
// vectors.  Same outputs and sign convention as the other panel kernels (stage1_panel.cu, stage1_panel_reg.cu,
// stage1_panel_blk.cu; reference: qr / lq of svd_parallel.h:133-226 with householder of svd_serial.h:194-201,
// H x = -sign(x0) ||x|| e1): R (or L) in A with exact zeros below the diagonal, V with explicit unit diagonal,
// V2 = V S^T with S = -T of the compact-WY form (svd_parallel.h:97-113).
//
// The Householder QR factorisation of a full-rank panel is unique once the sign rule is fixed, so it can be obtained from
// ANY QR factorisation (Ballard, Demmel, Grigori, Jacquelin, Nguyen, Solomonik: "Reconstructing Householder vectors from
// tall-skinny QR", 2014).  With P = [A1; A2] (A1 = top b x b block):
//     G  = P^T P                                    one pass over the panel, DMMA (mma.sync.m8n8k4.f64), exact products of
//                                                   the elements in double, deterministic reduction      -- chol_gram_kernel
//                                                   (the distributed QR panel sums the rows below A1 and adds A1^T A1 later)
//     G  = R^T R                                    Cholesky (R upper, positive diagonal), P = Q R
//     A1 - S R = L U~                               LU without pivoting of (Q1 - S) R; s_i = -sign(pivot_i) is chosen while
//                                                   eliminating (|pivot| >= R_ii: no growth), U~ = U R
//     Y  = [L; A2 U~^-1]                            the Householder vectors;  R_hh = S R
//     T^-1 = diag(Y^T Y)/2 + striu(Y^T Y)           = -L^T S U^-1 because Q = P R^-1 is orthonormal (the paper's T = -U S L^-T);
//                                                   U^-1 = R M1, M1 = U~^-1                  (all b x b, in double)
//     V2 = -Y T^T = [-L T^T ; A2 M2], M2 = -M1 T^T                                           -- chol_algebra_kernel (1 CTA)
//     [Y2 | V2_2] = A2 [M1 | M2]                    second pass, rows independent             -- chol_apply_kernel
// Two passes over the panel + O(b^3) work on one SM instead of b (or b/8) grid-wide exchanges: the time no longer grows
// with the number of CTAs that must agree per column, and no CTA ever waits for another one (safe beside resident
// stage-2 grids and persistent update kernels).
//
// Accuracy: Cholesky-QR squares the condition number of the PANEL (not of the matrix): relative error ~ eps_double *
// kappa(P)^2 in R and eps_T * kappa(P) in Y.  The algebra kernel checks the pivot ratios min_j R_jj^2 / G_jj; below
// `guard` it leaves everything untouched and raises status[0], which turns the fallback launch that follows in the
// stream (one of the exchange-based kernels, gated on the same word) from a no-op into the real factorisation.
#include <algorithm>
#include <type_traits>
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace svdb200 {
namespace {

#ifndef SVDB_PANEL_TIMING
#define SVDB_PANEL_TIMING 0
#endif
__device__ long long g_chol_dbg[16];
#define CHOL_TICK(k)                                          \
    do {                                                      \
        if (SVDB_PANEL_TIMING && threadIdx.x == 0) {          \
            long long _t = clock64();                         \
            g_chol_dbg[k] += _t - tick;                       \
            tick = _t;                                        \
        }                                                     \
    } while (0)

constexpr int kGramThreads = 256, kGramWarps = 8, kGramCluster = 8;
constexpr int kAlgThreads = 512;
constexpr int kApplyThreads = 256, kApplyRows = 64, kApplyPad = 4;

__device__ __forceinline__ void dmma884(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
}

// panel element (r, c): QR panels A[r*lda + c], LQ panels (kTrans) A[c*lda + r]
template <typename T, bool kTrans>
__device__ __forceinline__ size_t pidx(size_t lda, int r, int c) {
    return kTrans ? (size_t)c * lda + r : (size_t)r * lda + c;
}

// ---- pass 1: partial Gram matrices of the rows [row0, m) ----------------------------------------------------------------
// G2 = sum_r p_r^T p_r is computed tile by tile (8 x 8, upper triangle of tiles) with DMMA: for a k-step of 4 rows the A
// fragment of tile row ti and the B fragment of tile column tj are the SAME register (lane l holds P[r + l%4][8t + l/4]).
// Tile-packed output: part[cluster][tile idx][64].
template <typename T, bool kTrans, int NB8>
__global__ void __launch_bounds__(kGramThreads, 1)
chol_gram_kernel(const T* __restrict__ A, size_t lda, int row0, int m, int rows_per_cta, int cs, double* __restrict__ part) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int NT = NB8 * (NB8 + 1) / 2, NE = NT * 64;
    double* sm = reinterpret_cast<double*>(smem_raw);      // kGramWarps x NE
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int kq = lane & 3, cq = lane >> 2;
    const int rbeg = row0 + blockIdx.x * rows_per_cta, rend = min(m, rbeg + rows_per_cta);
    double acc[NT][2];
#pragma unroll
    for (int i = 0; i < NT; ++i) { acc[i][0] = 0.0; acc[i][1] = 0.0; }
    for (int r = rbeg + w * 8; r < rend; r += kGramWarps * 8) {
        double f0[NB8], f1[NB8];
        const int ra = r + kq, rb = r + 4 + kq;
#pragma unroll
        for (int t = 0; t < NB8; ++t) {
            const int col = 8 * t + cq;
            f0[t] = ra < rend ? (double)A[pidx<T, kTrans>(lda, ra, col)] : 0.0;
            f1[t] = rb < rend ? (double)A[pidx<T, kTrans>(lda, rb, col)] : 0.0;
        }
        int idx = 0;
#pragma unroll
        for (int ti = 0; ti < NB8; ++ti)
#pragma unroll
            for (int tj = ti; tj < NB8; ++tj) { dmma884(acc[idx][0], acc[idx][1], f0[ti], f0[tj]); ++idx; }
        idx = 0;
#pragma unroll
        for (int ti = 0; ti < NB8; ++ti)
#pragma unroll
            for (int tj = ti; tj < NB8; ++tj) { dmma884(acc[idx][0], acc[idx][1], f1[ti], f1[tj]); ++idx; }
    }
    // the 8 warps' tiles: element (lane/4, 2*(lane%4) + s) of tile idx sits at idx*64 + 2*lane + s
#pragma unroll
    for (int i = 0; i < NT; ++i)
        *reinterpret_cast<double2*>(sm + (size_t)w * NE + i * 64 + 2 * lane) = make_double2(acc[i][0], acc[i][1]);
    __syncthreads();
    for (int e = tid; e < NE; e += kGramThreads) {
        double s = sm[e];
#pragma unroll
        for (int q = 1; q < kGramWarps; ++q) s += sm[(size_t)q * NE + e];
        sm[e] = s;
    }
    if (cs > 1) {
        cg::cluster_group cl = cg::this_cluster();
        cl.sync();
        const int cr = (int)cl.block_rank(), cid = blockIdx.x / cs;
        const int per = (NE + cs - 1) / cs;
        for (int e = cr * per + tid; e < min(NE, (cr + 1) * per); e += kGramThreads) {
            double s = 0.0;
            for (int q = 0; q < cs; ++q) s += *cl.map_shared_rank(sm + e, q);
            part[(size_t)cid * NE + e] = s;
        }
        cl.sync();                                         // nobody exits while a peer still reads its sums
    } else {
        __syncthreads();
        for (int e = tid; e < NE; e += kGramThreads) part[(size_t)blockIdx.x * NE + e] = sm[e];
    }
}

// ---- small dense helpers of the algebra kernel (double, shared memory, leading dimension B + 1) --------------------------
// All b x b products run on the FP64 tensor-core path (mma.sync.m8n8k4): one 8 x 8 output tile per warp at a time (two in
// flight), k in steps of 4.  range(ti, tj, ks0, ks1) gives the k-step range of output tile (ti, tj) -- the operands are
// triangular, most tiles need a fraction of the k range -- or returns false when the tile is not part of this product.
// out(i, j, v) is called once for every element of a participating tile.
template <int B, class FA, class FB, class FR, class FO>
__device__ __forceinline__ void mm_dmma(int tid, int nthr, FA a, FB b, FR range, FO out) {
    constexpr int NT = B / 8;
    const int lane = tid & 31, w = tid >> 5, nw = nthr >> 5;
    const int fr = lane >> 2, fk = lane & 3;
    for (int t0 = w; t0 < NT * NT; t0 += 2 * nw) {
        const int t1 = t0 + nw;
        const int ti0 = t0 / NT, tj0 = t0 % NT, ti1 = t1 / NT, tj1 = t1 % NT;
        int a0 = 0, a1 = 0, b0 = 0, b1 = 0;
        const bool on0 = range(ti0, tj0, a0, a1), on1 = t1 < NT * NT && range(ti1, tj1, b0, b1);
        double c00 = 0.0, c01 = 0.0, c10 = 0.0, c11 = 0.0;
        if (!on0) a1 = a0;
        if (!on1) b1 = b0;
        const int n0 = max(a1 - a0, 0), n1 = max(b1 - b0, 0);
        for (int q = 0; q < max(n0, n1); ++q) {
            if (q < n0) {
                const int k = 4 * (a0 + q) + fk;
                dmma884(c00, c01, a(8 * ti0 + fr, k), b(k, 8 * tj0 + fr));
            }
            if (q < n1) {
                const int k = 4 * (b0 + q) + fk;
                dmma884(c10, c11, a(8 * ti1 + fr, k), b(k, 8 * tj1 + fr));
            }
        }
        if (on0) { out(8 * ti0 + fr, 8 * tj0 + 2 * fk, c00); out(8 * ti0 + fr, 8 * tj0 + 2 * fk + 1, c01); }
        if (on1) { out(8 * ti1 + fr, 8 * tj1 + 2 * fk, c10); out(8 * ti1 + fr, 8 * tj1 + 2 * fk + 1, c11); }
    }
}

// X = U^-1 for an upper triangular U given by the accessor u(i, j) (j >= i): the 8 x 8 diagonal blocks by back
// substitution (one thread per column, reciprocals of the diagonal formed in parallel first), then
// X_ab = -X_aa (U_ab X_bb) for blocks of 8, 16, 32 (log depth, tensor-core products).  X gets exact zeros below the
// diagonal.  Ends with a __syncthreads().
template <int B, class FU>
__device__ __forceinline__ void tri_inv_upper(FU u, double* __restrict__ X, double* __restrict__ tmp, double* __restrict__ dinv, int tid,
                                              int nthr) {
    constexpr int LD = B + 1;
    constexpr int S0 = B < 8 ? B : 8;
    for (int e = tid; e < B * B; e += nthr) X[(e / B) * LD + e % B] = 0.0;
    if (tid < B) dinv[tid] = 1.0 / u(tid, tid);
    __syncthreads();
    if (tid < B) {
        const int j = tid, d0 = (j / S0) * S0, jl = j - d0;
        double x[S0];
#pragma unroll
        for (int il = S0 - 1; il >= 0; --il) {
            double s0 = 0.0, s1 = 0.0;
#pragma unroll
            for (int kl = il + 1; kl < S0; ++kl)
                if (kl <= jl) { if ((kl - il) & 1) s0 += u(d0 + il, d0 + kl) * x[kl]; else s1 += u(d0 + il, d0 + kl) * x[kl]; }
            const double di = dinv[d0 + il];
            x[il] = il == jl ? di : (il < jl ? -(s0 + s1) * di : 0.0);
        }
#pragma unroll
        for (int il = 0; il < S0; ++il)
            if (il <= jl) X[(d0 + il) * LD + j] = x[il];
    }
#pragma unroll
    for (int s = S0; s < B; s *= 2) {
        __syncthreads();
        const int st = s / 8;                                  // tiles per block edge
        // tmp_ab = U_ab X_bb for every pair (a, b) = (2p, 2p+1) of s-blocks
        mm_dmma<B>(tid, nthr, [&](int i, int k) { return u(i, k); }, [&](int k, int j) { return X[k * LD + j]; },
                   [&](int ti, int tj, int& k0, int& k1) {
                       const int bi = ti / st, bj = tj / st;
                       if ((bi & 1) != 0 || bj != bi + 1) return false;
                       k0 = bj * s / 4; k1 = (8 * tj + 8) / 4;      // k in the b block, k <= j
                       return true;
                   },
                   [&](int i, int j, double v) { tmp[i * LD + j] = v; });
        __syncthreads();
        mm_dmma<B>(tid, nthr, [&](int i, int k) { return X[i * LD + k]; }, [&](int k, int j) { return tmp[k * LD + j]; },
                   [&](int ti, int tj, int& k0, int& k1) {
                       const int bi = ti / st, bj = tj / st;
                       if ((bi & 1) != 0 || bj != bi + 1) return false;
                       k0 = 8 * ti / 4; k1 = (bi + 1) * s / 4;      // k in the a block, k >= i
                       return true;
                   },
                   [&](int i, int j, double v) { X[i * LD + j] = -v; });
    }
    __syncthreads();
}

constexpr size_t chol_algebra_smem(int b) { return ((size_t)6 * b * (b + 1) + 4 * b + 8 * (b < 32 ? 32 : b) + 64) * sizeof(double); }

// ---- the b x b algebra: one CTA ------------------------------------------------------------------------------------------
// part: np tile-packed partial Gram matrices -- of the rows >= b when add_top != 0 (the kernel then adds A1^T A1), of all rows
// otherwise (np == 0: zero); top: the b x b top block in panel
// coordinates, element (r, c) at top[r*ldt + c] (kTopT == false) or top[c*ldt + r] (kTopT == true), overwritten with R_hh
// (exact zeros below the diagonal); top_d != nullptr: the input top block comes from there instead (dense, double, r*B + c:
// the distributed LQ panel, where it arrives with the all-reduced Gram matrix).  vtop / v2top receive the top b rows of V
// and V2 (V2 element (r, c) at v2top[r*ldv2r + c*ldv2c]).  mcat (b x 2b, row-major) = [M1 | M2] for the second pass.
//
// With Q = P R^-1 orthonormal, Y^T Y follows from the LU factors alone: T^-1 = diag(Y^T Y)/2 + striu(Y^T Y) = -L^T S U^-1
// (U = U~ R^-1), i.e. T = -U S L^-T, the formula of the reconstruction paper; here T^-1 is formed and inverted, which
// needs triangular products only:  M1 = U~^-1,  U^-1 = R M1,  T^-1 = -L^T S U^-1,  M2 = -M1 T^T,  V2 top = -L T^T.
template <typename T, bool kTopT, int B>
__global__ void __launch_bounds__(kAlgThreads, 1)
chol_algebra_kernel(T* __restrict__ top, size_t ldt, const double* __restrict__ top_d, const double* __restrict__ part, int np,
                    T* __restrict__ vtop, T* __restrict__ v2top, size_t ldv2r, size_t ldv2c, T* __restrict__ mcat, int* __restrict__ status,
                    double guard, int add_top) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    constexpr int LD = B + 1, NB8 = B / 8, NT = NB8 * (NB8 + 1) / 2, NE = NT * 64;
    double* Gc = reinterpret_cast<double*>(smem_raw);   // G2 -> G -> reduced Gram matrix (upper); R^T below the diagonal as rows finish
    double* W = Gc + B * LD;         // A1 under elimination; later scratch of the inversions
    double* LU = W + B * LD;         // L (strictly lower) and U~ (upper)
    double* M1 = LU + B * LD;        // U~^-1
    double* Ui = M1 + B * LD;        // U^-1 = R M1; later T
    double* S5 = Ui + B * LD;        // T^-1
    double* gdiag = S5 + B * LD;
    double* rdiag = gdiag + B;
    double* sgn = rdiag + B;
    double* dinv = sgn + B;
    double* sc = dinv + B;           // 32 step scalars (ring buffers), then 8 x BP doubles of pivot row / column buffers
    int* ctl = reinterpret_cast<int*>(sc + 32 + 8 * (B < 32 ? 32 : B));
    const int tid = threadIdx.x;
    long long tick = SVDB_PANEL_TIMING ? clock64() : 0;
    (void)tick;

    // ---- G2 (deterministic sum of the partials; all loads of a thread are issued before the first use), A1 -----------------
    {
        constexpr int NU = (NE + kAlgThreads - 1) / kAlgThreads, NV = (B * B + kAlgThreads - 1) / kAlgThreads;
        double tv[NV], sreg[NU];
#pragma unroll
        for (int u = 0; u < NV; ++u) {
            const int e = tid + u * kAlgThreads;
            const int r = kTopT ? e % B : e / B, c = kTopT ? e / B : e % B;
            tv[u] = 0.0;
            if (e < B * B) tv[u] = top_d ? top_d[r * B + c] : (double)top[kTopT ? (size_t)c * ldt + r : (size_t)r * ldt + c];
        }
#pragma unroll
        for (int u = 0; u < NU; ++u) sreg[u] = 0.0;
        for (int p0 = 0; p0 < np; p0 += 4) {
            double v[NU][4];
#pragma unroll
            for (int u = 0; u < NU; ++u)
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int e = tid + u * kAlgThreads;
                    v[u][q] = (e < NE && p0 + q < np) ? __ldcg(part + (size_t)(p0 + q) * NE + e) : 0.0;
                }
#pragma unroll
            for (int u = 0; u < NU; ++u)
#pragma unroll
                for (int q = 0; q < 4; ++q) sreg[u] += v[u][q];
        }
#pragma unroll
        for (int u = 0; u < NU; ++u) {
            const int e = tid + u * kAlgThreads;
            if (e < NE) {
                const int idx = e >> 6, within = e & 63;
                int ti = 0, rem = idx;
                while (rem >= NB8 - ti) { rem -= NB8 - ti; ++ti; }
                const int tj = ti + rem;
                Gc[(8 * ti + (within >> 3)) * LD + 8 * tj + (within & 7)] = sreg[u];
            }
        }
#pragma unroll
        for (int u = 0; u < NV; ++u) {
            const int e = tid + u * kAlgThreads;
            const int r = kTopT ? e % B : e / B, c = kTopT ? e / B : e % B;
            if (e < B * B) W[r * LD + c] = tv[u];
        }
    }
    if (tid == 0) ctl[0] = 0;
    __syncthreads();
    CHOL_TICK(0);
    // ---- G = G2 + A1^T A1 (upper tiles) -- only when pass 1 left the top block out (add_top); otherwise the partials are G already ----
    if (add_top) {
        mm_dmma<B>(tid, kAlgThreads, [&](int i, int k) { return W[k * LD + i]; }, [&](int k, int j) { return W[k * LD + j]; },
                   [](int ti, int tj, int& k0, int& k1) { k0 = 0; k1 = B / 4; return tj >= ti; },
                   [&](int i, int j, double v) { Gc[i * LD + j] += v; });
        __syncthreads();
    }
    if (tid < B) gdiag[tid] = Gc[tid * LD + tid];
    CHOL_TICK(1);
    // ---- Cholesky (as a square-root-free elimination; row i of R is row i of the reduced matrix / sqrt(g_ii)) and the LU
    //      factorisation of A1 - S R, one column per step, ONE barrier per step.  The loop is bound by latency: the dependent
    //      chain of the step scalars (tools/probes/fp64_latency.cu on this GPU: DFMA 8, 1/x 82, rsqrt 77, barrier + hand-over
    //      through shared memory 113 cycles) and each warp's own instruction stream.  Hence:
    //        * both matrices stay in registers for the whole elimination (row k on warp k % 16, column j on lane j % 32); per
    //          step only the pivot rows and the pivot column of W go through shared memory, published by their owners;
    //        * the chain is cut into three that run on different warps: iteration t runs Cholesky step t (update, 1/g), a
    //          helper lane that forms sqrt(g_tt) (and the guard), and LU step t-2 (update, pivot = w - s sqrt(g), 1/pivot);
    //        * an owner warp updates the row it has to publish first, and does the part it owns first;
    //        * the updates are unconditional (no per-element predicates): finished rows / columns become garbage that is
    //          never published.
    //      Measured 900 (b = 32) / 1370 (b = 64) cycles per step; profiles/r02_summary.md has the history. ---------------------------
    constexpr int NW = kAlgThreads / 32;
    constexpr int RPW = B >= NW ? B / NW : 1, CPT = B >= 32 ? B / 32 : 1;
    constexpr int BP = B < 32 ? 32 : B;      // padded row length of the exchange buffers (lanes beyond B read / write padding)
    const int lane = tid & 31, wid = tid >> 5;
    double* rowG = sc + 32;          // 4 x BP (row t: written in iteration t-1, read by Cholesky step t, the helper, and LU step t in iteration t+2)
    double* rowW = rowG + 4 * BP;    // 2 x BP
    double* colW = rowW + 2 * BP;    // 2 x BP
    double* scC = sc;                // 4 x {1/g_tt}
    double* scH = sc + 4;            // 4 x {1/sqrt(g_tt), sqrt(g_tt)}
    double* scL = sc + 12;           // 2 x {s, 1/pivot}
    // Registers: g[p][q] = G[wid + 16p][lane + 32q], same for W.  The updates below are UNCONDITIONAL: elements outside
    // the live part (finished rows / columns, the lower triangle of G) turn into garbage that is never published.
    double g[RPW][CPT], wv[RPW][CPT];
#pragma unroll
    for (int p = 0; p < RPW; ++p)
#pragma unroll
        for (int q = 0; q < CPT; ++q) {
            const int k = wid + NW * p, j = lane + 32 * q;
            const bool in = k < B && j < B;
            g[p][q] = in ? Gc[min(k, j) * LD + max(k, j)] : 0.0;
            wv[p][q] = in ? W[k * LD + j] : 0.0;
        }
    // run f(p) for the compile-time p equal to the (warp-uniform) ps
    auto with_p = [&](int ps, auto&& f) {
        if (ps == 0) f(std::integral_constant<int, 0>{});
        if constexpr (RPW > 1) { if (ps == 1) f(std::integral_constant<int, 1>{}); }
        if constexpr (RPW > 2) { if (ps == 2) f(std::integral_constant<int, 2>{}); }
        if constexpr (RPW > 3) { if (ps == 3) f(std::integral_constant<int, 3>{}); }
    };
    auto with_q = [&](int qs, auto&& f) {
        if (qs == 0) f(std::integral_constant<int, 0>{});
        if constexpr (CPT > 1) { if (qs == 1) f(std::integral_constant<int, 1>{}); }
    };
    __syncthreads();                 // gdiag
    if (wid == 0) {                  // row 0 of G and 1/g_00
#pragma unroll
        for (int q = 0; q < CPT; ++q) rowG[lane + 32 * q] = g[0][q];
        if (lane == 0) scC[0] = 1.0 / g[0][0];
    }
    __syncthreads();
    for (int t = 0; t <= B; ++t) {
        const int i = t - 2;                                  // LU step of this iteration (valid from t = 2)
        const bool lown = t >= 1 && t - 1 < B && wid == (t - 1) % NW;     // this warp owns row t-1 = i+1: on the LU chain
        auto lu_part = [&]() {
            if (t < 1) return;
            double ui[CPT], lk[RPW];
            if (i >= 0) {
                const double s = scL[(i & 1) * 2], pinv = scL[(i & 1) * 2 + 1], rsq = scH[(i & 3) * 2];
                const double* rg = rowG + (i & 3) * BP;
                const double* rw = rowW + (i & 1) * BP;
                const double* cw = colW + (i & 1) * BP;
                double ri[CPT];
#pragma unroll
                for (int q = 0; q < CPT; ++q) {
                    ri[q] = rg[lane + 32 * q] * rsq;          // R[i][j]
                    ui[q] = rw[lane + 32 * q] - s * ri[q];    // U~[i][j]
                }
#pragma unroll
                for (int p = 0; p < RPW; ++p) lk[p] = cw[wid + NW * p] * pinv;
                if (lown) {                                   // the row that has to be published goes first
                    with_p((t - 1) / NW, [&](auto pc) {
#pragma unroll
                        for (int q = 0; q < CPT; ++q) wv[pc][q] -= lk[pc] * ui[q];
                    });
                }
                if (wid == i % NW) {                          // the owner of row i: row i of U~ and of R
#pragma unroll
                    for (int q = 0; q < CPT; ++q) {
                        const int j = lane + 32 * q;
                        if (j > i && j < B) {
                            LU[i * LD + j] = ui[q];
                            Gc[j * LD + i] = ri[q];           // stored transposed below the diagonal
                        }
                    }
                }
            }
            if (lown) {                                       // publish row t-1 of W and the scalars of LU step t-1
                const int r = t - 1;
                with_p(r / NW, [&](auto pc) {
#pragma unroll
                    for (int q = 0; q < CPT; ++q) rowW[(r & 1) * BP + lane + 32 * q] = wv[pc][q];
                    if (lane == (r & 31)) {
                        with_q(r >> 5, [&](auto qc) {
                            const double wii = wv[pc][qc];
                            const double rii = scH[(r & 3) * 2 + 1];      // formed by the helper one iteration earlier
                            const double s = -copysign(1.0, wii);
                            const double piv = wii - s * rii;
                            scL[(r & 1) * 2] = s; scL[(r & 1) * 2 + 1] = 1.0 / piv;
                            LU[r * LD + r] = piv; sgn[r] = s;
                        });
                    }
                });
            }
            if (i >= 0) {
                const int ps = lown ? (t - 1) / NW : -1;
#pragma unroll
                for (int p = 0; p < RPW; ++p) {
                    if (p != ps) {
#pragma unroll
                        for (int q = 0; q < CPT; ++q) wv[p][q] -= lk[p] * ui[q];
                    }
                }
                if (lane == 0) {                              // column i of L
#pragma unroll
                    for (int p = 0; p < RPW; ++p) {
                        const int k = wid + NW * p;
                        if (k > i && k < B) LU[k * LD + i] = lk[p];
                    }
                }
            }
            if (t - 1 < B && lane == ((t - 1) & 31)) {        // every warp: its rows of column t-1 of W
                with_q((t - 1) >> 5, [&](auto qc) {
#pragma unroll
                    for (int p = 0; p < RPW; ++p) colW[((t - 1) & 1) * BP + wid + NW * p] = wv[p][qc];
                });
            }
        };
        if (lown) lu_part();
        if (t < B) {                                          // ---- Cholesky step t ----
            const double ginv = scC[t & 3];
            const double* rg = rowG + (t & 3) * BP;
            double gi[CPT], gk[RPW];
#pragma unroll
            for (int q = 0; q < CPT; ++q) gi[q] = rg[lane + 32 * q];
#pragma unroll
            for (int p = 0; p < RPW; ++p) gk[p] = rg[wid + NW * p] * ginv;
            const bool cown = t + 1 < B && wid == (t + 1) % NW;           // this warp owns row t+1: on the Cholesky chain
            if (cown) {
                const int r = t + 1;
                with_p(r / NW, [&](auto pc) {
#pragma unroll
                    for (int q = 0; q < CPT; ++q) {
                        g[pc][q] -= gk[pc] * gi[q];
                        rowG[(r & 3) * BP + lane + 32 * q] = g[pc][q];
                    }
                    if (lane == (r & 31)) with_q(r >> 5, [&](auto qc) { scC[r & 3] = 1.0 / g[pc][qc]; });
                });
            }
            const int ps = cown ? (t + 1) / NW : -1;
#pragma unroll
            for (int p = 0; p < RPW; ++p) {
                if (p != ps) {
#pragma unroll
                    for (int q = 0; q < CPT; ++q) g[p][q] -= gk[p] * gi[q];
                }
            }
            if (wid == (t + NW / 2) % NW && lane == 0) {      // helper: sqrt(g_tt) and the guard, off both chains
                const double gtt = rg[t];
                if ((!(gtt > guard * gdiag[t]) || !(gtt < 1e300)) && ctl[0] == 0) { ctl[0] = 1; ctl[1] = t; ctl[2] = __float_as_int((float)(gtt / gdiag[t])); }
                const double rsq = rsqrt(gtt), rii = gtt * rsq;
                scH[(t & 3) * 2] = rsq; scH[(t & 3) * 2 + 1] = rii; rdiag[t] = rii;
            }
        }
        if (!lown) lu_part();
        __syncthreads();
    }
    CHOL_TICK(2);
    if (ctl[0] != 0) {
        if (tid == 0) { status[0] = 1; status[1] += 1; status[2] = ctl[1]; status[3] = ctl[2]; }     // [2], [3]: column and pivot ratio of the last panel given up
        return;
    }
    auto Lf = [&](int r, int c) { return c < r ? LU[r * LD + c] : (c == r ? 1.0 : 0.0); };
    auto Uf = [&](int r, int c) { return c >= r ? LU[r * LD + c] : 0.0; };
    auto Rf = [&](int r, int c) { return c > r ? Gc[c * LD + r] : (c == r ? rdiag[r] : 0.0); };
    // ---- M1 = U~^-1 ------------------------------------------------------------------------------------------------------------
    tri_inv_upper<B>(Uf, M1, W, dinv, tid, kAlgThreads);
    CHOL_TICK(3);
    // ---- U^-1 = R M1 (upper x upper) ----------------------------------------------------------------------------------------------
    mm_dmma<B>(tid, kAlgThreads, Rf, [&](int k, int j) { return M1[k * LD + j]; },
               [](int ti, int tj, int& k0, int& k1) { k0 = 2 * ti; k1 = tj >= ti ? 2 * tj + 2 : k0; return true; },
               [&](int i, int j, double v) { Ui[i * LD + j] = v; });
    __syncthreads();
    CHOL_TICK(4);
    // ---- T^-1 = -L^T S U^-1 (upper) --------------------------------------------------------------------------------------------------
    mm_dmma<B>(tid, kAlgThreads, [&](int i, int k) { return Lf(k, i) * sgn[k]; }, [&](int k, int j) { return Ui[k * LD + j]; },
               [](int ti, int tj, int& k0, int& k1) { k0 = 2 * ti; k1 = tj >= ti ? 2 * tj + 2 : k0; return true; },
               [&](int i, int j, double v) { S5[i * LD + j] = -v; });
    __syncthreads();
    CHOL_TICK(5);
    // ---- T (into Ui; W is scratch) ----------------------------------------------------------------------------------------------------
    double* Tm = Ui;
    tri_inv_upper<B>([&](int r, int c) { return c >= r ? S5[r * LD + c] : 0.0; }, Tm, W, dinv, tid, kAlgThreads);
    CHOL_TICK(6);
    // ---- outputs ---------------------------------------------------------------------------------------------------------------------
    // M2 = -M1 T^T (b x b), V2 top block = -L T^T (lower triangular)
    mm_dmma<B>(tid, kAlgThreads, [&](int i, int k) { return M1[i * LD + k]; }, [&](int k, int j) { return Tm[j * LD + k]; },
               [](int ti, int tj, int& k0, int& k1) { k0 = 2 * max(ti, tj); k1 = B / 4; return true; },
               [&](int i, int j, double v) { mcat[(size_t)i * (2 * B) + B + j] = (T)(-v); });
    mm_dmma<B>(tid, kAlgThreads, Lf, [&](int k, int j) { return Tm[j * LD + k]; },
               [](int ti, int tj, int& k0, int& k1) { k0 = 2 * tj; k1 = ti >= tj ? 2 * ti + 2 : k0; return true; },
               [&](int i, int j, double v) { v2top[(size_t)i * ldv2r + (size_t)j * ldv2c] = (T)(j <= i ? -v : 0.0); });
    for (int e = tid; e < B * B; e += kAlgThreads) {
        const int r = kTopT ? e % B : e / B, c = kTopT ? e / B : e % B;
        top[kTopT ? (size_t)c * ldt + r : (size_t)r * ldt + c] = (T)(sgn[r] * Rf(r, c));
    }
    for (int e = tid; e < B * B; e += kAlgThreads) {
        const int r = e / B, c = e % B;
        vtop[(size_t)r * B + c] = (T)Lf(r, c);
        mcat[(size_t)r * (2 * B) + c] = (T)M1[r * LD + c];
    }
    if (tid == 0) status[0] = 0;
    CHOL_TICK(7);
    if (SVDB_PANEL_TIMING && tid == 0) g_chol_dbg[15] += 1;
}

// ---- pass 2: [Y2 | V2_2] = A2 [M1 | M2], zeros into A2 ----------------------------------------------------------------------
template <typename T, int N> __device__ __forceinline__ void ldn(const T* p, T (&v)[N]) {
    if constexpr (N % 4 == 0 && sizeof(T) == 4) {
#pragma unroll
        for (int q = 0; q < N / 4; ++q) {
            const float4 t = *reinterpret_cast<const float4*>(p + 4 * q);
            v[4 * q] = t.x; v[4 * q + 1] = t.y; v[4 * q + 2] = t.z; v[4 * q + 3] = t.w;
        }
    } else if constexpr (N % 2 == 0 && sizeof(T) == 8) {
#pragma unroll
        for (int q = 0; q < N / 2; ++q) {
            const double2 t = *reinterpret_cast<const double2*>(p + 2 * q);
            v[2 * q] = t.x; v[2 * q + 1] = t.y;
        }
    } else {
#pragma unroll
        for (int q = 0; q < N; ++q) v[q] = p[q];
    }
}
template <typename T, int N> __device__ __forceinline__ void stn(T* p, const T (&v)[N]) {
    if constexpr (N % 4 == 0 && sizeof(T) == 4) {
#pragma unroll
        for (int q = 0; q < N / 4; ++q) *reinterpret_cast<float4*>(p + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
    } else if constexpr (N % 2 == 0 && sizeof(T) == 8) {
#pragma unroll
        for (int q = 0; q < N / 2; ++q) *reinterpret_cast<double2*>(p + 2 * q) = make_double2(v[2 * q], v[2 * q + 1]);
    } else {
#pragma unroll
        for (int q = 0; q < N; ++q) p[q] = v[q];
    }
}

constexpr size_t chol_apply_smem(int b, size_t esz) { return ((size_t)b * 2 * b + (size_t)b * (kApplyRows + kApplyPad)) * esz; }

// Rows [row0, m) of the panel (element (r, c) as in pidx); outputs: V rows (r*B + c), V2 element (r, c) at
// V2[r*ldv2r + c*ldv2c] (either ldv2r == B, ldv2c == 1 or ldv2r == 1), zeros into the panel rows.
template <typename T, bool kTrans, int B>
__global__ void __launch_bounds__(kApplyThreads)
chol_apply_kernel(T* __restrict__ A, size_t lda, int row0, int m, const T* __restrict__ mcat, T* __restrict__ V, T* __restrict__ V2,
                  size_t ldv2r, size_t ldv2c, const int* __restrict__ status) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (status[0] != 0) return;
    constexpr int RB = kApplyRows, LDA = RB + kApplyPad, NC = 2 * B;
    constexpr int TN = NC >= 16 ? NC / 16 : 1;
    T* Ms = reinterpret_cast<T*>(smem_raw);          // B x 2B
    T* As = Ms + B * NC;                             // B x LDA (k-major)
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int rbase = row0 + blockIdx.x * RB;
    for (int e = tid; e < B * NC; e += kApplyThreads) Ms[e] = mcat[e];
    if (!kTrans) {
        for (int e = tid; e < RB * B; e += kApplyThreads) {
            const int r = e / B, k = e % B;
            As[k * LDA + r] = rbase + r < m ? A[(size_t)(rbase + r) * lda + k] : (T)0;
        }
    } else {
        for (int e = tid; e < RB * B; e += kApplyThreads) {
            const int k = e / RB, r = e % RB;
            As[k * LDA + r] = rbase + r < m ? A[(size_t)k * lda + rbase + r] : (T)0;
        }
    }
    __syncthreads();
    const int r0 = ty * 4, j0 = tx * TN;
    T acc[4][TN];
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
        for (int q = 0; q < TN; ++q) acc[p][q] = (T)0;
    if (j0 < NC) {
#pragma unroll 4
        for (int k = 0; k < B; ++k) {
            T av[4], bv[TN];
            ldn<T, 4>(As + k * LDA + r0, av);
            ldn<T, TN>(Ms + k * NC + j0, bv);
#pragma unroll
            for (int p = 0; p < 4; ++p)
#pragma unroll
                for (int q = 0; q < TN; ++q) acc[p][q] += av[p] * bv[q];
        }
    }
    __syncthreads();                                 // As is reused below
    const bool v2_strided = ldv2r == 1;              // V2 element (r, c) at V2[c*ldv2c + r]: staged through shared memory
    if (j0 < B) {
#pragma unroll
        for (int p = 0; p < 4; ++p)
            if (rbase + r0 + p < m) stn<T, TN>(V + (size_t)(rbase + r0 + p) * B + j0, acc[p]);
    } else if (j0 < NC) {
        if (!v2_strided) {
#pragma unroll
            for (int p = 0; p < 4; ++p)
                if (rbase + r0 + p < m) stn<T, TN>(V2 + (size_t)(rbase + r0 + p) * ldv2r + (j0 - B), acc[p]);
        } else {
#pragma unroll
            for (int q = 0; q < TN; ++q)
#pragma unroll
                for (int p = 0; p < 4; ++p) As[(j0 - B + q) * LDA + r0 + p] = acc[p][q];
        }
    }
    if (v2_strided) {
        __syncthreads();
        for (int e = tid; e < RB * B; e += kApplyThreads) {
            const int c = e / RB, r = e % RB;
            if (rbase + r < m) V2[(size_t)c * ldv2c + rbase + r] = As[c * LDA + r];
        }
    }
    if (!kTrans) {
        for (int e = tid; e < RB * B; e += kApplyThreads) {
            const int r = e / B, c = e % B;
            if (rbase + r < m) A[(size_t)(rbase + r) * lda + c] = (T)0;
        }
    } else {
        for (int e = tid; e < RB * B; e += kApplyThreads) {
            const int c = e / RB, r = e % RB;
            if (rbase + r < m) A[(size_t)c * lda + rbase + r] = (T)0;
        }
    }
}

// cudaFuncSetAttribute costs ~1 us of host time per call: once per kernel instantiation and device
template <class K>
inline cudaError_t smem_attr_once(Ctx* c, K kern, size_t smem, bool (&done)[16]) {
    const int dev = c->device & 15;
    if (done[dev]) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) done[dev] = true;
    return e;
}

struct GramShape { int rows, ng, cs, np; };
inline GramShape gram_shape(int mrows, int num_sms) {
    GramShape g;
    if (mrows <= 0) { g.rows = 8; g.ng = 0; g.cs = 1; g.np = 0; return g; }
    const int target = std::max(1, std::min(num_sms / kGramCluster * kGramCluster, (mrows + 63) / 64));
    g.rows = ((mrows + target - 1) / target + 7) / 8 * 8;
    g.ng = (mrows + g.rows - 1) / g.rows;
    g.cs = g.ng >= kGramCluster ? kGramCluster : (g.ng >= 4 ? 4 : (g.ng >= 2 ? 2 : 1));
    g.ng = (g.ng + g.cs - 1) / g.cs * g.cs;
    g.np = g.ng / g.cs;
    return g;
}

template <typename T, bool kTrans, int B>
int gram_launch(Ctx* c, const T* a, size_t lda, int row0, int m, double* part, const GramShape& g, cudaStream_t stream) {
    constexpr int NB8 = B / 8, NE = NB8 * (NB8 + 1) / 2 * 64;
    auto kern = chol_gram_kernel<T, kTrans, NB8>;
    const size_t smem = (size_t)kGramWarps * NE * sizeof(double);
    { static bool attr_done[16] = {}; SVDB_CHECK(c, smem_attr_once(c, kern, smem, attr_done)); }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(g.ng);
    cfg.blockDim = dim3(kGramThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = g.cs;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    SVDB_CHECK(c, cudaLaunchKernelEx(&cfg, kern, a, lda, row0, m, g.rows, g.cs, part));
    c->launches++;
    return 0;
}

template <typename T, bool kTrans, int B>
int launch_chol(Ctx* c, T* a, size_t lda, int m, T* V, T* V2, cudaStream_t stream) {
    char* ws = reinterpret_cast<char*>(c->chol_ws);
    int* status = reinterpret_cast<int*>(ws);
    T* mcat = reinterpret_cast<T*>(ws + 256);
    double* part = reinterpret_cast<double*>(ws + 256 + 64 * 128 * 8);
    const GramShape g = gram_shape(m, c->num_sms);     // pass 1 over ALL rows: the partials sum to G itself
    SVDB_TRY((gram_launch<T, kTrans, B>(c, a, lda, 0, m, part, g, stream)));
    {
        auto kern = chol_algebra_kernel<T, kTrans, B>;
        const size_t smem = chol_algebra_smem(B);
        { static bool attr_done[16] = {}; SVDB_CHECK(c, smem_attr_once(c, kern, smem, attr_done)); }
        const size_t ldv2r = kTrans ? 1 : (size_t)B, ldv2c = kTrans ? (size_t)m : 1;
        kern<<<1, kAlgThreads, smem, stream>>>(a, lda, (const double*)nullptr, part, g.np, V, V2, ldv2r, ldv2c, mcat, status, c->cfg.chol_guard, 0);
        c->launches++;
    }
    {
        auto kern = chol_apply_kernel<T, kTrans, B>;
        const size_t smem = chol_apply_smem(B, sizeof(T));
        { static bool attr_done[16] = {}; SVDB_CHECK(c, smem_attr_once(c, kern, smem, attr_done)); }
        const size_t ldv2r = kTrans ? 1 : (size_t)B, ldv2c = kTrans ? (size_t)m : 1;
        const int grid = (m - B + kApplyRows - 1) / kApplyRows;
        kern<<<grid, kApplyThreads, smem, stream>>>(a, lda, B, m, mcat, V, V2, ldv2r, ldv2c, status);
        c->launches++;
    }
    SVDB_CHECK(c, cudaGetLastError());
    return 0;
}

}  // namespace

// 0: launched (the caller must enqueue a fallback panel kernel gated on chol_status()); 1: shape not covered
template <typename T, bool kTrans>
int launch_panel_chol(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream) {
    // not beside resident stage-2 grids (overlap_safe): measured slower there, its kernels disturb the latency-bound stage-2
    // chains of the list pipeline (2896 -> 2211-2551 GFLOP/s on the bench sweep)
    if (!c->chol_ws || m < 2 * b || c->overlap_safe) return 1;
    switch (b) {
        case 8: return launch_chol<T, kTrans, 8>(c, a, lda, m, V, V2, stream);
        case 16: return launch_chol<T, kTrans, 16>(c, a, lda, m, V, V2, stream);
        case 32: return launch_chol<T, kTrans, 32>(c, a, lda, m, V, V2, stream);
        case 64: return launch_chol<T, kTrans, 64>(c, a, lda, m, V, V2, stream);
        default: return 1;
    }
}
template int launch_panel_chol<float, false>(Ctx*, float*, size_t, int, int, float*, float*, cudaStream_t);
template int launch_panel_chol<float, true>(Ctx*, float*, size_t, int, int, float*, float*, cudaStream_t);
template int launch_panel_chol<double, false>(Ctx*, double*, size_t, int, int, double*, double*, cudaStream_t);
template int launch_panel_chol<double, true>(Ctx*, double*, size_t, int, int, double*, double*, cudaStream_t);

const int* chol_status(Ctx* c) { return reinterpret_cast<const int*>(c->chol_ws); }
int panel_chol_debug_read(long long* out16) {
    long long z[16] = {};
    if (cudaMemcpyFromSymbol(out16, g_chol_dbg, sizeof(z)) != cudaSuccess) return 1;
    cudaMemcpyToSymbol(g_chol_dbg, z, sizeof(z));
    return 0;
}

// ---- distributed LQ panel (dist.cu): the b x n' row panel is spread over the ranks by columns = by panel rows ---------------
// Every rank: Gram matrix of its local panel rows (the owner of the first trailing block also contributes the top b x b block
// as is) -> ONE all-reduce of [tile-packed G2 | A1] in double (dist.cu) -> the same b x b algebra on every
// rank (identical inputs => identical [M1 | M2]) -> second pass over the local rows, which leaves U^T and S U directly in
// the rank's local layout.  No gather of the row panel, no redundant factorisation of an n'-wide panel.
namespace {
template <typename T, int B>
__global__ void chol_pack_kernel(const double* __restrict__ part, int np, const T* __restrict__ top_src, size_t ldl, double* __restrict__ buf) {
    constexpr int NB8 = B / 8, NE = NB8 * (NB8 + 1) / 2 * 64;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < NE) {
        double s = 0.0;
        for (int p = 0; p < np; ++p) s += part[(size_t)p * NE + e];
        buf[e] = s;
    } else if (e < NE + B * B) {
        const int q = e - NE, c = q / B, r = q % B;          // panel element (r, c) of the top block sits at top_src[c*ldl + r]
        buf[NE + r * B + c] = top_src ? (double)top_src[(size_t)c * ldl + r] : 0.0;
    }
}

template <typename T, int B>
int dist_lq_gram(Ctx* c, const T* a2, size_t ldl, int row0, int ncl, bool own_top, double* buf, cudaStream_t stream) {
    constexpr int NB8 = B / 8, NE = NB8 * (NB8 + 1) / 2 * 64;
    char* ws = reinterpret_cast<char*>(c->chol_ws);
    double* part = reinterpret_cast<double*>(ws + 256 + 64 * 128 * 8);
    (void)row0;                                            // pass 1 covers all local rows (the top block's rows included: G, not G2)
    const GramShape g = gram_shape(ncl, c->num_sms);
    if (g.ng > 0) SVDB_TRY((gram_launch<T, true, B>(c, a2, ldl, 0, ncl, part, g, stream)));
    const int tot = NE + B * B;
    chol_pack_kernel<T, B><<<(tot + 255) / 256, 256, 0, stream>>>(part, g.np, own_top ? a2 : nullptr, ldl, buf);
    c->launches++;
    SVDB_CHECK(c, cudaGetLastError());
    return 0;
}

template <typename T, int B>
int dist_lq_finish(Ctx* c, T* a2, size_t ldl, int row0, int ncl, bool own_top, const double* buf, T* ut_loc, T* u2_loc, cudaStream_t stream) {
    constexpr int NB8 = B / 8, NE = NB8 * (NB8 + 1) / 2 * 64;
    char* ws = reinterpret_cast<char*>(c->chol_ws);
    int* status = reinterpret_cast<int*>(ws) + 4;          // own status / counter pair: [4] = last panel, [5] = panels given up
    T* mcat = reinterpret_cast<T*>(ws + 256);
    T* scratch = reinterpret_cast<T*>(ws + 256 + 64 * 128 * 8 + 18 * 2304 * 8);     // 3 x b x b: outputs nobody needs on non-owners
    {
        auto kern = chol_algebra_kernel<T, true, B>;
        const size_t smem = chol_algebra_smem(B);
        { static bool attr_done[16] = {}; SVDB_CHECK(c, smem_attr_once(c, kern, smem, attr_done)); }
        if (own_top)
            kern<<<1, kAlgThreads, smem, stream>>>(a2, ldl, buf + NE, buf, 1, ut_loc, u2_loc, (size_t)1, (size_t)ncl, mcat, status, c->cfg.chol_guard, 0);
        else
            kern<<<1, kAlgThreads, smem, stream>>>(scratch, (size_t)B, buf + NE, buf, 1, scratch + B * B, scratch + 2 * B * B, (size_t)1, (size_t)B,
                                                   mcat, status, c->cfg.chol_guard, 0);
        c->launches++;
    }
    if (ncl > row0) {
        auto kern = chol_apply_kernel<T, true, B>;
        const size_t smem = chol_apply_smem(B, sizeof(T));
        { static bool attr_done[16] = {}; SVDB_CHECK(c, smem_attr_once(c, kern, smem, attr_done)); }
        const int grid = (ncl - row0 + kApplyRows - 1) / kApplyRows;
        kern<<<grid, kApplyThreads, smem, stream>>>(a2, ldl, row0, ncl, mcat, ut_loc, u2_loc, (size_t)1, (size_t)ncl, status);
        c->launches++;
    }
    SVDB_CHECK(c, cudaGetLastError());
    return 0;
}
}  // namespace

size_t chol_dist_buf_elems(int b) { const int nb8 = b / 8; return (size_t)nb8 * (nb8 + 1) / 2 * 64 + (size_t)b * b; }
bool chol_dist_supported(const Ctx* c, int b) { return c->chol_ws && c->cfg.panel_chol && (b == 8 || b == 16 || b == 32 || b == 64); }

template <typename T>
int chol_dist_lq_gram(Ctx* c, const T* a2, size_t ldl, int b, int row0, int ncl, bool own_top, double* buf, cudaStream_t stream) {
    switch (b) {
        case 8: return dist_lq_gram<T, 8>(c, a2, ldl, row0, ncl, own_top, buf, stream);
        case 16: return dist_lq_gram<T, 16>(c, a2, ldl, row0, ncl, own_top, buf, stream);
        case 32: return dist_lq_gram<T, 32>(c, a2, ldl, row0, ncl, own_top, buf, stream);
        case 64: return dist_lq_gram<T, 64>(c, a2, ldl, row0, ncl, own_top, buf, stream);
        default: return SVDB200_E_CAPACITY;
    }
}
template <typename T>
int chol_dist_lq_finish(Ctx* c, T* a2, size_t ldl, int b, int row0, int ncl, bool own_top, const double* buf, T* ut_loc, T* u2_loc,
                        cudaStream_t stream) {
    switch (b) {
        case 8: return dist_lq_finish<T, 8>(c, a2, ldl, row0, ncl, own_top, buf, ut_loc, u2_loc, stream);
        case 16: return dist_lq_finish<T, 16>(c, a2, ldl, row0, ncl, own_top, buf, ut_loc, u2_loc, stream);
        case 32: return dist_lq_finish<T, 32>(c, a2, ldl, row0, ncl, own_top, buf, ut_loc, u2_loc, stream);
        case 64: return dist_lq_finish<T, 64>(c, a2, ldl, row0, ncl, own_top, buf, ut_loc, u2_loc, stream);
        default: return SVDB200_E_CAPACITY;
    }
}
template int chol_dist_lq_gram<float>(Ctx*, const float*, size_t, int, int, int, bool, double*, cudaStream_t);
template int chol_dist_lq_gram<double>(Ctx*, const double*, size_t, int, int, int, bool, double*, cudaStream_t);
template int chol_dist_lq_finish<float>(Ctx*, float*, size_t, int, int, int, bool, const double*, float*, float*, cudaStream_t);
template int chol_dist_lq_finish<double>(Ctx*, double*, size_t, int, int, int, bool, const double*, double*, double*, cudaStream_t);
// ---- distributed QR panel (dist.cu): the m x b column panel lives on one rank ------------------------------------------------
// The owner runs pass 1 and the algebra, then ONE broadcast carries the raw rows b .. m-1 of the panel plus [M1 | M2], the
// top blocks of V and V2 and the status ((m - b) b + 4 b^2 + 4 elements instead of the 2 m b of [V | V S^T]); every rank runs
// the second pass on its copy.
namespace {
template <typename T>
__global__ void qr_pack_kernel(T* __restrict__ A, size_t lda, int m, int b, T* __restrict__ raw, T* __restrict__ flag, const int* __restrict__ status) {
    const bool bad = status[0] != 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) flag[0] = bad ? (T)1 : (T)0;
    if (bad) return;
    const size_t tot = (size_t)(m - b) * b;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / b, cc = e - r * b;
        T* src = A + (r + b) * lda + cc;
        raw[e] = *src;
        *src = (T)0;
    }
}
// early variant: the raw rows leave before the factorisation (the broadcast overlaps pass 1 and the algebra, which then read the
// contiguous copy); the panel rows are zeroed afterwards, once the status is known
template <typename T>
__global__ void qr_copy_kernel(const T* __restrict__ A, size_t lda, int m, int b, T* __restrict__ raw) {
    const size_t tot = (size_t)(m - b) * b;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / b, cc = e - r * b;
        raw[e] = A[(r + b) * lda + cc];
    }
}
template <typename T>
__global__ void qr_zero_kernel(T* __restrict__ A, size_t lda, int m, int b, T* __restrict__ flag, const int* __restrict__ status) {
    const bool bad = status[0] != 0;
    if (blockIdx.x == 0 && threadIdx.x == 0) flag[0] = bad ? (T)1 : (T)0;
    if (bad) return;
    const size_t tot = (size_t)(m - b) * b;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (size_t)gridDim.x * blockDim.x) {
        const size_t r = e / b, cc = e - r * b;
        A[(r + b) * lda + cc] = (T)0;
    }
}
template <typename T>
__global__ void qr_unpack_kernel(const T* __restrict__ small, int b, T* __restrict__ V, T* __restrict__ V2, int* __restrict__ status) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const bool bad = small[2 * b * b] != (T)0;
    if (e == 0) status[0] = bad ? 1 : 0;
    if (bad || e >= b * b) return;
    V[e] = small[e];
    V2[e] = small[b * b + e];
}

template <typename T, int B>
int dist_qr_owner(Ctx* c, T* a, size_t lda, int m, T* qsend, cudaStream_t stream) {
    char* ws = reinterpret_cast<char*>(c->chol_ws);
    int* status = reinterpret_cast<int*>(ws) + 8;
    double* part = reinterpret_cast<double*>(ws + 256 + 64 * 128 * 8);
    T* raw = qsend;
    T* mcat = qsend + (size_t)(m - B) * B;
    T* vtop = mcat + 2 * B * B;
    T* v2top = vtop + B * B;
    T* flag = v2top + B * B;
    const GramShape g = gram_shape(m - B, c->num_sms);
    SVDB_TRY((gram_launch<T, false, B>(c, a, lda, B, m, part, g, stream)));
    auto kern = chol_algebra_kernel<T, false, B>;
    const size_t smem = chol_algebra_smem(B);
    { static bool attr_done[16] = {}; SVDB_CHECK(c, smem_attr_once(c, kern, smem, attr_done)); }
    kern<<<1, kAlgThreads, smem, stream>>>(a, lda, (const double*)nullptr, part, g.np, vtop, v2top, (size_t)B, (size_t)1, mcat, status, c->cfg.chol_guard, 1);
    c->launches++;
    const size_t tot = (size_t)(m - B) * B;
    int blocks = (int)std::min<size_t>((tot + 1023) / 1024, (size_t)4 * c->num_sms);
    qr_pack_kernel<T><<<blocks, 256, 0, stream>>>(a, lda, m, B, raw, flag, status);
    c->launches++;
    SVDB_CHECK(c, cudaGetLastError());
    return 0;
}
// early variant, owner: phase 0 = copy the raw rows out (then the caller starts their broadcast); phase 1 = pass 1 on the copy,
// algebra, flag, zeros into the panel rows (then the caller broadcasts the small tail of the message)
template <typename T, int B>
int dist_qr_owner_early(Ctx* c, T* a, size_t lda, int m, T* qsend, int phase, cudaStream_t stream) {
    char* ws = reinterpret_cast<char*>(c->chol_ws);
    int* status = reinterpret_cast<int*>(ws) + 8;
    double* part = reinterpret_cast<double*>(ws + 256 + 64 * 128 * 8);
    T* raw = qsend;
    T* mcat = qsend + (size_t)(m - B) * B;
    T* vtop = mcat + 2 * B * B;
    T* v2top = vtop + B * B;
    T* flag = v2top + B * B;
    const size_t tot = (size_t)(m - B) * B;
    const int blocks = (int)std::min<size_t>((tot + 1023) / 1024, (size_t)4 * c->num_sms);
    if (phase == 0) {
        qr_copy_kernel<T><<<blocks, 256, 0, stream>>>(a, lda, m, B, raw);
        c->launches++;
        SVDB_CHECK(c, cudaGetLastError());
        return 0;
    }
    const GramShape g = gram_shape(m - B, c->num_sms);
    SVDB_TRY((gram_launch<T, false, B>(c, raw, (size_t)B, 0, m - B, part, g, stream)));
    auto kern = chol_algebra_kernel<T, false, B>;
    const size_t smem = chol_algebra_smem(B);
    { static bool attr_done[16] = {}; SVDB_CHECK(c, smem_attr_once(c, kern, smem, attr_done)); }
    kern<<<1, kAlgThreads, smem, stream>>>(a, lda, (const double*)nullptr, part, g.np, vtop, v2top, (size_t)B, (size_t)1, mcat, status, c->cfg.chol_guard, 1);
    c->launches++;
    qr_zero_kernel<T><<<blocks, 256, 0, stream>>>(a, lda, m, B, flag, status);
    c->launches++;
    SVDB_CHECK(c, cudaGetLastError());
    return 0;
}
template <typename T, int B>
int dist_qr_all(Ctx* c, T* qsend, int m, T* V, T* V2, cudaStream_t stream) {
    char* ws = reinterpret_cast<char*>(c->chol_ws);
    int* status = reinterpret_cast<int*>(ws) + 8;
    T* raw = qsend;
    T* mcat = qsend + (size_t)(m - B) * B;
    qr_unpack_kernel<T><<<(B * B + 255) / 256, 256, 0, stream>>>(mcat + 2 * B * B, B, V, V2, status);
    c->launches++;
    auto kern = chol_apply_kernel<T, false, B>;
    const size_t smem = chol_apply_smem(B, sizeof(T));
    { static bool attr_done[16] = {}; SVDB_CHECK(c, smem_attr_once(c, kern, smem, attr_done)); }
    const int grid = (m - B + kApplyRows - 1) / kApplyRows;
    kern<<<grid, kApplyThreads, smem, stream>>>(raw, (size_t)B, 0, m - B, mcat, V + (size_t)B * B, V2 + (size_t)B * B, (size_t)B, (size_t)1, status);
    c->launches++;
    SVDB_CHECK(c, cudaGetLastError());
    return 0;
}
}  // namespace

size_t chol_dist_qr_elems(size_t m, int b) { return (m - b) * b + 4 * (size_t)b * b + 4; }
const int* chol_dist_qr_status(Ctx* c) { return reinterpret_cast<const int*>(c->chol_ws) + 8; }
template <typename T>
int chol_dist_qr_owner(Ctx* c, T* a, size_t lda, int m, int b, T* qsend, cudaStream_t stream) {
    switch (b) {
        case 8: return dist_qr_owner<T, 8>(c, a, lda, m, qsend, stream);
        case 16: return dist_qr_owner<T, 16>(c, a, lda, m, qsend, stream);
        case 32: return dist_qr_owner<T, 32>(c, a, lda, m, qsend, stream);
        case 64: return dist_qr_owner<T, 64>(c, a, lda, m, qsend, stream);
        default: return SVDB200_E_CAPACITY;
    }
}
template <typename T>
int chol_dist_qr_owner_early(Ctx* c, T* a, size_t lda, int m, int b, T* qsend, int phase, cudaStream_t stream) {
    switch (b) {
        case 8: return dist_qr_owner_early<T, 8>(c, a, lda, m, qsend, phase, stream);
        case 16: return dist_qr_owner_early<T, 16>(c, a, lda, m, qsend, phase, stream);
        case 32: return dist_qr_owner_early<T, 32>(c, a, lda, m, qsend, phase, stream);
        case 64: return dist_qr_owner_early<T, 64>(c, a, lda, m, qsend, phase, stream);
        default: return SVDB200_E_CAPACITY;
    }
}
template int chol_dist_qr_owner_early<float>(Ctx*, float*, size_t, int, int, float*, int, cudaStream_t);
template int chol_dist_qr_owner_early<double>(Ctx*, double*, size_t, int, int, double*, int, cudaStream_t);
template <typename T>
int chol_dist_qr_all(Ctx* c, T* qsend, int m, int b, T* V, T* V2, cudaStream_t stream) {
    switch (b) {
        case 8: return dist_qr_all<T, 8>(c, qsend, m, V, V2, stream);
        case 16: return dist_qr_all<T, 16>(c, qsend, m, V, V2, stream);
        case 32: return dist_qr_all<T, 32>(c, qsend, m, V, V2, stream);
        case 64: return dist_qr_all<T, 64>(c, qsend, m, V, V2, stream);
        default: return SVDB200_E_CAPACITY;
    }
}
template int chol_dist_qr_owner<float>(Ctx*, float*, size_t, int, int, float*, cudaStream_t);
template int chol_dist_qr_owner<double>(Ctx*, double*, size_t, int, int, double*, cudaStream_t);
template int chol_dist_qr_all<float>(Ctx*, float*, int, int, float*, float*, cudaStream_t);
template int chol_dist_qr_all<double>(Ctx*, double*, int, int, double*, double*, cudaStream_t);

// panels the distributed LQ path gave up on since the handle was created (device word; the caller synchronises)
const int* chol_dist_status(Ctx* c) { return reinterpret_cast<const int*>(c->chol_ws) + 4; }

}  // namespace svdb200

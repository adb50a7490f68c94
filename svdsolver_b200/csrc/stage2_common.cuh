// Building blocks shared by the stage-2 (band -> bidiagonal) kernels: progress polling, the reference's reflector
// arithmetic (svd_serial.h:189-216, matrix.h:59-62) and the bit-faithful window product (matrix.h:243-246).
#pragma once
#include <climits>
#include "common.cuh"

namespace svdb200 {
namespace s2 {

// Thread tiling of one window product C = X * Y (nr x L times L x nc): every thread owns a 4 x 2
// register tile (rows ry + q*RT, columns cx and cx + CT).  Lanes of a warp run along the columns,
// so Y loads are conflict-free and X loads are broadcasts; odd leading dimensions keep the (at
// most two) distinct X rows of a warp in different banks.
constexpr int kTileR = 4, kTileC = 2, kNewPerThread = 4;

// Where element (r, col) of the matrix being chased lives (DESIGN §3.4c).  Dense: row-major n x n, r*n + col.  Packed:
// the 3c diagonals -(c-1) .. 2c-1 that every window of either schedule lies in, row-major with 3c entries per row,
// r*3c + col - r + c - 1.  A window row segment is contiguous in both.  kC > 0: the band as a compile-time constant.
template <bool kPacked, int kC = 0>
struct Layout {
    size_t ld;      // elements per row: n (dense) or 3c (packed)
    int c;
    __device__ __forceinline__ size_t operator()(int r, int col) const {
        if constexpr (kPacked) {
            const int cc = kC > 0 ? kC : c;
            return (size_t)r * (size_t)(3 * cc - 1) + (size_t)(col + cc - 1);      // = r*3c + (col - r + c - 1)
        } else {
            return (size_t)r * ld + col;
        }
    }
};
template <bool kPacked, int kC = 0>
__host__ __device__ __forceinline__ Layout<kPacked, kC> make_layout(int n, int c) {
    return Layout<kPacked, kC>{kPacked ? (size_t)3 * c : (size_t)n, c};
}

__host__ __device__ inline int stage2_threads(int c) {
    int ct = (c + 1) / 2;
    int need = ct * ct;                         // RIGHT: CT = RT = ceil(c/2); LEFT: CT = c, RT = ceil(c/4)
    int need_left = c * ((c + 3) / 4);
    if (need_left > need) need = need_left;
    return ((need + 31) / 32) * 32;
}

// Wait until the predecessor sweep has completed `need` window ops.  `seen` caches the last value read from its
// counter: counters only grow, so when the predecessor is already far enough ahead no memory access is needed at all
// (two L2 round trips per op otherwise).  The poll itself is an acquire load: everything the CTA reads from other
// CTAs afterwards goes through L2 (ld.global.cg), so the L1 invalidation an acquire implies costs nothing here.
__device__ __forceinline__ int wait_progress(const int* p, int need, int seen) {
    if (seen >= need) return seen;
    int v;
    unsigned polls = 0;
    unsigned long long t0 = 0;
    while ((v = ld_acquire(p)) < need) {
        __nanosleep(20);
        if ((++polls & 0xfffu) == 0u) {               // a predecessor that never advances must not hang the GPU: trap after 30 s
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            if (t0 == 0) t0 = now;
            else if (now - t0 > 30000000000ull) __trap();
        }
    }
    return v;
}

// Sequential, unfused sum of squares in index order (matrix.h:59-62) + Householder scalars.
// guard (complete schedule only): a zero vector keeps alpha = tau = 0, i.e. H = I, instead of dividing by zero
template <typename T>
__device__ __forceinline__ void reflector_scalars(const T* x, int xs, int L, T* sc, bool guard) {
    T acc = (T)0;
    int i = 0;
    for (; i + 8 <= L; i += 8) {               // the loads are independent: let them pipeline
        T v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = x[(i + u) * xs];
#pragma unroll
        for (int u = 0; u < 8; ++u) acc = RN<T>::add(acc, RN<T>::mul(v[u], v[u]));
    }
    for (; i < L; ++i) {
        T v = x[i * xs];
        acc = RN<T>::add(acc, RN<T>::mul(v, v));
    }
    T alpha, tau;
    if (guard && acc == (T)0) { alpha = (T)0; tau = (T)0; }
    else householder_scalars<T>(x[0], RN<T>::sqrt(acc), alpha, tau);
    sc[0] = alpha;
    sc[1] = tau;
}

// H = I - tau w w^T exactly as svd_serial.h:199-211 (w_0 = 1, w_i = x_i * alpha).
template <typename T>
__device__ __forceinline__ void build_h(const T* x, int xs, int L, const T* sc, T* H, int ldh, int tx, int ty, int tys) {
    const T alpha = sc[0], mtau = -sc[1];
    if (tx < L) {
        const int j = tx;
        const T wj = (j == 0) ? (T)1 : RN<T>::mul(x[j * xs], alpha);
        for (int i = ty; i < L; i += tys) {
            T wi = (i == 0) ? (T)1 : RN<T>::mul(x[i * xs], alpha);
            T h = RN<T>::mul(RN<T>::add((T)0, RN<T>::mul(wi, wj)), mtau);
            if (i == j) h = RN<T>::add((T)1, h);
            H[i * ldh + j] = h;
        }
    }
}

// out(nr x nc) = X(nr x L) * Y(L x nc), k ascending from +0, unfused (matrix.h:243-246).
// Every finished element is handed to sink(r, cc, value).
// kL > 0: the band is a compile-time constant (leading dimensions too) and interior windows have L == kL -- that case runs
// a fully unrolled loop whose shared-memory operands are base + immediate (the generic loop spends a third of its issue
// slots on address arithmetic, prof_r1_s2c).  Same products, same order, same rounding.
template <typename T, int kL, typename Sink>
__device__ __forceinline__ void window_product(const T* X, int ldx, const T* Y, int ldy, int nr, int nc, int L, int CT, int RT,
                                               Sink sink, int tid) {
    const int cx = tid % CT, ry = tid / CT;
    if (ry >= RT) return;
    T acc[kTileR][kTileC];
#pragma unroll
    for (int q = 0; q < kTileR; ++q)
#pragma unroll
        for (int s2 = 0; s2 < kTileC; ++s2) acc[q][s2] = (T)0;
    int xr[kTileR];
#pragma unroll
    for (int q = 0; q < kTileR; ++q) xr[q] = min(ry + q * RT, nr - 1) * ldx;
    const int y0 = min(cx, nc - 1), y1 = min(cx + CT, nc - 1);
    if (kL > 0 && L == kL) {
        const T* Y0 = Y + y0;
        const T* Y1 = Y + y1;
        const T* Xq[kTileR];
#pragma unroll
        for (int q = 0; q < kTileR; ++q) Xq[q] = X + xr[q];
#pragma unroll
        for (int k = 0; k < (kL > 0 ? kL : 1); k += 4) {
            T yv[4][2], xv[4][kTileR];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                yv[u][0] = Y0[(k + u) * ldy];
                yv[u][1] = Y1[(k + u) * ldy];
#pragma unroll
                for (int q = 0; q < kTileR; ++q) xv[u][q] = Xq[q][k + u];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int q = 0; q < kTileR; ++q) {
                    acc[q][0] = RN<T>::add(acc[q][0], RN<T>::mul(xv[u][q], yv[u][0]));
                    acc[q][1] = RN<T>::add(acc[q][1], RN<T>::mul(xv[u][q], yv[u][1]));
                }
        }
    } else {
        int k = 0;
        for (; k + 4 <= L; k += 4) {               // operands of 4 steps are fetched before they are consumed
            T yv[4][2], xv[4][kTileR];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                yv[u][0] = Y[(k + u) * ldy + y0];
                yv[u][1] = Y[(k + u) * ldy + y1];
#pragma unroll
                for (int q = 0; q < kTileR; ++q) xv[u][q] = X[xr[q] + k + u];
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
#pragma unroll
                for (int q = 0; q < kTileR; ++q) {
                    acc[q][0] = RN<T>::add(acc[q][0], RN<T>::mul(xv[u][q], yv[u][0]));
                    acc[q][1] = RN<T>::add(acc[q][1], RN<T>::mul(xv[u][q], yv[u][1]));
                }
        }
        for (; k < L; ++k) {
            const T yv0 = Y[k * ldy + y0], yv1 = Y[k * ldy + y1];
#pragma unroll
            for (int q = 0; q < kTileR; ++q) {
                const T xv = X[xr[q] + k];
                acc[q][0] = RN<T>::add(acc[q][0], RN<T>::mul(xv, yv0));
                acc[q][1] = RN<T>::add(acc[q][1], RN<T>::mul(xv, yv1));
            }
        }
    }
#pragma unroll
    for (int q = 0; q < kTileR; ++q) {
        const int r = ry + q * RT;
        if (r < nr) {
            if (cx < nc) sink(r, cx, acc[q][0]);
            if (cx + CT < nc) sink(r, cx + CT, acc[q][1]);
        }
    }
}


}  // namespace s2
}  // namespace svdb200

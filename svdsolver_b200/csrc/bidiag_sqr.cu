// Implicit SHIFTED QR for the singular values of the bidiagonal (SURVEY 8f rank 3, north star: "GPU implicit-shift kernel").
// The reference's serial::qrd (svd_serial.h:368-422) is the zero-shift iteration only (impl_zero_shift, 314-333), float
// only, and converges linearly; this kernel runs Golub-Kahan SVD steps with shifts (sqr_core.h: LAPACK dbdsqr's shifted
// top-to-bottom chase) in double arithmetic for both element types.
//
// A QR sweep is a sequential recurrence along the diagonal; what can overlap are CONSECUTIVE sweeps (sweep s+1 may work on
// position i once sweep s has finished position i+2), provided their shifts are known when they start at the top.  One
// warp therefore pipelines up to kLanes sweeps per pass -- lane l at position lo + t - 3 l, __syncwarp per step -- whose
// shifts are the smallest singular values of the trailing block of the window (bisection on 2 kLanes entries, one shift
// per lane): the small-bulge multishift form of the iteration.  A sweep that makes the last off-diagonal entry negligible
// deflates it at once and publishes the new bottom to the sweeps behind it.  Between passes: negligible entries are
// zeroed, the bottom unreduced window is located with ballots, zero diagonal entries are rotated out (they split B).
// Measured convergence (tests/test_sqr_cpu.py, the same core on the host): ~1.2 n passes and 2-4 n sweeps in total, against
// ~n log(1/tol) SWEEPS PER VALUE for the zero-shift iteration.  Bisection (bidiag_bisect.cu) stays the solver for large n:
// it is embarrassingly parallel, this iteration is not.
#include "common.cuh"
#include "sqr_core.h"

namespace svdb200 {
namespace {

constexpr int kLanes = 8;                 // sweeps in flight (a pass deflates ~1 value: more lanes only add wasted sweeps)
constexpr double kTol = 8.881784197001252e-16;   // 8 eps: a sweep leaves O(eps) noise in e, a tighter test never settles

template <typename T>
__device__ void warp_sort_desc(T* v, int npad) {
    for (int k = 2; k <= npad; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < npad; i += 32) {
                int ixj = i ^ j;
                if (ixj > i) {
                    T a = v[i], b = v[ixj];
                    bool desc = ((i & k) == 0);
                    if (desc ? (a < b) : (a > b)) { v[i] = b; v[ixj] = a; }
                }
            }
            __syncwarp();
        }
}

// info[0] = sweeps, info[1] = status (0 ok, 1 sweep budget exhausted), info[2] = passes
template <typename T, bool kSmem>
__global__ void __launch_bounds__(32, 1)
bidiag_sqr_kernel(T* __restrict__ d_g, T* __restrict__ e_g, int n, T* __restrict__ sigma, T* __restrict__ sortbuf, int npad,
                  long long* __restrict__ info, double* __restrict__ ws) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ double z2[4 * kLanes];
    __shared__ double mu_s[kLanes];
    __shared__ int bot_s;
    // the iteration runs on a DOUBLE copy of the bidiagonal for both element types (float storage would round d / e after
    // each of the ~3 n sweeps): shared memory up to n = 12800, a global workspace above
    double* d = kSmem ? reinterpret_cast<double*>(smem_raw) : ws;
    double* e = d + n;
    const int lane = threadIdx.x;
    for (int i = lane; i < n; i += 32) d[i] = (double)d_g[i];
    for (int i = lane; i < n - 1; i += 32) e[i] = (double)e_g[i];
    __syncwarp();
    long long sweeps = 0, passes = 0;
    const long long max_sweeps = 60LL * n + 1000;
    int hi = n - 1, status = 0;
    while (hi > 0) {
        if (sweeps >= max_sweeps) { status = 1; break; }
        // ---- bottom of the unreduced part: skip zero / negligible entries upwards --------------------------------
        while (hi > 0) {
            const int i = hi - 1 - lane;
            bool neg = true;
            if (i >= 0) {
                const double ei = e[i];
                neg = (ei == 0.0) || sqr_negligible(ei, d[i], d[i + 1], kTol);
                if (neg && ei != 0.0) e[i] = 0.0;
            }
            const unsigned m = __ballot_sync(0xffffffffu, !neg && i >= 0);
            if (m != 0u) { hi -= __ffs(m) - 1; break; }
            hi -= 32;
        }
        __syncwarp();
        if (hi <= 0) break;
        // ---- top of the window: first zero / negligible entry above hi-1 -----------------------------------------------
        int lo = hi - 1;
        while (lo > 0) {
            const int i = lo - 1 - lane;
            bool neg = true;
            if (i >= 0) {
                const double ei = e[i];
                neg = (ei == 0.0) || sqr_negligible(ei, d[i], d[i + 1], kTol);
                if (neg && ei != 0.0) e[i] = 0.0;
            }
            const unsigned m = __ballot_sync(0xffffffffu, neg || i < 0);
            if (m != 0u) { lo -= __ffs(m) - 1; break; }
            lo -= 32;
        }
        if (lo < 0) lo = 0;
        __syncwarp();
        const int nd = hi - lo + 1;
        // ---- zero diagonal entries split the window ------------------------------------------------------------------------
        double dmax = 0.0;
        for (int i = lo + lane; i <= hi; i += 32) dmax = fmax(dmax, fabs(d[i]));
        for (int o = 16; o > 0; o >>= 1) dmax = fmax(dmax, __shfl_xor_sync(0xffffffffu, dmax, o));
        bool zero_here = false;
        for (int i = lo + lane; i <= hi; i += 32) zero_here |= fabs(d[i]) <= kTol * dmax;
        if (__any_sync(0xffffffffu, zero_here)) {
            if (lane == 0) {
                for (int i = lo; i <= hi; ++i)
                    if (fabs(d[i]) <= kTol * dmax) {
                        d[i] = 0.0;
                        if (i < hi) sqr_chase_zero_row(d, e, i, hi);
                        else sqr_chase_zero_col(d, e, lo, hi);
                    }
            }
            __syncwarp();
            ++passes;
            continue;
        }
        // ---- shifts: the cnt smallest singular values of the trailing blk x blk block (never the whole spectrum of the
        // window: prod (B^T B - mu_k^2) must not vanish) -------------------------------------------------------------------
        const int cnt = min(kLanes, max(1, nd / 2));
        const int blk = min(nd, 2 * cnt);
        double bound = 0.0;
        if (lane == 0) {
            bound = sqr_fill_z2(d, e, hi - blk + 1, blk, z2);
            bot_s = hi;
        }
        bound = __shfl_sync(0xffffffffu, bound, 0);
        __syncwarp();
        if (lane < cnt) mu_s[lane] = bound > 0.0 ? bisect_kth(z2, blk, lane, 60, 4.5e-16) * bound : 0.0;
        __syncwarp();
        // ---- the pipelined sweeps ---------------------------------------------------------------------------------------------
        SqrCarry car = {0.0, 0.0};
        bool running = lane < cnt;
        const int steps = (hi - lo) + 3 * (cnt - 1);
        for (int t = 0; t < steps; ++t) {
            const int pos = lo + t - 3 * lane;
            const int bot = bot_s;
            if (running && pos >= lo) {
                if (pos >= bot || bot <= lo) {
                    running = false;                           // the window ended above this sweep's next position
                } else {
                    if (pos == lo) car = sqr_start(d[lo], e[lo], mu_s[lane]);
                    sqr_position(d, e, pos, lo, bot, car);
                    if (pos == bot - 1) {                      // finished: deflate the bottom entry if it converged
                        running = false;
                        if (sqr_negligible(e[bot - 1], d[bot - 1], d[bot], kTol)) { e[bot - 1] = 0.0; bot_s = bot - 1; }
                    }
                }
            }
            __syncwarp();
        }
        sweeps += cnt;
        ++passes;
    }
    __syncwarp();
    for (int i = lane; i < npad; i += 32) sortbuf[i] = (i < n) ? (T)fabs(d[i]) : (T)-1;
    __syncwarp();
    warp_sort_desc<T>(sortbuf, npad);
    for (int i = lane; i < n; i += 32) sigma[i] = sortbuf[i];
    for (int i = lane; i < n; i += 32) d_g[i] = (T)d[i];
    for (int i = lane; i < n - 1; i += 32) e_g[i] = (T)e[i];
    if (lane == 0 && info) { info[0] = sweeps; info[1] = status; info[2] = passes; }
}

}  // namespace

template <typename T>
int bidiag_sqr(Ctx* c, T* d, T* e, size_t n, T* sigma) {
    if (n < 2) return SVDB200_E_SHAPE;
    if (n > c->max_n) return SVDB200_E_CAPACITY;
    int npad = 1;
    while ((size_t)npad < n) npad <<= 1;
    if (c->wpart_elems < (size_t)npad) return SVDB200_E_CAPACITY;
    T* sortbuf = reinterpret_cast<T*>(c->wpart);
    const size_t smem = 2 * n * sizeof(double);
    int ni = (int)n;
    if (smem <= 200 * 1024) {
        auto kern = bidiag_sqr_kernel<T, true>;
        SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<1, 32, smem, c->stream>>>(d, e, ni, sigma, sortbuf, npad, c->qr_info, (double*)nullptr);
    } else {
        SVDB_TRY(reserve(c, c->bis_ws, sizeof(double) * (2 * c->max_n + 24)));   // double workspace shared with the bisection solver
        auto kern = bidiag_sqr_kernel<T, false>;
        kern<<<1, 32, 0, c->stream>>>(d, e, ni, sigma, sortbuf, npad, c->qr_info, reinterpret_cast<double*>(c->bis_ws.p));
    }
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    return 0;
}
template int bidiag_sqr<float>(Ctx*, float*, float*, size_t, float*);
template int bidiag_sqr<double>(Ctx*, double*, double*, size_t, double*);

}  // namespace svdb200

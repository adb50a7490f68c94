// QR diagonalisation of the bidiagonal.  Replaces csc586::serial::qrd<T> (svd_serial.h:368-422):
// Demmel-Kahan implicit zero-shift QR sweeps (impl_zero_shift, 314-333; rotate, 278-297) with the
// reference's convergence criteria (Criteria<T>, 138-166) and its deflation-from-both-ends driver;
// |d| sorted descending at the end (403-405).
//
// B200 design: a zero-shift sweep is a strictly sequential recurrence along the diagonal, but
// consecutive sweeps only need a distance of two positions (sweep s+1 at position k needs sweep s
// to have finished position k+1).  The kernel therefore runs up to blockDim.x sweeps concurrently
// as a software wavefront: lane l executes position (t - 2l) at time step t, d/e live in shared
// memory (global/L2 when n is too large), one __syncthreads per time step.  The deflation window
// [i_low, i_up] is re-evaluated between wavefront passes with the reference's own scan; every
// sweep is an exact orthogonal zero-shift QR sweep on a window that contains the reference's
// window, so sigma agrees with serial::qrd to the convergence threshold (not bit-for-bit: the
// number of sweeps per window differs).
#include "common.cuh"

namespace svdb200 {
namespace {

template <typename T> struct Rot { T c, s, r; };

// svd_serial.h:278-297
template <typename T>
__device__ __forceinline__ Rot<T> rotate(T u1, T u2) {
    Rot<T> p;
    if (u1 == (T)0) {
        p.c = (T)0; p.s = (T)1; p.r = u2;
    } else if (RN<T>::abs(u1) > RN<T>::abs(u2)) {
        T t1 = u2 / u1, t2 = RN<T>::sqrt((T)1 + t1 * t1), t3 = (T)1 / t2;
        p.c = t3; p.s = t1 * t3; p.r = u1 * t2;
    } else {
        T t1 = u1 / u2, t2 = RN<T>::sqrt((T)1 + t1 * t1), t3 = (T)1 / t2;
        p.c = t1 * t3; p.s = t3; p.r = u2 * t2;
    }
    return p;
}

template <typename T>
__device__ void bitonic_sort_desc(T* v, int npad) {
    for (int k = 2; k <= npad; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < npad; i += blockDim.x) {
                int ixj = i ^ j;
                if (ixj > i) {
                    T a = v[i], b = v[ixj];
                    bool desc = ((i & k) == 0);
                    if (desc ? (a < b) : (a > b)) { v[i] = b; v[ixj] = a; }
                }
            }
            __syncthreads();
        }
}

// info[0] = sweeps run, info[1] = status (0 ok, 1 max_iter reached), info[2] = passes
template <typename T, bool kSmem>
__global__ void __launch_bounds__(1024, 1)
bidiag_qr_kernel(T* __restrict__ d_g, T* __restrict__ e_g, int n, T* __restrict__ sigma, T* __restrict__ sortbuf,
                 int npad, long long* __restrict__ info) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int sh_low, sh_up, sh_done;
    __shared__ T sh_thr;
    T* d = kSmem ? reinterpret_cast<T*>(smem_raw) : d_g;
    T* e = kSmem ? d + n : e_g;
    const int tid = threadIdx.x, P = blockDim.x;
    if (kSmem) {
        for (int i = tid; i < n; i += P) d[i] = d_g[i];
        for (int i = tid; i < n - 1; i += P) e[i] = e_g[i];
        __syncthreads();
    }
    const unsigned long long max_iter_ref = (500ull * (unsigned long long)n) ^ 2ull;   // svd_serial.h:164 ('^' is XOR)
    // sweep budget: the reference's for float; 64x for double (tighter threshold => more sweeps)
    const unsigned long long max_iter = sizeof(T) == 4 ? max_iter_ref : 64ull * max_iter_ref;
    if (tid == 0) {
        // Criteria<T>::init (svd_serial.h:146-166); sigma[] doubles as scratch for lambda.
        // float: the reference's constants (eps 1e-8, umin 1e-10).  double: the reference does not
        // compile for double; its float-calibrated constants would cap the accuracy near 1e-7*sigma_1,
        // above the 1e-10 bar, so the double instantiation scales them (eps 1e-16, umin 1e-17).
        T eps = sizeof(T) == 4 ? (T)1e-8 : (T)1e-16, umin = sizeof(T) == 4 ? (T)1e-10 : (T)1e-17, tol = (T)100 * eps;
        T lam = RN<T>::abs(d[n - 1]), lmin = lam;
        for (int j = n - 2; j >= 0; --j) {
            lam = RN<T>::abs(d[j]) * lam / (lam + RN<T>::abs(e[j]));
            lmin = lam < lmin ? lam : lmin;
        }
        T mu = RN<T>::abs(d[0]), mmin = mu;
        for (int j = 0; j < n - 1; ++j) {
            mu = RN<T>::abs(d[j + 1]) * mu / (mu + RN<T>::abs(e[j]));
            mmin = mu < mmin ? mu : mmin;
        }
        T lb = lmin < mmin ? lmin : mmin;
        T a = tol * lb, b = (T)max_iter_ref * umin;
        sh_thr = a < b ? b : a;
        sh_low = 0;
        sh_up = n - 2;
        sh_done = 0;
    }
    __syncthreads();
    const T thr = sh_thr;
    unsigned long long iter = 0;
    long long passes = 0;
    int status = 0;
    int want = 32, prev_lo = -1, prev_up = -1;       // sweeps per pass adapt to the deflation rate
    while (true) {
        if (tid == 0) {
            // svd_serial.h:386-407
            int i_up = sh_up, i_low = sh_low;
            for (int i = i_up; i >= 1; --i) { i_up = i; if (RN<T>::abs(e[i]) > thr) break; }
            int j = i_up;
            for (int i = i_low; i < i_up; ++i) if (RN<T>::abs(e[i]) > thr) { j = i; break; }
            i_low = j;
            sh_up = i_up; sh_low = i_low;
            sh_done = ((i_up == i_low && RN<T>::abs(e[i_up]) <= thr) || (i_up < i_low)) ? 1 : 0;
        }
        __syncthreads();
        if (sh_done) break;
        if (iter >= max_iter) { status = 1; break; }
        const int lo = sh_low, nd = sh_up - sh_low + 2;   // window d[lo .. lo+nd-1], e[lo .. lo+nd-2]
        // A pass that ended without deflation doubles the number of pipelined sweeps, a deflation
        // halves it: no long runs of sweeps on an already converged window, and few passes when
        // convergence is slow.
        if (sh_low == prev_lo && sh_up == prev_up) want = want * 2 > P ? P : want * 2;
        else want = want / 2 < 32 ? 32 : want / 2;
        prev_lo = sh_low; prev_up = sh_up;
        int lanes = want < P ? want : P;
        if ((unsigned long long)lanes > max_iter - iter) lanes = (int)(max_iter - iter);
        T* dd = d + lo;
        T* ee = e + lo;
        Rot<T> rot = {(T)1, (T)0, (T)0}, rot_ = {(T)1, (T)0, (T)0};
        const int steps = nd + 2 * (lanes - 1);
        for (int t = 0; t < steps; ++t) {
            int k = t - 2 * tid;
            if (tid < lanes && k >= 0 && k < nd) {
                if (k < nd - 1) {                       // svd_serial.h:319-327
                    rot = rotate<T>(rot.c * dd[k], ee[k]);
                    if (k > 0) ee[k - 1] = rot.r * rot_.s;
                    rot_ = rotate<T>(rot_.c * rot.r, dd[k + 1] * rot.s);
                    dd[k] = rot_.r;
                } else {                                // svd_serial.h:329-331
                    T h = rot.c * dd[nd - 1];
                    ee[nd - 2] = h * rot_.s;
                    dd[nd - 1] = h * rot_.c;
                }
            }
            __syncthreads();
        }
        iter += (unsigned long long)lanes;
        ++passes;
    }
    // |d| sorted descending (svd_serial.h:403-405)
    for (int i = tid; i < npad; i += P) sortbuf[i] = (i < n) ? RN<T>::abs(d[i]) : (T)-1;
    __syncthreads();
    bitonic_sort_desc<T>(sortbuf, npad);
    for (int i = tid; i < n; i += P) sigma[i] = sortbuf[i];
    if (kSmem) {
        for (int i = tid; i < n; i += P) d_g[i] = d[i];
        for (int i = tid; i < n - 1; i += P) e_g[i] = e[i];
    }
    if (tid == 0 && info) { info[0] = (long long)iter; info[1] = status; info[2] = passes; }
}

}  // namespace

template <typename T>
int bidiag_qr(Ctx* c, T* d, T* e, size_t n, T* sigma) {
    if (n < 2) return SVDB200_E_SHAPE;
    if (n > c->max_n) return SVDB200_E_CAPACITY;
    ProfScope ps(c, 5, (double)n);
    // zero-shift QR needs ~n log(1/tol) sweeps: beyond a moderate n the independent-per-value bisection
    // solver (bidiag_bisect.cu) takes over
    if (c->cfg.qr_method == 2 || (c->cfg.qr_method == 0 && n > c->cfg.qr_auto_limit)) return bidiag_bisect<T>(c, d, e, n, sigma);
    if (c->cfg.qr_method == 3) return bidiag_sqr<T>(c, d, e, n, sigma);      // implicit shifted QR (bidiag_sqr.cu)
    int npad = 1;
    while ((size_t)npad < n) npad <<= 1;
    // sort buffer: reuse the stage-2 progress array region is int-sized; use wpart (>= 2*max_n elems)
    if (c->wpart_elems < (size_t)npad) return SVDB200_E_CAPACITY;
    T* sortbuf = reinterpret_cast<T*>(c->wpart);
    size_t smem = 2 * n * sizeof(T);
    int nt = 1024;
    if (n < 512) nt = (int)((n + 31) / 32) * 32 * 2;
    if (nt > 1024) nt = 1024;
    if (nt < 64) nt = 64;
    int ni = (int)n;
    if (smem <= 200 * 1024) {
        auto kern = bidiag_qr_kernel<T, true>;
        SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<1, nt, smem, c->stream>>>(d, e, ni, sigma, sortbuf, npad, c->qr_info);
    } else {
        auto kern = bidiag_qr_kernel<T, false>;
        kern<<<1, nt, 0, c->stream>>>(d, e, ni, sigma, sortbuf, npad, c->qr_info);
    }
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    return 0;
}

template int bidiag_qr<float>(Ctx*, float*, float*, size_t, float*);
template int bidiag_qr<double>(Ctx*, double*, double*, size_t, double*);

}  // namespace svdb200

// Singular values of the bidiagonal by bisection on the Golub-Kahan form: the scalable replacement for the
// QR diagonalisation (csc586::serial::qrd, svd_serial.h:368-422) at sizes where zero-shift QR sweeps are
// hopeless (zero-shift QR converges linearly: ~n log(1/tol) sweeps of n dependent rotations; at n = 16384
// in double the wavefront kernel of bidiag_qr.cu needs 107 s, this kernel tens of milliseconds).
//
// Every singular value is independent: thread k brackets the k-th smallest sigma with Sturm counts
// (bisect_core.h: three-term Sturm sequence of the Golub-Kahan tridiagonal, one FMA per step on the
// dependent chain, all lanes of a warp read the same z^2 element -> broadcast loads), in double for both
// element types.  Accuracy: backward stable in the entries of B (relative perturbations of a few ulp), so
// sigma is accurate to ~1e-15 sigma_max; output is sorted descending by construction (no sort pass).
#include <algorithm>
#include "bisect_core.h"
#include "common.cuh"

namespace svdb200 {
namespace {

// one block: ||B|| bound, scaled + floored squares of the off-diagonals, status words
template <typename T>
__global__ void __launch_bounds__(1024)
bisect_prep_kernel(const T* __restrict__ d, const T* __restrict__ e, int n, double* __restrict__ z2, double* __restrict__ params,
                   long long* __restrict__ info) {
    __shared__ double red[32];
    __shared__ double s_bound;
    // batched: one matrix per block; d / e rows of length n, z2 rows of length 2n, 8 params per matrix
    d += (size_t)blockIdx.x * n; e += (size_t)blockIdx.x * n;
    z2 += (size_t)blockIdx.x * 2 * n; params += (size_t)blockIdx.x * 8;
    double mx = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double di = fabs((double)d[i]);
        const double er = i < n - 1 ? fabs((double)e[i]) : 0.0;
        const double el = i > 0 ? fabs((double)e[i - 1]) : 0.0;
        mx = fmax(mx, di + fmax(er, el));                // max(||B||_1, ||B||_inf) >= ||B||_2
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
        if (threadIdx.x == 0) {
            s_bound = v;
            params[0] = v;
            info[0] = 0; info[1] = 0; info[2] = 0;
        }
    }
    __syncthreads();
    const double bound = s_bound;
    const double inv = bound > 0.0 ? 1.0 / bound : 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double a = (double)d[i] * inv;
        z2[2 * i] = fmax(a * a, kBisZ2Floor);
        if (i < n - 1) {
            double b = (double)e[i] * inv;
            z2[2 * i + 1] = fmax(b * b, kBisZ2Floor);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(64)
bisect_kernel(const double* __restrict__ z2, int n, const double* __restrict__ params, T* __restrict__ sigma, double rel_tol) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    z2 += (size_t)blockIdx.y * 2 * n; params += (size_t)blockIdx.y * 8; sigma += (size_t)blockIdx.y * n;
    const double bound = params[0];
    double s = 0.0;
    if (bound > 0.0) s = bisect_kth(z2, n, k, 200, rel_tol) * bound;
    sigma[n - 1 - k] = (T)s;
}

}  // namespace

// count > 1: d, e, sigma are count rows of length n (the batched small-matrix driver)
template <typename T>
int bidiag_bisect_batched(Ctx* c, const T* d, const T* e, size_t n, T* sigma, int count) {
    if (n < 1 || count < 1 || count > 65535) return SVDB200_E_SHAPE;
    const size_t need = (size_t)count * (2 * n + 8) + 16;
    SVDB_TRY(reserve(c, c->bis_ws, sizeof(double) * std::max(need, (size_t)(2 * c->max_n + 24))));
    double* params = reinterpret_cast<double*>(c->bis_ws.p);
    double* z2 = params + 8 * (size_t)count;
    const int ni = (int)n;
    bisect_prep_kernel<T><<<count, 1024, 0, c->stream>>>(d, e, ni, z2, params, c->qr_info);
    SVDB_CHECK(c, cudaGetLastError());
    const double rel_tol = sizeof(T) == 8 ? 4.440892098500626e-16 : 1.4901161193847656e-08;   // 2 eps(double) / 2^-26
    bisect_kernel<T><<<dim3((ni + 63) / 64, count), 64, 0, c->stream>>>(z2, ni, params, sigma, rel_tol);
    SVDB_CHECK(c, cudaGetLastError());
    c->launches += 2;
    return 0;
}

template <typename T>
int bidiag_bisect(Ctx* c, const T* d, const T* e, size_t n, T* sigma) {
    if (n > c->max_n) return SVDB200_E_CAPACITY;
    return bidiag_bisect_batched<T>(c, d, e, n, sigma, 1);
}

template int bidiag_bisect_batched<float>(Ctx*, const float*, const float*, size_t, float*, int);
template int bidiag_bisect_batched<double>(Ctx*, const double*, const double*, size_t, double*, int);
template int bidiag_bisect<float>(Ctx*, const float*, const float*, size_t, float*);
template int bidiag_bisect<double>(Ctx*, const double*, const double*, size_t, double*);

}  // namespace svdb200

// Transpose of a row-major matrix on the device: a wide m x n matrix (m < n) is reduced as its tall transpose
// (run_chain, capi.cu), so that sigma(A) = sigma(A^T) and the result, transposed back, is LAPACK gebrd's lower form.
#include <algorithm>
#include "common.cuh"

namespace svdb200 {
namespace {

constexpr int kTile = 32;
constexpr int kTileRows = 8;

// dst (cols x rows) = src (rows x cols)^T, both row-major, for matrix blockIdx.z of a batch (sS / sD elements between
// consecutive sources / destinations).  One 32 x 32 tile per CTA through shared memory with a padded stride (no bank
// conflicts on the transposed read); reads and writes are both along rows of 32 consecutive elements.
template <typename T>
__global__ void __launch_bounds__(kTile * kTileRows)
transpose_kernel(const T* __restrict__ src, size_t sS, size_t rows, size_t cols, T* __restrict__ dst, size_t sD) {
    __shared__ T tile[kTile][kTile + 1];
    src += (size_t)blockIdx.z * sS;
    dst += (size_t)blockIdx.z * sD;
    const size_t r0 = (size_t)blockIdx.y * kTile, c0 = (size_t)blockIdx.x * kTile;
    const int tx = threadIdx.x, ty = threadIdx.y;
#pragma unroll
    for (int i = ty; i < kTile; i += kTileRows) {
        const size_t r = r0 + i, c = c0 + tx;
        if (r < rows && c < cols) tile[i][tx] = src[r * cols + c];
    }
    __syncthreads();
#pragma unroll
    for (int i = ty; i < kTile; i += kTileRows) {
        const size_t r = c0 + i, c = r0 + tx;          // row of dst = column of src
        if (r < cols && c < rows) dst[r * rows + c] = tile[tx][i];
    }
}

}  // namespace

// dst[z] = src[z]^T for z < count: src[z] = src + z sS (rows x cols), dst[z] = dst + z sD (cols x rows)
template <typename T>
int transpose_batched(Ctx* c, const T* src, size_t sS, size_t rows, size_t cols, T* dst, size_t sD, size_t count) {
    for (size_t z0 = 0; z0 < count; z0 += 32768) {
        const unsigned zc = (unsigned)std::min<size_t>(32768, count - z0);
        const dim3 grid((unsigned)((cols + kTile - 1) / kTile), (unsigned)((rows + kTile - 1) / kTile), zc);
        transpose_kernel<T><<<grid, dim3(kTile, kTileRows), 0, c->stream>>>(src + z0 * sS, sS, rows, cols, dst + z0 * sD, sD);
        SVDB_CHECK(c, cudaGetLastError());
        c->launches++;
    }
    return 0;
}

template <typename T>
int transpose(Ctx* c, const T* src, size_t rows, size_t cols, T* dst) { return transpose_batched<T>(c, src, 0, rows, cols, dst, 0, 1); }

template int transpose_batched<float>(Ctx*, const float*, size_t, size_t, size_t, float*, size_t, size_t);
template int transpose_batched<double>(Ctx*, const double*, size_t, size_t, size_t, double*, size_t, size_t);
template int transpose<float>(Ctx*, const float*, size_t, size_t, float*);
template int transpose<double>(Ctx*, const double*, size_t, size_t, double*);

}  // namespace svdb200

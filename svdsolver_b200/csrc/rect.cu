// Transpose of a row-major matrix on the device: a wide m x n matrix (m < n) is reduced as its tall transpose
// (run_chain, capi.cu), so that sigma(A) = sigma(A^T) and the result, transposed back, is LAPACK gebrd's lower form.
#include "common.cuh"

namespace svdb200 {
namespace {

constexpr int kTile = 32;
constexpr int kTileRows = 8;

// dst (cols x rows) = src (rows x cols)^T, both row-major.  One 32 x 32 tile per CTA through shared
// memory with a padded stride (no bank conflicts on the transposed read); reads and writes are both
// along rows of 32 consecutive elements.
template <typename T>
__global__ void __launch_bounds__(kTile * kTileRows)
transpose_kernel(const T* __restrict__ src, size_t rows, size_t cols, T* __restrict__ dst) {
    __shared__ T tile[kTile][kTile + 1];
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

template <typename T>
int transpose(Ctx* c, const T* src, size_t rows, size_t cols, T* dst) {
    const dim3 grid((unsigned)((cols + kTile - 1) / kTile), (unsigned)((rows + kTile - 1) / kTile));
    transpose_kernel<T><<<grid, dim3(kTile, kTileRows), 0, c->stream>>>(src, rows, cols, dst);
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    return 0;
}

template int transpose<float>(Ctx*, const float*, size_t, size_t, float*);
template int transpose<double>(Ctx*, const double*, size_t, size_t, double*);

}  // namespace svdb200

// Rectangular m x n matrices through the panel-order reduction.
//
// Tall (m >= n): stage 1 runs in place on the m x n array (stage1_panel_order with rows = m); the
// top n x n block is then upper band, the rows below it zero, and stage 2 / the singular values run
// on that block (contiguous, ld = n) exactly as for a square matrix.
// Wide (m < n): sigma(A) = sigma(A^T).  A is transposed into the handle's scratch buffer (n x m,
// tall), reduced there, and the result is transposed back, so that `a` holds a LOWER band /
// bidiagonal matrix in its left m x m block (LAPACK gebrd's convention for m < n) and zeros right
// of it; e is then the sub-diagonal.
#include <algorithm>
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

template <typename T>
int transpose(Ctx* c, const T* src, size_t rows, size_t cols, T* dst) {
    const dim3 grid((unsigned)((cols + kTile - 1) / kTile), (unsigned)((rows + kTile - 1) / kTile));
    transpose_kernel<T><<<grid, dim3(kTile, kTileRows), 0, c->stream>>>(src, rows, cols, dst);
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    return 0;
}

// Scratch for A^T: allocated on the first wide call with that call's size, grown (never shrunk) when a
// larger wide matrix arrives; freed by svdb200_destroy.
int ensure_rect_ws(Ctx* c, size_t elems) {
    if (c->rect_ws_elems >= elems) return 0;
    if (c->rect_ws) {
        SVDB_CHECK(c, cudaStreamSynchronize(c->stream));   // earlier calls on this handle may still read it
        SVDB_CHECK(c, cudaFree(c->rect_ws));
        c->rect_ws = nullptr;
        c->rect_ws_elems = 0;
    }
    SVDB_CHECK(c, cudaMalloc(&c->rect_ws, c->esz * elems));
    c->rect_ws_elems = elems;
    return 0;
}

}  // namespace

// what: 1 = stage 1 (a -> band), 3 = + stage 2 (d, e: min(m, n) and min - 1 entries), 7 = + singular values (sigma, on
// d / e).  marks (optional, 4 events) are recorded after stage 1 (forward transpose included), after stage 2, after the
// singular values and after the transpose back.  Shapes are checked by the caller.
template <typename T>
int rect_chain(Ctx* c, T* a, size_t m, size_t n, size_t band, int what, T* d, T* e, T* sigma, cudaEvent_t* marks) {
    const bool wide = m < n;
    const size_t k = std::min(m, n);
    T* x = a;
    if (wide) {
        SVDB_TRY(ensure_rect_ws(c, m * n));
        x = reinterpret_cast<T*>(c->rect_ws);
        SVDB_TRY(transpose<T>(c, a, m, n, x));             // x = A^T: n x m, tall
    }
    SVDB_TRY(stage1_panel_order<T>(c, x, std::max(m, n), k, band));
    if (marks) SVDB_CHECK(c, cudaEventRecord(marks[0], c->stream));
    if (what & 2) SVDB_TRY(stage2_chase<T>(c, x, k, band, d, e));
    if (marks) SVDB_CHECK(c, cudaEventRecord(marks[1], c->stream));
    if (what & 4) SVDB_TRY(bidiag_qr<T>(c, d, e, k, sigma));
    if (marks) SVDB_CHECK(c, cudaEventRecord(marks[2], c->stream));
    if (wide) SVDB_TRY(transpose<T>(c, x, n, m, a));
    if (marks) SVDB_CHECK(c, cudaEventRecord(marks[3], c->stream));
    return 0;
}

template int rect_chain<float>(Ctx*, float*, size_t, size_t, size_t, int, float*, float*, float*, cudaEvent_t*);
template int rect_chain<double>(Ctx*, double*, size_t, size_t, size_t, int, double*, double*, double*, cudaEvent_t*);

}  // namespace svdb200

/* svdb200.h -- C ABI of the B200-native SVDSolver hot path
 * (dense -> band -> bidiagonal -> singular values; float and double).
 *
 * The reference (scrose/SVDSolver) has no FFI layer: its boundary is the C++ function level
 * (SURVEY 8b).  Each entry point below names the reference function it replaces (file:line under
 * the reference tree); include/svdb200_matrix.hpp carries the source-compatible C++ adapters
 * (csc586::gpu::cuda_brd_p1, csc586::parallel::brd_p1/brd_p2, csc586::serial::qrd) on top of it.
 *
 * Conventions
 *   - matrices are square n x n, dense ROW-MAJOR (what Matrix::flatten() yields, matrix.h:258,
 *     svd_cuda_2.cu:549), band | n, updated in place unless stated; the *_mn calls take
 *     rectangular m x n matrices (band | min(m, n));
 *   - every function returns an int status: 0 ok, <0 argument/shape error (SVDB200_E_*),
 *     >0 a CUDA / NCCL error code offset by SVDB200_CUDA_ERR / SVDB200_NCCL_ERR;
 *     no exceptions cross this boundary (the reference assert()s and ignores CUDA errors);
 *   - the caller owns host buffers; the handle owns a reusable device workspace and one stream;
 *     one handle per host thread / GPU, re-entrant across handles;
 *   - "_dev" variants take device pointers (inputs already resident in HBM) and enqueue on the
 *     handle's stream without synchronising; host-pointer variants copy H2D/D2H inside the call
 *     and return after completion, like the reference's timed region (timing.h:78-83).
 *   - there is NO CPU fallback: without a CUDA device every compute call fails with a status.
 */
#ifndef SVDB200_H
#define SVDB200_H
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct svdb200_ctx* svdb200_handle;

enum { SVDB200_F32 = 0, SVDB200_F64 = 1 };

/* Elimination order of stage 1.
 *   PANEL: full-height panel QR / full-width panel LQ + compact-WY trailing update -- the order of
 *          csc586::gpu::cuda_brd_p1 (svd_cuda_1.cu:750, svd_cuda_2.cu:1117) and of its CPU twin
 *          csc586::gpu::brd_p1 (svd_cpu.h:370).  The throughput path.
 *   TILE : flat-tree tile QR/LQ in the exact task order and arithmetic order of
 *          csc586::parallel::brd_p1 (svd_parallel.h:411-533); reproduces data/band_* including the
 *          sign of every band entry (SURVEY 8a'). */
enum { SVDB200_ORDER_PANEL = 0, SVDB200_ORDER_TILE = 1 };

enum {
    SVDB200_OK = 0,
    SVDB200_E_ARG = -1,        /* null pointer / bad enum */
    SVDB200_E_SHAPE = -2,      /* square calls: m != n, band == 0, n % band != 0 (matrix.h:407 needs t | n);
                                  m x n calls (*_mn): min(m, n) < 2, band == 0, min(m, n) % band != 0 */
    SVDB200_E_CAPACITY = -3,   /* exceeds what the handle was created for / what the kernel supports */
    SVDB200_E_NODEVICE = -4,   /* no usable CUDA device: there is no CPU fallback */
    SVDB200_E_NOCONV = -5,     /* QR diagonalisation hit max_iter (svd_serial.h:419) */
    SVDB200_E_STATE = -6,
    SVDB200_CUDA_ERR = 1000,   /* status = 1000 + cudaError_t */
    SVDB200_NCCL_ERR = 2000    /* status = 2000 + ncclResult_t */
};

int svdb200_version(void);
const char* svdb200_strerror(int status);
/* Last CUDA / NCCL error string seen by this handle (empty if none). */
const char* svdb200_last_error(svdb200_handle h);

/* Workspace for matrices up to max_n x max_n with band `band`, element type dtype.
 * Replaces the per-call cudaMalloc of the 6*n^2 arena (svd_cuda_2.cu:1126-1133). */
int svdb200_create(svdb200_handle* out, int device, size_t max_n, size_t band, int dtype);
int svdb200_destroy(svdb200_handle h);
/* Run on a caller-provided CUDA stream (a cudaStream_t passed as void*); NULL restores the
 * handle's own stream.  Lets a harness bracket the work with its own CUDA events. */
int svdb200_set_stream(svdb200_handle h, void* cuda_stream);
int svdb200_synchronize(svdb200_handle h);

/* ---- Stage 1: dense -> band (b+1 diagonals) -----------------------------------------------
 * Replaces csc586::gpu::cuda_brd_p1 (svd_cuda_2.cu:1117; order=PANEL) and
 * csc586::parallel::brd_p1<T> (svd_parallel.h:411; order=TILE).  `a` (n x n) is overwritten by
 * the band matrix (the reference mutates A in place and also returns it). */
int svdb200_dense_to_band_f32(svdb200_handle h, float* a, size_t m, size_t n, size_t band, int order);
int svdb200_dense_to_band_f64(svdb200_handle h, double* a, size_t m, size_t n, size_t band, int order);
int svdb200_dense_to_band_dev_f32(svdb200_handle h, float* a_dev, size_t m, size_t n, size_t band, int order);
int svdb200_dense_to_band_dev_f64(svdb200_handle h, double* a_dev, size_t m, size_t n, size_t band, int order);

/* ---- Stage 2: band -> bidiagonal ------------------------------------------------------------
 * Replaces csc586::parallel::brd_p2<T>(A, band) (svd_parallel.h:640-695) == gpu::brd_p2(A, band+1)
 * (svd_cpu.h:631).  Same window schedule (boundary behaviour included) and the same arithmetic
 * order, so that the result is bit-identical to the reference.  `a` is updated in place (the
 * reference leaves the full matrix updated); d (n) and e (n-1) receive diag(A), diag(A,1). */
int svdb200_band_to_bidiag_f32(svdb200_handle h, float* a, size_t m, size_t n, size_t band, float* d, float* e);
int svdb200_band_to_bidiag_f64(svdb200_handle h, double* a, size_t m, size_t n, size_t band, double* d, double* e);
int svdb200_band_to_bidiag_dev_f32(svdb200_handle h, float* a_dev, size_t m, size_t n, size_t band, float* d_dev, float* e_dev);
int svdb200_band_to_bidiag_dev_f64(svdb200_handle h, double* a_dev, size_t m, size_t n, size_t band, double* d_dev, double* e_dev);

/* Stage 2 and singular values of a band matrix in band storage: O(n band) device memory instead of n^2.
 * ab is LAPACK's upper band storage (dgbbrd / dsbtrd AB(ku+1+i-j, j); scipy's `ab` form, transposed), column by column:
 * ab[j*(band+1) + t] = A[j-band+t][j], t = 0..band, entries above the matrix ignored -- n x (band+1) elements, the layout
 * svdb200_dist_gather_band_dev_* returns.  A LOWER band matrix is passed as its transpose (same singular values).  ab is
 * const and not modified: it is copied into the handle's working buffer (max_n x 3 band elements, allocated on the first
 * call, freed by svdb200_destroy), which holds the 3 band diagonals every window of the chase lies in.  The windows, the
 * arithmetic and therefore d (n), e (n-1) are byte-identical to svdb200_band_to_bidiag_dev_* on the dense embedding of
 * the band.  n >= 2 (else SVDB200_E_SHAPE), 1 <= band <= the handle's band and n <= max_n (else SVDB200_E_CAPACITY); band
 * need not divide n.  The calls follow the handle's stage-2 schedule and singular-value method like svdb200_svdvals_*:
 * for the singular values of a generic band matrix set svdb200_set_stage2_schedule(h, 1) first -- under the default
 * (reference) schedule the un-chased last bulges leave sigma off by 1e-2 ... 1e-1 sigma_1.  Host-pointer variants copy ab
 * in and d / e / sigma out inside the call and fill svdb200_last_timings (h2d, stage 2, qr, d2h). */
int svdb200_band_to_bidiag_packed_f32(svdb200_handle h, const float* ab, size_t n, size_t band, float* d, float* e);
int svdb200_band_to_bidiag_packed_f64(svdb200_handle h, const double* ab, size_t n, size_t band, double* d, double* e);
int svdb200_band_to_bidiag_packed_dev_f32(svdb200_handle h, const float* ab_dev, size_t n, size_t band, float* d_dev, float* e_dev);
int svdb200_band_to_bidiag_packed_dev_f64(svdb200_handle h, const double* ab_dev, size_t n, size_t band, double* d_dev, double* e_dev);
int svdb200_band_svdvals_packed_f32(svdb200_handle h, const float* ab, size_t n, size_t band, float* sigma);
int svdb200_band_svdvals_packed_f64(svdb200_handle h, const double* ab, size_t n, size_t band, double* sigma);
int svdb200_band_svdvals_packed_dev_f32(svdb200_handle h, const float* ab_dev, size_t n, size_t band, float* sigma_dev);
int svdb200_band_svdvals_packed_dev_f64(svdb200_handle h, const double* ab_dev, size_t n, size_t band, double* sigma_dev);

/* ---- QR diagonalisation of the bidiagonal ----------------------------------------------------
 * Replaces csc586::serial::qrd<T> (svd_serial.h:368-422): Demmel-Kahan implicit zero-shift QR
 * sweeps (314-333) with the reference's convergence criteria (138-166), |sigma| sorted
 * descending.  d (n), e (n-1) are inputs; sigma (n) the output; *sweeps (optional) the number of
 * sweeps run.  The reference only compiles for float; the double entry point is the same
 * algorithm in double. */
int svdb200_bidiag_qr_f32(svdb200_handle h, const float* d, const float* e, size_t n, float* sigma, long long* sweeps);
int svdb200_bidiag_qr_f64(svdb200_handle h, const double* d, const double* e, size_t n, double* sigma, long long* sweeps);
int svdb200_bidiag_qr_dev_f32(svdb200_handle h, float* d_dev, float* e_dev, size_t n, float* sigma_dev);
int svdb200_bidiag_qr_dev_f64(svdb200_handle h, double* d_dev, double* e_dev, size_t n, double* sigma_dev);

/* ---- Bidiagonal reduction in one call: stage 1 then stage 2 (the two benchmark legs of
 * `svd_cpu multicore`, svd_cpu.cpp:234-238, chained on the same matrix).  `a` is overwritten by
 * the bidiagonalised matrix; d (n), e (n-1) receive the bidiagonal. */
int svdb200_bidiagonalize_f32(svdb200_handle h, float* a, size_t m, size_t n, size_t band, int order, float* d, float* e);
int svdb200_bidiagonalize_f64(svdb200_handle h, double* a, size_t m, size_t n, size_t band, int order, double* d, double* e);
int svdb200_bidiagonalize_dev_f32(svdb200_handle h, float* a_dev, size_t m, size_t n, size_t band, int order, float* d_dev, float* e_dev);
int svdb200_bidiagonalize_dev_f64(svdb200_handle h, double* a_dev, size_t m, size_t n, size_t band, int order, double* d_dev, double* e_dev);

/* ---- One-stage bidiagonalisation (cross-check path, SURVEY 8f rank 4) -------------------------------------------------
 * Replaces csc586::serial::brd<T> (svd_serial.h:233-266; its blocked / OpenMP twins block_brd 442, gpu::brd svd_cpu.h:441
 * compute the same factorisation): Golub-Kahan Householder bidiagonalisation, one column reflector and one row reflector
 * per step, same sign convention.  Runs the stage-1 panel driver with band 1 (O(n) small launches: a cross-check for the
 * two-stage path, not a throughput path).  `a` is overwritten by the bidiagonalised matrix; d (n), e (n-1) optional. */
int svdb200_bidiagonalize_onestage_f32(svdb200_handle h, float* a, size_t m, size_t n, float* d, float* e);
int svdb200_bidiagonalize_onestage_f64(svdb200_handle h, double* a, size_t m, size_t n, double* d, double* e);
int svdb200_bidiagonalize_onestage_dev_f32(svdb200_handle h, float* a_dev, size_t m, size_t n, float* d_dev, float* e_dev);
int svdb200_bidiagonalize_onestage_dev_f64(svdb200_handle h, double* a_dev, size_t m, size_t n, double* d_dev, double* e_dev);

/* The same for a LIST of independent matrices (sizes may differ; every n[i] <= max_n and band | n[i]): stage 2 of matrix i
 * runs on its own stream beside stage 1 of matrix i+1 (both are latency-bound at moderate n), and in the host-pointer
 * variant the H2D / D2H copies are double-buffered behind the kernels.  a, d, e are host arrays of `count` pointers
 * (device pointers for _dev, host pointers otherwise; d / e or single entries may be NULL).  Results are identical to
 * `count` calls of svdb200_bidiagonalize_*; this is what a benchmark loop over instances (timing.h:55-91) becomes when
 * the instances are handed over together. */
int svdb200_bidiagonalize_many_f32(svdb200_handle h, size_t count, float* const* a, const size_t* n, size_t band, int order, float* const* d, float* const* e);
int svdb200_bidiagonalize_many_f64(svdb200_handle h, size_t count, double* const* a, const size_t* n, size_t band, int order, double* const* d, double* const* e);
int svdb200_bidiagonalize_many_dev_f32(svdb200_handle h, size_t count, float* const* a_dev, const size_t* n, size_t band, int order, float* const* d_dev, float* const* e_dev);
int svdb200_bidiagonalize_many_dev_f64(svdb200_handle h, size_t count, double* const* a_dev, const size_t* n, size_t band, int order, double* const* d_dev, double* const* e_dev);
/* How svdb200_bidiagonalize_many_* schedules a list on `lanes` chains (pure host function, no handle, no device): the matrices
 * are partitioned over the chains longest-processing-time-first (a chain is bound by its stage-2 kernel, whose time is
 * proportional to n), run in ascending size inside a chain and are issued alternating between the chains.  order_out[j] =
 * index of the j-th matrix issued, chain_out[j] = its chain.  lanes: 1..4; the list calls use 2.  The results of the list
 * calls do not depend on the schedule. */
int svdb200_list_plan(int lanes, size_t count, const size_t* n, size_t* order_out, int* chain_out);

/* ---- Fused chain: singular values of a dense matrix (SURVEY 3.5) ------------------------------
 * dense -> brd_p1 -> brd_p2 -> qrd.  `a` is overwritten by the bidiagonalised matrix. */
int svdb200_svdvals_f32(svdb200_handle h, float* a, size_t m, size_t n, size_t band, int order, float* sigma);
int svdb200_svdvals_f64(svdb200_handle h, double* a, size_t m, size_t n, size_t band, int order, double* sigma);
int svdb200_svdvals_dev_f32(svdb200_handle h, float* a_dev, size_t m, size_t n, size_t band, int order, float* sigma_dev);
int svdb200_svdvals_dev_f64(svdb200_handle h, double* a_dev, size_t m, size_t n, size_t band, int order, double* sigma_dev);

/* ---- Rectangular m x n matrices (tall m > n and wide m < n; m == n allowed) -------------------------------------------
 * The panel order on A (m >= n) or on A^T (m < n): sigma(A) = sigma(A^T).  LAPACK gebrd's convention: `a` (m x n,
 * row-major) is overwritten by the reduced matrix in A's own shape -- for m >= n an upper band (dense_to_band_mn) or upper
 * bidiagonal matrix in the top n x n block with the rows below it zero; for m < n a LOWER band / bidiagonal matrix in the
 * left m x m block with the columns right of it zero.  d has min(m, n) entries, e min(m, n) - 1: the super-diagonal for
 * m >= n, the sub-diagonal for m < n.  sigma (min(m, n)) is descending.  With m == n each call returns byte for byte what
 * svdb200_dense_to_band_* / svdb200_bidiagonalize_* / svdb200_svdvals_* return with SVDB200_ORDER_PANEL.
 * Statuses: SVDB200_E_ARG for a null pointer or a dtype mismatch; SVDB200_E_SHAPE when min(m, n) < 2, band == 0 or band
 * does not divide min(m, n) (the longer side is arbitrary); SVDB200_E_CAPACITY when max(m, n) > max_n or band > the
 * handle's band.  Stage 2 and the singular values follow the handle's stage-2 schedule and singular-value method like
 * svdb200_svdvals_*: for the singular values of a generic matrix set svdb200_set_stage2_schedule(h, 1) first.
 * A wide matrix is transposed into a scratch buffer of the handle (m * n elements, allocated on the first wide call,
 * grown when a larger wide matrix arrives, freed by svdb200_destroy), reduced there and transposed back.  Host-pointer
 * variants stage through the handle's max_n^2 buffer and fill svdb200_last_timings, with both transposes counted in
 * stage 1. */
int svdb200_dense_to_band_mn_f32(svdb200_handle h, float* a, size_t m, size_t n, size_t band);
int svdb200_dense_to_band_mn_f64(svdb200_handle h, double* a, size_t m, size_t n, size_t band);
int svdb200_dense_to_band_mn_dev_f32(svdb200_handle h, float* a_dev, size_t m, size_t n, size_t band);
int svdb200_dense_to_band_mn_dev_f64(svdb200_handle h, double* a_dev, size_t m, size_t n, size_t band);
int svdb200_bidiagonalize_mn_f32(svdb200_handle h, float* a, size_t m, size_t n, size_t band, float* d, float* e);
int svdb200_bidiagonalize_mn_f64(svdb200_handle h, double* a, size_t m, size_t n, size_t band, double* d, double* e);
int svdb200_bidiagonalize_mn_dev_f32(svdb200_handle h, float* a_dev, size_t m, size_t n, size_t band, float* d_dev, float* e_dev);
int svdb200_bidiagonalize_mn_dev_f64(svdb200_handle h, double* a_dev, size_t m, size_t n, size_t band, double* d_dev, double* e_dev);
int svdb200_svdvals_mn_f32(svdb200_handle h, float* a, size_t m, size_t n, size_t band, float* sigma);
int svdb200_svdvals_mn_f64(svdb200_handle h, double* a, size_t m, size_t n, size_t band, double* sigma);
int svdb200_svdvals_mn_dev_f32(svdb200_handle h, float* a_dev, size_t m, size_t n, size_t band, float* sigma_dev);
int svdb200_svdvals_mn_dev_f64(svdb200_handle h, double* a_dev, size_t m, size_t n, size_t band, double* sigma_dev);

/* ---- Batched small matrices (BASELINE config 5) ------------------------------------------------
 * `count` independent n x n matrices stored back to back; sigma is count x n.  One matrix per
 * CTA-resident pipeline; shards by matrix across GPUs (one handle per GPU). */
int svdb200_svdvals_batched_f32(svdb200_handle h, float* a, size_t count, size_t n, size_t band, float* sigma);
int svdb200_svdvals_batched_f64(svdb200_handle h, double* a, size_t count, size_t n, size_t band, double* sigma);
int svdb200_svdvals_batched_dev_f32(svdb200_handle h, float* a_dev, size_t count, size_t n, size_t band, float* sigma_dev);
int svdb200_svdvals_batched_dev_f64(svdb200_handle h, double* a_dev, size_t count, size_t n, size_t band, double* sigma_dev);

/* The stages of the batched path one at a time (parity tests gate the band and the bidiagonal separately): what is a
 * bit mask, 1 = stage 1 (a: dense -> band), 2 = stage 2 (a: band -> bidiagonal; d / e, count x n each, optional),
 * 4 = singular values (of the bidiagonals just computed, or of caller-provided d / e when bit 2 is clear).
 * n <= 1024, band <= 64 (the range of the one-launch-per-step batched kernels). */
int svdb200_chain_batched_dev_f32(svdb200_handle h, float* a_dev, size_t count, size_t n, size_t band, int what, float* d_dev, float* e_dev, float* sigma_dev);
int svdb200_chain_batched_dev_f64(svdb200_handle h, double* a_dev, size_t count, size_t n, size_t band, int what, double* d_dev, double* e_dev, double* sigma_dev);

/* Batched rectangular matrices: `count` m x n row-major matrices back to back (stride m * n); with k = min(m, n), sigma
 * is count x k (each row descending), d and e are count x k (rows of length k; the last entry of an e row is unused).
 * `a` is overwritten as by the single-matrix _mn calls (LAPACK gebrd's convention: upper band / bidiagonal in the top
 * n x n block for m >= n, lower band / bidiagonal in the left m x m block for m < n, e then the sub-diagonal).  With m == n
 * the results are byte for byte those of svdb200_svdvals_batched_* / svdb200_chain_batched_dev_*.
 * The one-launch-per-step batched kernels take k <= 1024, band <= 64 and a tallest panel (max(m, n) rows) that fits the
 * batched panel's cluster shared memory (about 2500 rows in f64 at band 64, 5800 at band 32); this is decided before
 * anything is enqueued.  Outside that range svdvals_batched_mn runs the single-matrix chain once per matrix, one after
 * the other, with the bytes and the handle settings of svdb200_svdvals_mn_dev_*; chain_batched_mn_dev returns
 * SVDB200_E_CAPACITY and leaves `a` untouched.  what (chain call): 1 stage 1, 2 stage 2, 4 singular values, each bit its
 * own stage only (stage 2 alone of a wide batch takes the lower band stage 1 left).
 * Statuses: SVDB200_E_ARG for a null pointer, a dtype mismatch, what outside 1..7 or bit 4 without sigma; the shape and
 * capacity rules of the _mn calls; count == 0 returns 0 and does nothing.  The host variant allocates its device buffers
 * per call. */
int svdb200_svdvals_batched_mn_f32(svdb200_handle h, float* a, size_t count, size_t m, size_t n, size_t band, float* sigma);
int svdb200_svdvals_batched_mn_f64(svdb200_handle h, double* a, size_t count, size_t m, size_t n, size_t band, double* sigma);
int svdb200_svdvals_batched_mn_dev_f32(svdb200_handle h, float* a_dev, size_t count, size_t m, size_t n, size_t band, float* sigma_dev);
int svdb200_svdvals_batched_mn_dev_f64(svdb200_handle h, double* a_dev, size_t count, size_t m, size_t n, size_t band, double* sigma_dev);
int svdb200_chain_batched_mn_dev_f32(svdb200_handle h, float* a_dev, size_t count, size_t m, size_t n, size_t band, int what,
                                     float* d_dev, float* e_dev, float* sigma_dev);
int svdb200_chain_batched_mn_dev_f64(svdb200_handle h, double* a_dev, size_t count, size_t m, size_t n, size_t band, int what,
                                     double* d_dev, double* e_dev, double* sigma_dev);
/* Test hook for svdb200_bidiagonalize_many_*: dev_bufs[i] (device, n[i] x n[i] elements, or NULL) receives the band
 * matrix with which matrix i of the NEXT many-call enters stage 2; cleared by that call. */
int svdb200_set_band_capture(svdb200_handle h, void* const* dev_bufs, size_t count);

/* ---- Measurement helpers ------------------------------------------------------------------------
 * Device time (CUDA events on the handle's stream) of the stages of the LAST host-pointer compute call
 * (not the list calls), ms: h2d, d2h and every stage the call ran (stage 1 includes the transposes of a
 * wide matrix and the one-stage reduction); a stage the call did not run reports exactly 0.
 * svdvals_batched and svdvals_batched_mn interleave the stages of their matrices and report only h2d and d2h.
 * stage-1 sub-times: panel factorisations vs trailing updates are reported by svdb200_stage1_profile. */
int svdb200_last_timings(svdb200_handle h, double* ms_stage1, double* ms_stage2, double* ms_qr, double* ms_h2d, double* ms_d2h);
/* Per-kernel-class profiling.  When on, every launch of the hot-path kernels is bracketed by CUDA
 * events on the handle's stream and its duration and ALGORITHMIC work are accumulated per class:
 *   0 panel factorisation   (flops 2*m*b^2)            3 rank-b update C += P Q  (flops 2*M*N*b)
 *   1 W = V^T C             (flops 2*M*N*b)            4 stage-2 bulge chasing   (bytes 4*b*n^2*sizeof(T))
 *   2 W = C U^T             (flops 2*M*N*b)            5 QR diagonalisation      (n*sweeps steps)
 * get: arrays of SVDB200_PROFILE_CLASSES entries (ms, work, launches); reset clears them. */
#define SVDB200_PROFILE_CLASSES 6
int svdb200_set_profile(svdb200_handle h, int on);
int svdb200_get_profile(svdb200_handle h, double* ms, double* work, long long* launches);
int svdb200_reset_profile(svdb200_handle h);
/* Number of kernel launches issued by this handle since creation (the bench's gpu_launches). */
long long svdb200_launch_count(svdb200_handle h);
/* reference error metric gpu::Matrix<T>::mse (matrix_gpu.h:438-453), evaluated on the device. */
int svdb200_mse_f32(svdb200_handle h, const float* a, const float* b, size_t n, size_t band, float* out);
int svdb200_mse_f64(svdb200_handle h, const double* a, const double* b, size_t n, size_t band, double* out);
/* Deterministic U[lo,hi) fill of a DEVICE buffer (svdsolver_b200/synth.py documents the stream);
 * replaces matrix_generator / Matrix::fill(min,max) (svd_cuda_2.cu:1230, matrix_gpu.h:336). */
int svdb200_fill_uniform_dev_f32(svdb200_handle h, float* a_dev, size_t count, unsigned long long seed, double lo, double hi);
int svdb200_fill_uniform_dev_f64(svdb200_handle h, double* a_dev, size_t count, unsigned long long seed, double lo, double hi);
/* Register-resident FP64 (DMMA mma.sync m8n8k4 / DFMA) and FP32 (FFMA) peak probes: TFLOP/s. kind:
 * 0 = DFMA, 1 = DMMA f64, 2 = FFMA, 3 = TF32 mma.sync, 4 = TF32 tcgen05.mma (M128 N256 K8, operands
 * resident in shared memory, accumulator in TMEM).  Used as roofline denominators. */
int svdb200_probe_peak(svdb200_handle h, int kind, double* tflops);
/* FP32 trailing update on tcgen05/TMEM/TMA (3xTF32).  mode 0: never (mma.sync kernels only), 1: when
 * the updated block has at least min_elems elements (default), 2: always (tests).  min_elems <= 0
 * keeps the current threshold.  No effect on FP64 handles (tcgen05.mma has no f64 kind). */
int svdb200_set_tc05(svdb200_handle h, int mode, long long min_elems);
/* Stage-2 window schedule.  0 (default) = the reference's schedule, bit-for-bit (svd_parallel.h:640-695): its pair count
 * per sweep is floor((n - j2)/(w-1)) + 1 (the ceil at line 664 acts on an integer quotient), so when that division has a
 * remainder the last LEFT window leaves a bulge nobody chases and the bidiagonal's singular values drift from those of
 * the input (1e-3 sigma_1 on stage-1 outputs, up to 1e-1 on generic band matrices; SURVEY 0.3).  1 = complete chase:
 * the same windows and arithmetic, continued until they are empty; orthogonally equivalent to the input (sigma to
 * round-off).  Use 0 for parity with the reference, 1 when the singular values themselves matter. */
int svdb200_set_stage2_schedule(svdb200_handle h, int mode);
/* Stage-1 panel kernel (replaces qr_cuda / lq_cuda, svd_cuda_2.cu:881/959): 2 (default) = Cholesky-QR with reconstructed
 * Householder vectors (two passes over the panel, no exchange between CTAs; band 8/16/32/64, panel height >= 2 band) with
 * the blocked kernel as the fallback for ill-conditioned panels; 1 = blocked kernel, one exchange between the CTAs per
 * sub-panel of 8 columns (band a multiple of 8, <= 64); 0 = the per-column kernels (one exchange per column).  Same
 * factorisation (sign rule of svd_serial.h:194-201), results equal to round-off. */
int svdb200_set_panel_kernel(svdb200_handle h, int kind);
/* Smallest pivot ratio min_j R_jj^2 / G_jj the Cholesky-QR panel accepts (default 1e-3); panels below are redone by the
 * exchange-based kernels inside the same call.  svdb200_chol_fallback_count: how often that happened on this handle
 * (synchronises the handle's streams). */
int svdb200_set_chol_guard(svdb200_handle h, double guard);
int svdb200_chol_fallback_count(svdb200_handle h, long long* count);
int svdb200_debug_panel_blk_timing(long long* out16);
int svdb200_debug_panel_chol_timing(long long* out16);
/* Debug: per-phase cycle counters of the register panel kernel (all zero unless built with -DSVDB_PANEL_TIMING=1). */
int svdb200_debug_panel_timing(long long* out16);
/* same for the stage-2 kernel (-DSVDB_S2_TIMING=1): RIGHT ops of CTA 1 */
int svdb200_debug_stage2_timing(long long* out16);
/* 24 cycle counters of the band-32 latency-optimised kernel (CTA 1; slots documented in tools/stage2_only.py) */
int svdb200_debug_stage2_fast_timing(long long* out24);
/* Singular values of the bidiagonal (svdb200_bidiag_qr_*, svdb200_svdvals_*): method 0 = automatic (the
 * reference's zero-shift QR sweeps, serial::qrd svd_serial.h:368, for n <= auto_limit, bisection on the
 * Golub-Kahan form above: zero-shift QR needs ~n log(1/tol) sweeps), 1 = always zero-shift QR, 2 = always
 * bisection, 3 = implicit SHIFTED QR (Golub-Kahan steps with shifts from the trailing block, pipelined sweeps, double
 * arithmetic for both element types; the reference is zero-shift only, svd_serial.h:314-333).  auto_limit == 0 keeps the
 * current limit (default 1024). */
int svdb200_set_qr_method(svdb200_handle h, int method, size_t auto_limit);
/* Unit test of the tcgen05 building blocks (TMA box -> swizzled shared memory -> UMMA descriptors -> TMEM ->
 * tcgen05.ld): D(128 x 64) = A(128 x 32) B(32 x 64) in one TF32 pass.  a_mn/b_mn select the operand storage:
 * 0 = K-major (a: 128 x 32 row-major, b: B^T 64 x 32 row-major), 1 = MN-major (a: A^T 32 x 128, b: B 32 x 64).
 * All device pointers; out has 128*64+1 floats (last = TMEM base address bits), dump 6144 floats = the staged
 * A (16 KB) and B (8 KB) tiles as they sit in shared memory. */
int svdb200_tc05_selftest(svdb200_handle h, int a_mn, int b_mn, const float* a, const float* b, float* out, float* dump);

/* Trailing-update building blocks, exposed for parity tests and kernel-level benchmarks
 * (qr_apply / lq_apply, svd_parallel.h:243-281): all device pointers, row-major.
 *   W(b x ncols)   = V(mrows x b)^T * C(mrows x ncols)          [ldc]
 *   C(mrows x ncols) += P(mrows x b) * Q(b x ncols)
 *   W(mrows x b)   = C(mrows x ncols) * Ut(ncols x b) */
int svdb200_gemm_tn_dev_f32(svdb200_handle h, const float* v, const float* c, size_t ldc, size_t mrows, size_t ncols, size_t b, float* w);
int svdb200_gemm_tn_dev_f64(svdb200_handle h, const double* v, const double* c, size_t ldc, size_t mrows, size_t ncols, size_t b, double* w);
int svdb200_rank_update_dev_f32(svdb200_handle h, float* c, size_t ldc, size_t mrows, size_t ncols, size_t b, const float* p, const float* q, size_t ldq);
int svdb200_rank_update_dev_f64(svdb200_handle h, double* c, size_t ldc, size_t mrows, size_t ncols, size_t b, const double* p, const double* q, size_t ldq);
int svdb200_gemm_nn_dev_f32(svdb200_handle h, const float* c, size_t ldc, size_t mrows, size_t ncols, size_t b, const float* ut, float* w);
int svdb200_gemm_nn_dev_f64(svdb200_handle h, const double* c, size_t ldc, size_t mrows, size_t ncols, size_t b, const double* ut, double* w);

/* One stage-1 panel on its own (qr / lq of svd_parallel.h:133-226 in the panel order of svd_cuda_2.cu:881 / 959): the
 * m x b panel at a (leading dimension lda; trans != 0: the b x m ROW panel, factorised as its transpose) is overwritten
 * by R (zeros below the diagonal); v receives V (m x b, unit diagonal explicit), v2 = V S^T (m x b; trans: b x m) with
 * Q = I + V S V^T.  Exposed for kernel-level parity tests and timing of tall panels; m <= max_n, b <= band of the handle. */
int svdb200_panel_factor_dev_f32(svdb200_handle h, float* a_dev, size_t lda, size_t m, size_t b, int trans, float* v_dev, float* v2_dev);
int svdb200_panel_factor_dev_f64(svdb200_handle h, double* a_dev, size_t lda, size_t m, size_t b, int trans, double* v_dev, double* v2_dev);

/* ---- Multi-GPU stage 1 (BASELINE config 4): 1-D block-cyclic over columns, one process per GPU.
 * nccl_unique_id: the 128-byte ncclUniqueId produced by svdb200_dist_unique_id on rank 0 and
 * broadcast by the launcher (torch.distributed / MPI / a file).  a_local holds this rank's block
 * columns: global block-column j (width band) lives on rank j % nranks at local block j / nranks;
 * storage is row-major n x ncols_local. */
typedef struct svdb200_dist_ctx* svdb200_dist_handle;
int svdb200_dist_unique_id(void* out128);
int svdb200_dist_create(svdb200_dist_handle* out, int device, int rank, int nranks, const void* nccl_unique_id,
                        size_t n, size_t band, int dtype);
int svdb200_dist_destroy(svdb200_dist_handle h);
size_t svdb200_dist_local_cols(size_t n, size_t band, int rank, int nranks);
int svdb200_dist_dense_to_band_dev_f32(svdb200_dist_handle h, float* a_local_dev, size_t n, size_t band);
int svdb200_dist_dense_to_band_dev_f64(svdb200_dist_handle h, double* a_local_dev, size_t n, size_t band);
/* Hand-off to stage 2 (SURVEY 8e: "band gathered to one GPU first"): after svdb200_dist_dense_to_band_dev_*, the b+1
 * diagonals are collected from all ranks (one ncclAllGather of n (b+1) elements) into packed band storage on EVERY rank:
 * packed[gc * (band+1) + t] = A[gc - band + t][gc], t = 0..band (device, n x (band+1)). */
int svdb200_dist_gather_band_dev_f32(svdb200_dist_handle h, const float* a_local_dev, float* packed_dev);
int svdb200_dist_gather_band_dev_f64(svdb200_dist_handle h, const double* a_local_dev, double* packed_dev);
/* Singular values of a block-cyclically distributed matrix: stage 1 on all ranks, band gathered, stage 2 + singular
 * values on rank 0 (those stages are one sequential wavefront over an O(n b) band: one GPU per matrix).  sigma_dev (n,
 * device) is written on rank 0 only; a_local is overwritten by the rank's part of the band matrix. */
int svdb200_dist_svdvals_dev_f32(svdb200_dist_handle h, float* a_local_dev, float* sigma_dev);
int svdb200_dist_svdvals_dev_f64(svdb200_dist_handle h, double* a_local_dev, double* sigma_dev);
/* run-time switches of the handle's single-GPU stages (see svdb200_set_stage2_schedule / _qr_method / _tc05); -1 keeps */
int svdb200_dist_configure(svdb200_dist_handle h, int stage2_schedule, int qr_method, int tc05_mode);
/* LQ (row) panels of the distributed stage 1: 1 (default) = every rank forms the Gram matrix of its own columns of the
 * row panel, one all-reduce of band^2-sized data, identical band x band algebra on every rank (Cholesky-QR with
 * reconstructed Householder vectors); row panels whose pivot ratio falls below the guard are redone through the other
 * path (svdb200_dist_lq_fallback_count says how many); 0 = all-gather of the row panel, factorised redundantly on every
 * rank by the single-GPU panel kernels.  Same factorisation, results equal to round-off. */
int svdb200_dist_configure_panels(svdb200_dist_handle h, int lq_distributed);
long long svdb200_dist_lq_fallback_count(svdb200_dist_handle h);
int svdb200_dist_set_stream(svdb200_dist_handle h, void* cuda_stream);
long long svdb200_dist_launch_count(svdb200_dist_handle h);

#ifdef __cplusplus
}
#endif
#endif /* SVDB200_H */

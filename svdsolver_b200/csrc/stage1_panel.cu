// Stage 1, panel order: dense -> band by full-height panel QR / full-width panel LQ with a
// compact-WY trailing update.  Replaces csc586::gpu::cuda_brd_p1 (svd_cuda_1.cu:750,
// svd_cuda_2.cu:1117) / csc586::gpu::brd_p1 (svd_cpu.h:370) and their helpers qr_cuda/lq_cuda
// (svd_cuda_2.cu:881/959), hholder_cuda (797), wy_compact_cuda (838).
//
// Panel kernel (one launch per panel instead of ~25 launches per COLUMN):
//   * the m x b panel is distributed by rows over G CTAs and stays resident in shared memory for
//     the whole factorisation (an LQ row panel is loaded transposed, so one code path serves both);
//   * per column ONE all-reduce: every CTA publishes the dot products of the pivot column with all
//     b columns over its rows, the pivot-row owner publishes the pivot row; after the barrier every
//     CTA forms ||x||, the Householder scalars (sign convention of svd_serial.h:194-201:
//     H x = -sign(x0)||x|| e1), the rank-1 update coefficients and column j of the compact-WY
//     factor S (= -T, svd_parallel.h:97-113) redundantly from the reduced vector;
//   * two transports for the all-reduce:
//       kCluster = true : the CTAs form ONE thread-block cluster (<= 16 CTAs); partial vectors live
//                         in each CTA's shared memory and are read by the peers over DSMEM; the
//                         barrier is barrier.cluster (~0.2 us).  Used whenever the panel fits the
//                         cluster's shared memory (m*b*sizeof(T) <~ 3 MB).
//       kCluster = false: cooperative grid over up to 148 CTAs, partials through L2, software grid
//                         barrier (~2-3 us).  Used for the tall panels of large matrices.
//   * partial sums are combined in a fixed association, so the result is deterministic.
// Outputs: R (or L) written into A with exact zeros below the diagonal of the panel, V (m x b,
// unit diagonal explicit), V2 = V S^T, and S.
#include <algorithm>
#include <cooperative_groups.h>
#include "common.cuh"

namespace cg = cooperative_groups;

namespace svdb200 {

// register-resident fast path (stage1_panel_reg.cu): 0 = ran, 1 = shape not covered
template <typename T, bool kTrans>
int launch_panel_reg(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream, bool cooperative);
// blocked kernel, one exchange per 8 columns (stage1_panel_blk.cu): same convention
template <typename T, bool kTrans>
int launch_panel_blk(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream);
// Cholesky-QR panel with reconstructed Householder vectors (stage1_panel_chol.cu): 0 = launched -- a fallback kernel gated
// on chol_status() must follow in the stream --, 1 = shape not covered
template <typename T, bool kTrans>
int launch_panel_chol(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream);
const int* chol_status(Ctx* c);

namespace {

constexpr int kPanelThreads = 256;

// Panel element (r, c): r in [0,m) along the reflector direction, c in [0,b).
//   kTrans == false (QR): A[r*lda + c]        kTrans == true (LQ): A[c*lda + r]
template <typename T, bool kTrans, bool kCluster>
__global__ void __launch_bounds__(kPanelThreads)
panel_factor_kernel(T* __restrict__ A, size_t lda, int m, int b, int rows_per_cta, T* __restrict__ V, T* __restrict__ V2,
                    T* __restrict__ S_out, T* __restrict__ red, unsigned* __restrict__ bar, int Gb, size_t sA, size_t sV,
                    const int* __restrict__ run_if) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (run_if != nullptr && *run_if == 0) return;       // fallback launch behind the Cholesky-QR panel: only when it gave up
    const int tid = threadIdx.x, nt = blockDim.x;
    // Gb > 0: batched launch, clusters of Gb CTAs, one matrix (element strides sA / sV) per cluster
    const int G = Gb > 0 ? Gb : gridDim.x, g = Gb > 0 ? blockIdx.x % Gb : blockIdx.x;
    if (Gb > 0) {
        const size_t mat = blockIdx.x / Gb;
        A += mat * sA; V += mat * sV; V2 += mat * sV;
    }
    const int r0 = g * rows_per_cta;
    const int R = max(0, min(rows_per_cta, m - r0));     // local rows
    const int ld = b + 1;
    const int slot = 2 * b;                              // b dots + b pivot-row values
    T* lred = reinterpret_cast<T*>(smem_raw);            // 2 * slot : this CTA's published vectors (cluster mode)
    T* Ps = lred + 2 * slot;                             // R x ld
    T* Gm = Ps + (size_t)rows_per_cta * ld;              // b x b : Gm[c][j] = v_c^T v_j (c < j)
    T* zs = Gm + b * b;                                  // b : reduced dots
    T* piv = zs + b;                                     // b : pivot row
    T* fs = piv + b;                                     // b : update coefficients
    T* taus = fs + b;                                    // b
    T* psum = taus + b;                                  // blockDim : chunk sums
    unsigned gen = 0;
    const int tx = tid % b, tyy = tid / b;               // 2-D view: b columns x rgroups rows
    const int rgroups = max(1, nt / b);
    const bool in2d = tyy < rgroups;
    const int lane = tid & 31, wrp = tid >> 5, nwarps = nt >> 5;

    // ---- load the local slice --------------------------------------------------------------------
    if (!kTrans) {
        if (in2d)
            for (int rl = tyy; rl < R; rl += rgroups) Ps[rl * ld + tx] = A[(size_t)(r0 + rl) * lda + tx];
    } else {
        for (int c = wrp; c < b; c += nwarps)
            for (int rl = lane; rl < R; rl += 32) Ps[rl * ld + c] = A[(size_t)c * lda + (r0 + rl)];
    }
    for (int e = tid; e < b * b; e += nt) Gm[e] = (T)0;
    __syncthreads();

    const int kmax = min(b, m);
    for (int j = 0; j < kmax; ++j) {
        // ---- phase A: local dots of column j (rows > j) with every column ---------------------------
        const int lo = max(0, j + 1 - r0);               // first local row with global index > j
        if (in2d) {
            T acc = (T)0;
            for (int rl = lo + tyy; rl < R; rl += rgroups) acc += Ps[rl * ld + tx] * Ps[rl * ld + j];
            psum[tyy * b + tx] = acc;
        }
        __syncthreads();
        T* mine = kCluster ? lred + (j & 1) * slot : red + ((size_t)(j & 1) * (G + 1) + g) * slot;
        T* pivslot = kCluster ? lred + (j & 1) * slot + b : red + ((size_t)(j & 1) * (G + 1) + G) * slot;
        const bool owner = (j >= r0 && j < r0 + R);
        for (int c = tid; c < b; c += nt) {
            T acc = psum[c];
            for (int grp = 1; grp < rgroups; ++grp) acc += psum[grp * b + c];
            if (kCluster) mine[c] = acc; else st_cg(&mine[c], acc);
            if (owner) {
                if (kCluster) pivslot[c] = Ps[(j - r0) * ld + c]; else st_cg(&pivslot[c], Ps[(j - r0) * ld + c]);
            }
        }
        if (kCluster) cg::this_cluster().sync(); else grid_barrier(bar, (unsigned)G, gen);
        // ---- phase B: all-reduce in a fixed association ------------------------------------------------
        {
            const int chunk = (G + rgroups - 1) / rgroups;
            const int jowner = j / rows_per_cta;
            if (in2d) {
                const int c = tx, part = tyy;
                const int q0 = part * chunk, q1 = min(G, q0 + chunk);
                T acc = (T)0;
                if (kCluster) {
                    cg::cluster_group cl = cg::this_cluster();
#pragma unroll 4
                    for (int q = q0; q < q1; ++q) acc += cl.map_shared_rank(lred, q)[(j & 1) * slot + c];
                    if (part == 0) piv[c] = cl.map_shared_rank(lred, jowner)[(j & 1) * slot + b + c];
                } else {
                    const T* buf = red + (size_t)(j & 1) * (G + 1) * slot;
#pragma unroll 8
                    for (int q = q0; q < q1; ++q) acc += ld_cg(&buf[(size_t)q * slot + c]);
                    if (part == 0) piv[c] = ld_cg(&buf[(size_t)G * slot + c]);
                }
                psum[part * b + c] = acc;
            }
            __syncthreads();
            for (int c = tid; c < b; c += nt) {
                T acc = psum[c];
                for (int part = 1; part < rgroups; ++part) acc += psum[part * b + c];
                zs[c] = acc;
            }
        }
        __syncthreads();
        // ---- phase C: scalars, Gram column, rank-1 update -----------------------------------------------
        const T x0 = piv[j];
        const T normsq = zs[j] + x0 * x0;
        const T nrm = sqrt(normsq);
        const double sgn = -copysign(1.0, (double)x0);
        const double u1 = (double)x0 - sgn * (double)nrm;
        const T alpha = (T)(1.0 / u1);
        const T tau = (T)(-sgn * u1 / (double)nrm);
        const T beta = (T)(sgn * (double)nrm);           // R_jj = -sign(x0) ||x||
        for (int c = tid; c < b; c += nt) {
            if (c > j) {
                // w^T a_c with w = [1; alpha*x_{>j}] :  piv[c] + alpha * sum_{r>j} x_r a_rc
                fs[c] = tau * (piv[c] + alpha * zs[c]);
            } else if (c < j) {
                // v_c^T v_j = V[j][c] * 1 + alpha * sum_{r>j} V[r][c] x_r
                Gm[c * b + j] = piv[c] + alpha * zs[c];
            } else {
                taus[j] = tau;
            }
        }
        // scale the pivot column into w (rows > j), store beta on the pivot row
        for (int rl = lo + tid; rl < R; rl += nt) Ps[rl * ld + j] *= alpha;
        if (owner && tid == 0) Ps[(j - r0) * ld + j] = beta;
        __syncthreads();
        // rows >= j, columns > j :  a_rc -= w_r * f_c
        if (in2d && tx > j) {
            const int lo2 = max(0, j - r0);
            const T f = fs[tx];
            for (int rl = lo2 + tyy; rl < R; rl += rgroups) {
                T wv = (r0 + rl == j) ? (T)1 : Ps[rl * ld + j];
                Ps[rl * ld + tx] -= wv * f;
            }
        }
        __syncthreads();
    }

    // ---- epilogue ------------------------------------------------------------------------------------
    // V(row, k) = 1 (row == k), Ps (row > k), 0 (row < k); the factored panel goes back into A with
    // exact zeros below the diagonal.
    if (!kTrans) {
        if (in2d)
            for (int rl = tyy; rl < R; rl += rgroups) {
                const int row = r0 + rl, c = tx;
                T vv = (row == c) ? (T)1 : (row > c ? Ps[rl * ld + c] : (T)0);
                if (c >= kmax) vv = (T)0;
                V[(size_t)row * b + c] = vv;
                A[(size_t)row * lda + c] = (c >= row) ? Ps[rl * ld + c] : (T)0;
            }
    } else {
        if (in2d)
            for (int rl = tyy; rl < R; rl += rgroups) {
                const int row = r0 + rl, c = tx;
                T vv = (row == c) ? (T)1 : (row > c ? Ps[rl * ld + c] : (T)0);
                if (c >= kmax) vv = (T)0;
                V[(size_t)row * b + c] = vv;
            }
        for (int c = wrp; c < b; c += nwarps)
            for (int rl = lane; rl < R; rl += 32) {
                const int row = r0 + rl;
                A[(size_t)c * lda + row] = (c >= row) ? Ps[rl * ld + c] : (T)0;
            }
    }
    __syncthreads();
    // V2 = V S^T with S = -T and T^{-1} = D + striu(V^T V), D = diag(1/tau)  (equivalent to the
    // recurrence of svd_parallel.h:97-113, but off the per-column critical path): every row x of V2
    // solves  x (D + U)^T = -v  by back substitution, in place over the row of V held in Ps.
    for (int rl = tid; rl < R; rl += nt) {
        const int row = r0 + rl;
        T* x = Ps + rl * ld;
        const int khi = min(kmax - 1, row);
        for (int c = b - 1; c > khi; --c) x[c] = (T)0;
        for (int c = khi; c >= 0; --c) {
            T acc = (row == c) ? (T)-1 : -x[c];          // -v[c]
            for (int k = c + 1; k <= khi; ++k) acc -= x[k] * Gm[c * b + k];
            x[c] = acc * taus[c];
        }
    }
    __syncthreads();
    if (!kTrans) {
        if (in2d)
            for (int rl = tyy; rl < R; rl += rgroups) V2[(size_t)(r0 + rl) * b + tx] = Ps[rl * ld + tx];
    } else {
        for (int c = wrp; c < b; c += nwarps)
            for (int rl = lane; rl < R; rl += 32) V2[(size_t)c * m + (r0 + rl)] = Ps[rl * ld + c];
    }
    // S itself (b x b, upper triangular) is only needed by callers that ask for it: CTA 0 rebuilds it
    // from the Gram matrix with the reference recurrence S[0:j,j] = -tau_j S[0:j,0:j] g_j, S[j][j] = -tau_j.
    if (g == 0 && S_out != nullptr) {
        __syncthreads();
        T* Ss = psum;                                     // reuse: needs b*b <= blockDim only for small b
        (void)Ss;
        if (tid == 0) {
            for (int j = 0; j < kmax; ++j) {
                for (int r = 0; r < j; ++r) {
                    T acc = (T)0;
                    for (int c = r; c < j; ++c) acc += S_out[r * b + c] * Gm[c * b + j];
                    S_out[r * b + j] = -taus[j] * acc;
                }
                S_out[j * b + j] = -taus[j];
                for (int r = j + 1; r < b; ++r) S_out[r * b + j] = (T)0;
            }
        }
    }
    // no CTA may exit while a peer can still read its shared memory
    if (kCluster) cg::this_cluster().sync();
}

inline size_t panel_smem_bytes(int rows, int b, size_t esz) {
    return ((size_t)4 * b + (size_t)rows * (b + 1) + (size_t)b * b + 4 * (size_t)b + kPanelThreads + 8) * esz;
}

template <typename T, bool kTrans>
int launch_panel_exchange(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream);

template <typename T, bool kTrans>
int launch_panel(Ctx* c, T* a, size_t lda, int m, int b, T* V = nullptr, T* V2 = nullptr, cudaStream_t stream = nullptr) {
    if (!stream) stream = c->stream;
    ProfScope ps(c, 0, 2.0 * (double)m * (double)b * (double)b);
    if (!V) V = reinterpret_cast<T*>(c->v);
    if (!V2) V2 = reinterpret_cast<T*>(c->v2);
    c->panel_run_if = nullptr;
    if (c->cfg.panel_chol) {
        const int st = launch_panel_chol<T, kTrans>(c, a, lda, m, b, V, V2, stream);
        if (st == 0) c->panel_run_if = chol_status(c);        // the exchange-based kernel below runs only if the guard tripped
        else if (st != 1) return st;
    }
    const int st = launch_panel_exchange<T, kTrans>(c, a, lda, m, b, V, V2, stream);
    c->panel_run_if = nullptr;
    return st;
}

template <typename T, bool kTrans>
int launch_panel_exchange(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream) {
    if (c->cfg.panel_blk) {
        int st = launch_panel_blk<T, kTrans>(c, a, lda, m, b, V, V2, stream);
        if (st != 1) return st;
    }
    // register-resident kernel for tall panels (grid transport); cluster-sized panels are issue-bound
    // either way and stay on the shared-memory kernel below
    constexpr int kPanelRegMinRows = 768;
    if (m > kPanelRegMinRows) {
        int st = launch_panel_reg<T, kTrans>(c, a, lda, m, b, V, V2, stream, stream == c->stream);
        if (st != 1) return st;
    }
    T* S = nullptr;      // the compact-WY factor itself is not needed: V2 = V S^T is produced directly
    T* red = reinterpret_cast<T*>(c->red);
    unsigned* bar = c->bar;
    // ---- cluster transport when the panel fits the shared memory of one cluster ---------------------
    if (c->cluster_ok) {
        int G = (m + 31) / 32;
        if (G > c->cluster_ok) G = c->cluster_ok;
        if (G < 1) G = 1;
        int rows = (m + G - 1) / G;
        G = (m + rows - 1) / rows;
        size_t smem = panel_smem_bytes(rows, b, sizeof(T));
        if (smem <= 200 * 1024) {
            auto kern = panel_factor_kernel<T, kTrans, true>;
            SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            if (G > 8) SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(G);
            cfg.blockDim = dim3(kPanelThreads);
            cfg.dynamicSmemBytes = smem;
            cfg.stream = stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = G;
            attr[0].val.clusterDim.y = 1;
            attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a, lda, m, b, rows, V, V2, S, red, bar, 0, (size_t)0, (size_t)0, c->panel_run_if);
            if (e == cudaSuccess) {
                c->launches++;
                return 0;
            }
            cudaGetLastError();           // cluster shape not schedulable here: use the grid transport
            c->cluster_ok = c->cluster_ok > 8 ? 8 : 0;
            return launch_panel_exchange<T, kTrans>(c, a, lda, m, b, V, V2, stream);
        }
    }
    // ---- cooperative-grid transport -----------------------------------------------------------------------
    int G = (m + 63) / 64;
    if (G > c->num_sms) G = c->num_sms;
    if (G > kMaxPanelCtas) G = kMaxPanelCtas;
    if (G < 1) G = 1;
    int rows = (m + G - 1) / G;
    G = (m + rows - 1) / rows;
    size_t smem = panel_smem_bytes(rows, b, sizeof(T));
    if (smem > 227 * 1024) return SVDB200_E_CAPACITY;
    auto kern = panel_factor_kernel<T, kTrans, false>;
    SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    SVDB_CHECK(c, cudaMemsetAsync(c->bar, 0, 2 * sizeof(unsigned), stream));
    int gb0 = 0;
    size_t zero = 0;
    const int* run_if = c->panel_run_if;
    void* args[] = {&a, &lda, &m, &b, &rows, &V, &V2, &S, &red, &bar, &gb0, &zero, &zero, &run_if};
    SVDB_CHECK(c, cudaLaunchCooperativeKernel((void*)kern, dim3(G), dim3(kPanelThreads), args, smem, stream));
    c->launches++;
    return 0;
}

}  // namespace

// panel factorisation for other translation units (the multi-GPU driver in dist.cu)
template <typename T, bool kTrans>
int launch_panel_public(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream) {
    return launch_panel<T, kTrans>(c, a, lda, m, b, V, V2, stream);
}
template int launch_panel_public<float, false>(Ctx*, float*, size_t, int, int, float*, float*, cudaStream_t);
template int launch_panel_public<float, true>(Ctx*, float*, size_t, int, int, float*, float*, cudaStream_t);
template int launch_panel_public<double, false>(Ctx*, double*, size_t, int, int, double*, double*, cudaStream_t);
template int launch_panel_public<double, true>(Ctx*, double*, size_t, int, int, double*, double*, cudaStream_t);

// Batched panels (uniform shape): one thread-block cluster per matrix, panel resident in the cluster's shared
// memory, all-reduce over DSMEM.  Used by the small-matrix batched driver (BASELINE configs[4]).
template <typename T, bool kTrans>
int panel_batched(Ctx* c, T* a, size_t lda, size_t sA, int m, int b, T* V, T* V2, size_t sV, int count) {
    if (count <= 0 || m <= 0) return 0;
    int G = (m + 127) / 128;                       // <= 128 rows per CTA: few, fat CTAs (many matrices share the GPU)
    if (G > 8) G = 8;
    int rows = (m + G - 1) / G;
    G = (m + rows - 1) / rows;
    const size_t smem = panel_smem_bytes(rows, b, sizeof(T));
    if (smem > 200 * 1024) return SVDB200_E_CAPACITY;
    auto kern = panel_factor_kernel<T, kTrans, true>;
    SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    T* S = nullptr;
    T* red = nullptr;
    unsigned* bar = nullptr;
    for (int z0 = 0; z0 < count; z0 += 16384) {
        const int zc = std::min(16384, count - z0);
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)(G * zc));
        cfg.blockDim = dim3(kPanelThreads);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = c->stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = G;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        T* az = a + (size_t)z0 * sA;
        T* vz = V + (size_t)z0 * sV;
        T* v2z = V2 + (size_t)z0 * sV;
        SVDB_CHECK(c, cudaLaunchKernelEx(&cfg, kern, az, lda, m, b, rows, vz, v2z, S, red, bar, G, sA, sV, (const int*)nullptr));
        c->launches++;
    }
    return 0;
}
template int panel_batched<float, false>(Ctx*, float*, size_t, size_t, int, int, float*, float*, size_t, int);
template int panel_batched<float, true>(Ctx*, float*, size_t, size_t, int, int, float*, float*, size_t, int);
template int panel_batched<double, false>(Ctx*, double*, size_t, size_t, int, int, double*, double*, size_t, int);
template int panel_batched<double, true>(Ctx*, double*, size_t, size_t, int, int, double*, double*, size_t, int);

// Driver: same panel sequence as svd_cpu.h:382-423 / svd_cuda_2.cu:1148-1213.
//
// Look-ahead: the rank-b update of a half-step is split so that the part the NEXT panel lives in
// (its b rows / b columns) is updated first; the next panel is then factorised on a second,
// high-priority stream while the main stream finishes the (much larger) rest of the update.
// QR reflectors use (v, v2), LQ reflectors (vb, v2b), so a panel in flight never overwrites
// reflectors that the concurrent update still reads.  In profiling mode the steps are serialised
// so that per-kernel-class times stay meaningful.
template <typename T>
int stage1_panel_order(Ctx* c, T* a, size_t n, size_t band) {
    if (band == 0 || n == 0 || n % band != 0) return SVDB200_E_SHAPE;
    if (band > (size_t)kMaxBand || n > c->max_n || band > c->band) return SVDB200_E_CAPACITY;
    const int b = (int)band;
    T* Vq = reinterpret_cast<T*>(c->v);
    T* V2q = reinterpret_cast<T*>(c->v2);
    T* Vl = reinterpret_cast<T*>(c->vb);
    T* V2l = reinterpret_cast<T*>(c->v2b);
    T* W = reinterpret_cast<T*>(c->w);
    const bool ahead = !c->profile && c->aux_stream != nullptr;
    cudaStream_t s0 = c->stream, s1 = ahead ? c->aux_stream : c->stream;
    if (ahead) {   // the aux stream must see everything enqueued on the main stream so far
        SVDB_CHECK(c, cudaEventRecord(c->lev[0], s0));
        SVDB_CHECK(c, cudaStreamWaitEvent(s1, c->lev[0], 0));
    }
    // first QR panel
    SVDB_TRY((launch_panel<T, false>(c, a, n, (int)n, b, Vq, V2q, s1)));
    if (ahead) SVDB_CHECK(c, cudaEventRecord(c->lev[1], s1));
    for (size_t k = 0; k < n; k += band) {
        const size_t m = n - k;                 // panel height
        const size_t nc = n - k - band;         // columns right of the QR panel
        // svd_cpu.h:396 skips the LQ half-step when only one column is left; the one-stage Golub-Kahan order
        // (serial::brd, svd_serial.h:248) still applies that length-1 reflector (a sign flip): c->onestage
        const bool has_lq = c->onestage ? (k + band < n) : (k + band < n - 1);
        if (ahead) SVDB_CHECK(c, cudaStreamWaitEvent(s0, c->lev[1], 0));   // QR panel k is done
        if (nc > 0) {
            T* A2 = a + k * n + k + band;
            SVDB_TRY(gemm_tn<T>(c, Vq, A2, n, m, nc, band, W));                         // W = V^T A2
            if (has_lq) {
                SVDB_TRY(rank_update<T>(c, A2, n, band, nc, band, V2q, W, nc));          // rows of the LQ panel first
                if (ahead) {
                    SVDB_CHECK(c, cudaEventRecord(c->lev[2], s0));
                    SVDB_CHECK(c, cudaStreamWaitEvent(s1, c->lev[2], 0));
                }
                SVDB_TRY((launch_panel<T, true>(c, A2, n, (int)nc, b, Vl, V2l, s1)));    // LQ panel (look-ahead)
                if (ahead) SVDB_CHECK(c, cudaEventRecord(c->lev[3], s1));
                if (m > band) {
                    c->reserve_now = ahead ? kLookaheadReserve : 0;          // the LQ panel runs beside this
                    const int st = rank_update<T>(c, A2 + band * n, n, m - band, nc, band, V2q + band * band, W, nc);
                    c->reserve_now = 0;
                    SVDB_TRY(st);
                }
            } else {
                SVDB_TRY(rank_update<T>(c, A2, n, m, nc, band, V2q, W, nc));             // A2 += (V S^T) W
            }
        }
        if (has_lq) {
            const size_t mr = m - band;         // rows below the LQ row panel
            if (ahead) SVDB_CHECK(c, cudaStreamWaitEvent(s0, c->lev[3], 0));             // LQ panel is done
            if (mr > 0) {
                T* A3 = a + (k + band) * n + k + band;
                SVDB_TRY(gemm_nn<T>(c, A3, n, mr, nc, band, Vl, W));                     // W = A3 U^T
                SVDB_TRY(rank_update<T>(c, A3, n, mr, band, band, W, V2l, nc));          // columns of the next QR panel first
                if (ahead) {
                    SVDB_CHECK(c, cudaEventRecord(c->lev[2], s0));
                    SVDB_CHECK(c, cudaStreamWaitEvent(s1, c->lev[2], 0));
                }
                SVDB_TRY((launch_panel<T, false>(c, A3, n, (int)mr, b, Vq, V2q, s1)));   // QR panel k+1 (look-ahead)
                if (ahead) SVDB_CHECK(c, cudaEventRecord(c->lev[1], s1));
                if (nc > band) {
                    c->reserve_now = ahead ? kLookaheadReserve : 0;          // QR panel k+1 runs beside this
                    const int st = rank_update<T>(c, A3 + band, n, mr, nc - band, band, W, V2l + band, nc);
                    c->reserve_now = 0;
                    SVDB_TRY(st);
                }
            }
        } else if (nc > 0) {
            // no LQ for this step (only when the trailing block is a single column): next QR panel directly,
            // once the update just enqueued on the main stream has landed
            if (ahead) {
                SVDB_CHECK(c, cudaEventRecord(c->lev[2], s0));
                SVDB_CHECK(c, cudaStreamWaitEvent(s1, c->lev[2], 0));
            }
            SVDB_TRY((launch_panel<T, false>(c, a + (k + band) * n + k + band, n, (int)(m - band), b, Vq, V2q, s1)));
            if (ahead) SVDB_CHECK(c, cudaEventRecord(c->lev[1], s1));
        }
    }
    if (ahead) SVDB_CHECK(c, cudaStreamWaitEvent(s0, c->lev[1], 0));
    return 0;
}

template int stage1_panel_order<float>(Ctx*, float*, size_t, size_t);
template int stage1_panel_order<double>(Ctx*, double*, size_t, size_t);

}  // namespace svdb200

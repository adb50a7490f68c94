// Multi-GPU stage 1 (BASELINE config 4): dense -> band with the matrix distributed 1-D
// block-cyclically over COLUMNS (block = band), one process per GPU, NCCL over NVLink/NVSwitch.
// The reference has no multi-GPU path (SURVEY 2b); the single-GPU panel order
// (cuda_brd_p1, svd_cuda_2.cu:1117) is distributed as follows, per block step k:
//   QR half-step : the owner of block column k factorises the full-height panel locally
//                  (all rows are local under a column distribution) and ncclBroadcast()s
//                  [V | V S^T] (2*m*b elements); every rank updates its local trailing columns
//                  with the same two GEMMs as the single-GPU path.
//   LQ half-step : the b x n' row panel spans all ranks.  Default: Cholesky-QR with reconstructed Householder vectors
//                  (stage1_panel_chol.cu) -- every rank forms the Gram matrix of ITS columns of the row panel, ONE
//                  ncclAllReduce of b^2-sized data in double ([G | top block]), the same b x b algebra on every rank,
//                  then a local pass that leaves U^T and S U in the rank's own layout: a distributed (TSQR-like) panel
//                  with 50 KB of traffic instead of a gather of b*n' elements and a redundant n'-wide factorisation.
//                  The panel's status word is read back by the host (after the concurrent part of the QR update has been
//                  enqueued): a row panel below the pivot-ratio guard -- e.g. the first one of a matrix with a large
//                  common mean -- is redone through the fallback, identically on every rank.
//                  Fallback (also: band not 8/16/32/64, panels narrower than 2 b, svdb200_dist_configure_panels(h, 0)): ncclAllGather of
//                  the local pieces, every rank factorises the SAME assembled panel redundantly.
//                  W = A U^T is a sum over the column distribution: local partial product +
//                  ncclAllReduce(sum) of m' x b, then the local rank-b update.
// Traffic per block step is O(n*b) elements against O(n^2*b/P) flops per rank.
// NCCL is bound at run time (dlopen), so the single-GPU library has no link-time dependency on it.
#include <dlfcn.h>
#include <nccl.h>
#include <new>
#include "common.cuh"

namespace svdb200 {
template <typename T, bool kTrans> int launch_panel_public(Ctx* c, T* a, size_t lda, int m, int b, T* V, T* V2, cudaStream_t stream);
// distributed Cholesky-QR LQ panel (stage1_panel_chol.cu)
size_t chol_dist_buf_elems(int b);
bool chol_dist_supported(const Ctx* c, int b);
template <typename T> int chol_dist_lq_gram(Ctx* c, const T* a2, size_t ldl, int b, int row0, int ncl, bool own_top, double* buf, cudaStream_t stream);
template <typename T> int chol_dist_lq_finish(Ctx* c, T* a2, size_t ldl, int b, int row0, int ncl, bool own_top, const double* buf, T* ut_loc,
                                              T* u2_loc, cudaStream_t stream);
const int* chol_dist_status(Ctx* c);
// distributed Cholesky-QR QR panel: owner part (pass 1, algebra, pack), then the second pass on every rank
size_t chol_dist_qr_elems(size_t m, int b);
const int* chol_dist_qr_status(Ctx* c);
template <typename T> int chol_dist_qr_owner(Ctx* c, T* a, size_t lda, int m, int b, T* qsend, cudaStream_t stream);
template <typename T> int chol_dist_qr_all(Ctx* c, T* qsend, int m, int b, T* V, T* V2, cudaStream_t stream);
template <typename T> int chol_dist_qr_owner_early(Ctx* c, T* a, size_t lda, int m, int b, T* qsend, int phase, cudaStream_t stream);

namespace {

struct NcclApi {
    void* lib = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclBroadcast) Broadcast = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    bool ok = false;
};

NcclApi& nccl() {
    static NcclApi api;
    if (api.lib) return api;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        api.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (api.lib) break;
    }
    if (!api.lib) return api;
#define SVDB_SYM(field, name) api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.lib, name))
    SVDB_SYM(GetUniqueId, "ncclGetUniqueId");
    SVDB_SYM(CommInitRank, "ncclCommInitRank");
    SVDB_SYM(CommDestroy, "ncclCommDestroy");
    SVDB_SYM(Broadcast, "ncclBroadcast");
    SVDB_SYM(AllGather, "ncclAllGather");
    SVDB_SYM(AllReduce, "ncclAllReduce");
    SVDB_SYM(GetErrorString, "ncclGetErrorString");
#undef SVDB_SYM
    api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.Broadcast && api.AllGather && api.AllReduce;
    return api;
}

struct Dist {
    Ctx* ctx = nullptr;          // workspace + stream (created through svdb200_create)
    ncclComm_t comm = nullptr;
    int rank = 0, nranks = 1;
    size_t n = 0, band = 0;
    void* rowpanel = nullptr;    // band x n   : assembled LQ row panel (global column order)
    void* gather = nullptr;      // nranks x band x ncl_max : all-gather landing zone
    void* sendbuf = nullptr;     // band x ncl_max
    void* ut_loc = nullptr;      // ncl_max x band
    void* u2_loc = nullptr;      // band x ncl_max
    void* vv = nullptr;          // [V | V S^T] of a QR panel, contiguous (2 x n x band): ONE broadcast per panel
    void* bandsend = nullptr;    // ncl_max x (band+1) : this rank's band columns, packed
    void* bandall = nullptr;     // nranks x ncl_max x (band+1) : all-gather landing zone
    double* lqbuf = nullptr;     // distributed LQ panel: [tile-packed Gram matrix | top block], all-reduced in double
    int lq_dist = 1;             // 1: LQ panels by local Gram matrix + all-reduce (no gather of the row panel); 0: gather + redundant panel
    int* h_status = nullptr;     // pinned: [0..3] status words of the last distributed LQ panel, [8..11] of the last QR panel
    cudaEvent_t ev_status = nullptr, ev_qstatus = nullptr;
    void* qsend = nullptr;       // QR panel message: raw rows | [M1 | M2] | top blocks of V, V2 | status
    int qr_dist = 1;             // 1: QR panels travel as raw rows + band x band factors (second pass on every rank); 0: [V | V S^T]
    cudaStream_t bc_stream = nullptr;  // the raw QR panel rows are broadcast on this third stream while the owner factorises
    cudaEvent_t ev_raw = nullptr, ev_rawdone = nullptr;
    long long qr_fallbacks = 0;
    long long lq_fallbacks = 0;  // row panels the Cholesky-QR path gave up on (redone through the gather path)
    size_t ncl_max = 0;
};

#define SVDB_NCCL(d, expr)                                                           \
    do {                                                                             \
        ncclResult_t _r = (expr);                                                    \
        if (_r != ncclSuccess) {                                                     \
            (d)->ctx->last_error = std::string(#expr) + ": " +                       \
                                   (nccl().GetErrorString ? nccl().GetErrorString(_r) : "nccl error"); \
            return SVDB200_NCCL_ERR + (int)_r;                                       \
        }                                                                            \
    } while (0)

template <typename T> ncclDataType_t nccl_type();
template <> ncclDataType_t nccl_type<float>() { return ncclFloat32; }
template <> ncclDataType_t nccl_type<double>() { return ncclFloat64; }

// local block lb of rank r holds global block lb * P + r
__host__ __device__ inline size_t first_local_block_after(size_t k, int r, int P) {
    // number of local blocks with global index <= k
    return k >= (size_t)r ? (k - r) / P + 1 : 0;
}

// pack rows [0,b) x local cols [c0, c0+ncl) (ld = ldl) into a contiguous b x ncl_max buffer
template <typename T>
__global__ void pack_rows_kernel(const T* __restrict__ a, size_t ldl, int b, size_t ncl, size_t ncl_max, T* __restrict__ out) {
    size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)b * ncl_max) return;
    size_t r = e / ncl_max, c = e % ncl_max;
    out[e] = c < ncl ? a[r * ldl + c] : (T)0;
}
// gathered [rank][b][ncl_max] -> row panel b x np in global column order.
// Global trailing block t (0-based among the trailing blocks, global block index k+1+t) lives on
// rank (k+1+t) % P at position (its local block index) - (first local trailing block of that rank).
template <typename T>
__global__ void assemble_panel_kernel(const T* __restrict__ gathered, int b, size_t np, size_t ncl_max, size_t k, int P,
                                      T* __restrict__ panel) {
    size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)b * np) return;
    size_t r = e / np, gc = e % np;
    size_t t = gc / b, within = gc % b;
    size_t gblock = k + 1 + t;
    int owner = (int)(gblock % P);
    size_t lb = gblock / P, lb0 = first_local_block_after(k, owner, P);
    size_t lc = (lb - lb0) * b + within;
    panel[r * np + gc] = gathered[((size_t)owner * b + r) * ncl_max + lc];
}
// local slices of the factored panel / reflectors for this rank:
//   a rows [0,b) x local trailing cols  <- panel columns owned by this rank
//   ut_loc (ncl x b) <- Ut (np x b) rows owned ; u2_loc (b x ncl) <- U2 (b x np) columns owned
template <typename T>
__global__ void scatter_local_kernel(const T* __restrict__ panel, const T* __restrict__ ut, const T* __restrict__ u2, int b, size_t np,
                                     size_t ncl, size_t k, int rank, int P, T* __restrict__ a, size_t ldl, T* __restrict__ ut_loc,
                                     T* __restrict__ u2_loc) {
    size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (size_t)b * ncl) return;
    size_t r = e / ncl, lc = e % ncl;
    size_t lb0 = first_local_block_after(k, rank, P);
    size_t gblock = (lb0 + lc / b) * P + rank;
    size_t gc = (gblock - (k + 1)) * b + lc % b;
    a[r * ldl + lc] = panel[r * np + gc];
    u2_loc[r * ncl + lc] = u2[r * np + gc];
    ut_loc[lc * b + r] = ut[gc * b + r];
}

// ---- band hand-off to stage 2 (SURVEY K3 / 8e: "band gathered to one GPU first") --------------------------------------
// Packed band storage, column by column: packed[gc * (b+1) + t] = A[gc - b + t][gc], t = 0 .. b (zero above the matrix) --
// the b+1 diagonals stage 1 leaves, n (b+1) elements instead of n^2.
template <typename T>
__global__ void pack_band_local_kernel(const T* __restrict__ a, size_t ldl, size_t ncl, int b, int rank, int P, T* __restrict__ out) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= ncl * (size_t)(b + 1)) return;
    const size_t lc = e / (b + 1);
    const int t = (int)(e - lc * (b + 1));
    const size_t gc = ((lc / b) * P + rank) * b + lc % b;
    const long long row = (long long)gc - b + t;
    out[e] = row >= 0 ? a[(size_t)row * ldl + lc] : (T)0;
}
// gathered [rank][lc][t] -> packed [gc][t] (global column order)
template <typename T>
__global__ void unpack_band_global_kernel(const T* __restrict__ gathered, size_t n, size_t ncl_max, int b, int P, T* __restrict__ packed) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * (size_t)(b + 1)) return;
    const size_t gc = e / (b + 1);
    const int t = (int)(e - gc * (b + 1));
    const size_t gb = gc / b;
    const int r = (int)(gb % P);
    const size_t lc = (gb / P) * b + gc % b;
    packed[e] = gathered[((size_t)r * ncl_max + lc) * (b + 1) + t];
}

// Look-ahead (same scheme as the single-GPU driver, stage1_panel.cu): the part of an update that the NEXT panel lives in
// is applied first; the panel (and its collective) then runs on the high-priority aux stream s1 while the main stream s0
// finishes the much larger rest of the update.
//   s1: [QR panel k on its owner] Bcast(V) Bcast(V2)            | pack, AllGather, assemble, LQ panel (every rank), scatter
//   s0: W = V^T A2, update of the b rows of the LQ panel ........| rest of the QR update | W = A3 U^T, AllReduce(W),
//       update of the b columns of QR panel k+1 (its owner) -> s1 starts panel k+1 | rest of the LQ update
// QR reflectors live in (v, v2), LQ reflectors in (vb, v2b): a panel in flight never overwrites reflectors that the
// concurrent update still reads.  Every rank issues the collectives in the same order (Bcast, Bcast, AllGather, AllReduce
// per step); NCCL serialises operations of one communicator across streams, which is the order the data needs anyway.
template <typename T>
int dist_stage1(Dist* d, T* a, size_t n, size_t band) {
    Ctx* c = d->ctx;
    const int P = d->nranks, rk = d->rank, b = (int)band;
    const size_t nb = n / band;
    const size_t ldl = svdb200_dist_local_cols(n, band, rk, P);
    T* V = reinterpret_cast<T*>(d->vv);                  // QR reflectors: [V (m x b) | V S^T (m x b)] back to back, one message
    T* V2 = V;                                           // set per panel: V + m * band
    T* Vl = reinterpret_cast<T*>(c->vb);
    T* V2l = reinterpret_cast<T*>(c->v2b);
    T* W = reinterpret_cast<T*>(c->w);
    T* rowpanel = reinterpret_cast<T*>(d->rowpanel);
    T* gathered = reinterpret_cast<T*>(d->gather);
    T* sendbuf = reinterpret_cast<T*>(d->sendbuf);
    T* ut_loc = reinterpret_cast<T*>(d->ut_loc);
    T* u2_loc = reinterpret_cast<T*>(d->u2_loc);
    const bool ahead = !c->profile && c->aux_stream != nullptr;
    cudaStream_t s0 = c->stream, s1 = ahead ? c->aux_stream : c->stream;
    cudaEvent_t evQ = c->lev[1], evR = c->lev[2], evL = c->lev[3], evP = c->lev[0];
    if (ahead) {   // the aux stream must see everything enqueued on the main stream so far
        SVDB_CHECK(c, cudaEventRecord(evP, s0));
        SVDB_CHECK(c, cudaStreamWaitEvent(s1, evP, 0));
    }
    // QR panel k: factorisation on its owner + broadcast of the reflectors.  Fast path (Cholesky-QR panel): the owner runs
    // pass 1 and the b x b algebra and broadcasts the RAW panel rows with the small factors; every rank then forms
    // [V | V S^T] with the second pass on its copy -- half the bytes of broadcasting [V | V S^T], and the copy arrives in the
    // layout the update reads.  The panel's status word travels with the message and is read by the host in qr_panel_finish
    // (top of the step that needs V): a panel below the pivot-ratio guard is redone by the exchange-based kernels on the owner
    // and broadcast as [V | V S^T], identically decided on every rank.
    bool qr_pending = false;
    size_t qr_pending_k = 0;
    auto qr_panel_slow = [&](size_t k, bool allow_chol) -> int {
        const size_t o = k * band, m = n - o;
        const int owner = (int)(k % P);
        T* v2k = V + m * band;
        if (rk == owner) {
            const int keep = c->cfg.panel_chol;
            if (!allow_chol) c->cfg.panel_chol = 0;
            const int st = launch_panel_public<T, false>(c, a + o * ldl + (k / P) * band, ldl, (int)m, b, V, v2k, s1);
            c->cfg.panel_chol = keep;
            SVDB_TRY(st);
        }
        if (P > 1) SVDB_NCCL(d, nccl().Broadcast(V, V, 2 * m * band, nccl_type<T>(), owner, d->comm, s1));
        return 0;
    };
    auto qr_panel_and_bcast = [&](size_t k) -> int {
        const size_t o = k * band, m = n - o;
        const int owner = (int)(k % P);
        qr_pending = false;
        if (P > 1 && d->qr_dist && chol_dist_supported(c, b) && m >= 2 * band) {
            T* qs = reinterpret_cast<T*>(d->qsend);
            if (ahead && d->bc_stream) {
                // the raw rows travel on a third stream while the owner runs pass 1 and the algebra on its copy; the small
                // tail of the message ([M1 | M2], top blocks, status) follows on s1.  Every rank issues the two broadcasts
                // in this order.
                cudaStream_t s2 = d->bc_stream;
                const size_t nraw = (m - band) * band, ntail = 4 * band * band + 4;
                if (rk == owner) SVDB_TRY(chol_dist_qr_owner_early<T>(c, a + o * ldl + (k / P) * band, ldl, (int)m, b, qs, 0, s1));
                SVDB_CHECK(c, cudaEventRecord(d->ev_raw, s1));                 // (non-owners: the previous panel's copy has been consumed)
                SVDB_CHECK(c, cudaStreamWaitEvent(s2, d->ev_raw, 0));
                SVDB_NCCL(d, nccl().Broadcast(qs, qs, nraw, nccl_type<T>(), owner, d->comm, s2));
                SVDB_CHECK(c, cudaEventRecord(d->ev_rawdone, s2));
                if (rk == owner) SVDB_TRY(chol_dist_qr_owner_early<T>(c, a + o * ldl + (k / P) * band, ldl, (int)m, b, qs, 1, s1));
                SVDB_NCCL(d, nccl().Broadcast(qs + nraw, qs + nraw, ntail, nccl_type<T>(), owner, d->comm, s1));
                SVDB_CHECK(c, cudaStreamWaitEvent(s1, d->ev_rawdone, 0));
            } else {
                if (rk == owner) SVDB_TRY(chol_dist_qr_owner<T>(c, a + o * ldl + (k / P) * band, ldl, (int)m, b, qs, s1));
                SVDB_NCCL(d, nccl().Broadcast(qs, qs, chol_dist_qr_elems(m, b), nccl_type<T>(), owner, d->comm, s1));
            }
            SVDB_TRY(chol_dist_qr_all<T>(c, qs, (int)m, b, V, V + m * band, s1));
            SVDB_CHECK(c, cudaMemcpyAsync(d->h_status + 8, chol_dist_qr_status(c), 4 * sizeof(int), cudaMemcpyDeviceToHost, s1));
            SVDB_CHECK(c, cudaEventRecord(d->ev_qstatus, s1));
            qr_pending = true;
            qr_pending_k = k;
            return 0;
        }
        SVDB_TRY(qr_panel_slow(k, true));
        if (ahead) SVDB_CHECK(c, cudaEventRecord(evQ, s1));
        return 0;
    };
    auto qr_panel_finish = [&]() -> int {
        if (!qr_pending) return 0;
        qr_pending = false;
        SVDB_CHECK(c, cudaEventSynchronize(d->ev_qstatus));
        if (d->h_status[8] != 0) {
            d->qr_fallbacks++;
            SVDB_TRY(qr_panel_slow(qr_pending_k, false));
        }
        if (ahead) SVDB_CHECK(c, cudaEventRecord(evQ, s1));
        return 0;
    };
    SVDB_TRY(qr_panel_and_bcast(0));
    for (size_t k = 0; k < nb; ++k) {
        const size_t o = k * band, m = n - o;
        const bool has_lq = (o + band < n - 1);
        const size_t lb0 = first_local_block_after(k, rk, P);        // first local block with global index > k
        const size_t ncl = ldl - lb0 * band;                         // local trailing columns
        V2 = V + m * band;
        // ---- QR half-step ------------------------------------------------------------------------------
        SVDB_TRY(qr_panel_finish());                                 // (host: status of panel k; fallback if it was given up)
        if (ahead) SVDB_CHECK(c, cudaStreamWaitEvent(s0, evQ, 0));   // reflectors of panel k have arrived
        T* A2 = a + o * ldl + lb0 * band;
        if (ncl > 0) {
            SVDB_TRY(gemm_tn<T>(c, V, A2, ldl, m, ncl, band, W));
            if (has_lq) SVDB_TRY(rank_update<T>(c, A2, ldl, band, ncl, band, V2, W, ncl));               // rows of the LQ panel first
            else SVDB_TRY(rank_update<T>(c, A2, ldl, m, ncl, band, V2, W, ncl));
        }
        if (!has_lq) {
            // last steps: no LQ; the next QR panel (if any) follows directly
            if (k + 1 < nb) {
                if (ahead) { SVDB_CHECK(c, cudaEventRecord(evP, s0)); SVDB_CHECK(c, cudaStreamWaitEvent(s1, evP, 0)); }
                SVDB_TRY(qr_panel_and_bcast(k + 1));
            }
            continue;
        }
        // ---- LQ half-step ------------------------------------------------------------------------------
        const size_t np = n - o - band;                              // global width of the row panel
        const size_t mr = m - band;
        if (ahead) { SVDB_CHECK(c, cudaEventRecord(evR, s0)); SVDB_CHECK(c, cudaStreamWaitEvent(s1, evR, 0)); }
        const bool own_top = (int)((k + 1) % P) == rk && ncl > 0;          // my first b trailing columns are the panel's top block
        // s1: gather the b x np row panel on every rank, factorise it redundantly, scatter the local slices
        auto lq_gather_path = [&]() -> int {
            size_t cnt = (size_t)b * d->ncl_max;
            pack_rows_kernel<T><<<(unsigned)((cnt + 255) / 256), 256, 0, s1>>>(A2, ldl, b, ncl, d->ncl_max, sendbuf);
            c->launches++;
            if (P > 1) SVDB_NCCL(d, nccl().AllGather(sendbuf, gathered, cnt, nccl_type<T>(), d->comm, s1));
            else SVDB_CHECK(c, cudaMemcpyAsync(gathered, sendbuf, cnt * sizeof(T), cudaMemcpyDeviceToDevice, s1));
            size_t tot = (size_t)b * np;
            assemble_panel_kernel<T><<<(unsigned)((tot + 255) / 256), 256, 0, s1>>>(gathered, b, np, d->ncl_max, k, P, rowpanel);
            c->launches++;
            // every rank factorises the same panel: Ut (np x b) -> vb, U2 (b x np) -> v2b
            SVDB_TRY((launch_panel_public<T, true>(c, rowpanel, np, (int)np, b, Vl, V2l, s1)));
            if (ncl > 0) {
                size_t cnt2 = (size_t)b * ncl;
                scatter_local_kernel<T><<<(unsigned)((cnt2 + 255) / 256), 256, 0, s1>>>(rowpanel, Vl, V2l, b, np, ncl, k, rk, P, A2, ldl,
                                                                                        ut_loc, u2_loc);
                c->launches++;
            }
            return 0;
        };
        bool lq_pending = false;
        if (d->lq_dist && chol_dist_supported(c, b) && np >= 2 * band) {
            // s1: local Gram matrix -> all-reduce -> algebra (every rank) -> local second pass (gated on the guard); the
            // status word comes back to the host, which looks at it only after the rest of the QR update is enqueued
            const int row0 = own_top ? b : 0;
            SVDB_TRY(chol_dist_lq_gram<T>(c, A2, ldl, b, row0, (int)ncl, own_top, d->lqbuf, s1));
            if (P > 1) SVDB_NCCL(d, nccl().AllReduce(d->lqbuf, d->lqbuf, chol_dist_buf_elems(b), ncclFloat64, ncclSum, d->comm, s1));
            SVDB_TRY(chol_dist_lq_finish<T>(c, A2, ldl, b, row0, (int)ncl, own_top, d->lqbuf, ut_loc, u2_loc, s1));
            SVDB_CHECK(c, cudaMemcpyAsync(d->h_status, chol_dist_status(c), 4 * sizeof(int), cudaMemcpyDeviceToHost, s1));
            SVDB_CHECK(c, cudaEventRecord(d->ev_status, s1));
            lq_pending = true;
        } else {
            SVDB_TRY(lq_gather_path());
            if (ahead) SVDB_CHECK(c, cudaEventRecord(evL, s1));
        }
        // s0: the rest of the QR update runs beside the LQ panel
        if (ncl > 0 && mr > 0) {
            c->reserve_now = ahead ? kLookaheadReserve : 0;                  // the LQ panel runs beside this
            const int st = rank_update<T>(c, A2 + band * ldl, ldl, mr, ncl, band, V2 + band * band, W, ncl);
            c->reserve_now = 0;
            SVDB_TRY(st);
        }
        if (lq_pending) {
            // Identical numbers on every rank => identical status => every rank takes the same branch (and issues the same
            // collectives).  A row panel whose pivot ratio fell below the guard was left untouched: redo it by the gather path.
            SVDB_CHECK(c, cudaEventSynchronize(d->ev_status));
            if (d->h_status[0] != 0) {
                d->lq_fallbacks++;
                SVDB_TRY(lq_gather_path());
            }
            if (ahead) SVDB_CHECK(c, cudaEventRecord(evL, s1));
        }
        if (ahead) SVDB_CHECK(c, cudaStreamWaitEvent(s0, evL, 0));
        if (mr > 0) {
            T* A3 = a + (o + band) * ldl + lb0 * band;
            if (ncl > 0) SVDB_TRY(gemm_nn<T>(c, A3, ldl, mr, ncl, band, ut_loc, W));
            else SVDB_CHECK(c, cudaMemsetAsync(W, 0, mr * band * sizeof(T), s0));
            if (P > 1) SVDB_NCCL(d, nccl().AllReduce(W, W, mr * band, nccl_type<T>(), ncclSum, d->comm, s0));
            const bool own_next = (int)((k + 1) % P) == rk && ncl > 0;     // my first b trailing columns are QR panel k+1
            if (own_next) SVDB_TRY(rank_update<T>(c, A3, ldl, mr, band, band, W, u2_loc, ncl));   // columns of the next QR panel first
            if (ahead) { SVDB_CHECK(c, cudaEventRecord(evP, s0)); SVDB_CHECK(c, cudaStreamWaitEvent(s1, evP, 0)); }
            if (!ahead && ncl > 0) {
                // single stream: finish the update before the next panel
                if (own_next) { if (ncl > band) SVDB_TRY(rank_update<T>(c, A3 + band, ldl, mr, ncl - band, band, W, u2_loc + band, ncl)); }
                else SVDB_TRY(rank_update<T>(c, A3, ldl, mr, ncl, band, W, u2_loc, ncl));
            }
            SVDB_TRY(qr_panel_and_bcast(k + 1));                           // s1: panel k+1 + broadcast
            if (ahead && ncl > 0) {
                c->reserve_now = kLookaheadReserve;                          // QR panel k+1 (on its owner) runs beside this
                int st = 0;
                if (own_next) { if (ncl > band) st = rank_update<T>(c, A3 + band, ldl, mr, ncl - band, band, W, u2_loc + band, ncl); }
                else st = rank_update<T>(c, A3, ldl, mr, ncl, band, W, u2_loc, ncl);
                c->reserve_now = 0;
                SVDB_TRY(st);
            }
        } else if (k + 1 < nb) {
            if (ahead) { SVDB_CHECK(c, cudaEventRecord(evP, s0)); SVDB_CHECK(c, cudaStreamWaitEvent(s1, evP, 0)); }
            SVDB_TRY(qr_panel_and_bcast(k + 1));
        }
    }
    SVDB_TRY(qr_panel_finish());
    if (ahead) {   // everything the aux stream did is ordered before the caller's next work on the main stream
        SVDB_CHECK(c, cudaEventRecord(evQ, s1));
        SVDB_CHECK(c, cudaStreamWaitEvent(s0, evQ, 0));
    }
    SVDB_CHECK(c, cudaGetLastError());
    return 0;
}

// every rank ends up with the packed band (n x (b+1), global column order) in `packed`
template <typename T>
int dist_gather_band(Dist* d, const T* a, T* packed) {
    Ctx* c = d->ctx;
    const int P = d->nranks, rk = d->rank, b = (int)d->band;
    const size_t n = d->n, ldl = svdb200_dist_local_cols(n, d->band, rk, P);
    T* sendb = reinterpret_cast<T*>(d->bandsend);
    T* all = reinterpret_cast<T*>(d->bandall);
    const size_t cnt = d->ncl_max * (size_t)(b + 1);
    cudaStream_t s0 = c->stream;
    SVDB_CHECK(c, cudaMemsetAsync(sendb, 0, cnt * sizeof(T), s0));
    if (ldl > 0) {
        const size_t tot = ldl * (size_t)(b + 1);
        pack_band_local_kernel<T><<<(unsigned)((tot + 255) / 256), 256, 0, s0>>>(a, ldl, ldl, b, rk, P, sendb);
        c->launches++;
    }
    if (P > 1) SVDB_NCCL(d, nccl().AllGather(sendb, all, cnt, nccl_type<T>(), d->comm, s0));
    else SVDB_CHECK(c, cudaMemcpyAsync(all, sendb, cnt * sizeof(T), cudaMemcpyDeviceToDevice, s0));
    const size_t tot = n * (size_t)(b + 1);
    unpack_band_global_kernel<T><<<(unsigned)((tot + 255) / 256), 256, 0, s0>>>(all, n, d->ncl_max, b, P, packed);
    c->launches++;
    SVDB_CHECK(c, cudaGetLastError());
    return 0;
}

// stage 1 distributed, then the band goes to rank 0, which runs stage 2 on the packed band and the singular values
// (replicas only there: one sequential wavefront over an O(n b) band, SURVEY 8e)
template <typename T>
int dist_svdvals(Dist* d, T* a, T* sigma) {
    Ctx* c = d->ctx;
    const size_t n = d->n, band = d->band;
    SVDB_TRY(dist_stage1<T>(d, a, n, band));
    void* pk = nullptr;
    SVDB_CHECK(c, cudaMalloc(&pk, sizeof(T) * n * (band + 1)));
    T* packed = reinterpret_cast<T*>(pk);
    int st = dist_gather_band<T>(d, a, packed);
    if (st == 0 && d->rank == 0) {
        st = stage2_chase_packed<T>(c, packed, n, band, reinterpret_cast<T*>(c->d), reinterpret_cast<T*>(c->e));
        if (st == 0) st = bidiag_qr<T>(c, reinterpret_cast<T*>(c->d), reinterpret_cast<T*>(c->e), n, sigma);
    }
    cudaStreamSynchronize(c->stream);
    cudaFree(pk);
    return st;
}

}  // namespace
}  // namespace svdb200

using namespace svdb200;

extern "C" {

size_t svdb200_dist_local_cols(size_t n, size_t band, int rank, int nranks) {
    if (band == 0 || nranks <= 0 || n % band != 0 || rank < 0 || rank >= nranks) return 0;
    size_t nb = n / band, mine = nb / nranks + ((size_t)rank < nb % nranks ? 1 : 0);
    return mine * band;
}

int svdb200_dist_unique_id(void* out128) {
    if (!out128) return SVDB200_E_ARG;
    if (!nccl().ok) return SVDB200_E_STATE;
    ncclUniqueId id;
    ncclResult_t r = nccl().GetUniqueId(&id);
    if (r != ncclSuccess) return SVDB200_NCCL_ERR + (int)r;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    std::memcpy(out128, &id, 128);
    return 0;
}

int svdb200_dist_create(svdb200_dist_handle* out, int device, int rank, int nranks, const void* nccl_unique_id, size_t n, size_t band,
                        int dtype) {
    if (!out || nranks < 1 || rank < 0 || rank >= nranks) return SVDB200_E_ARG;
    if (band == 0 || n == 0 || n % band != 0) return SVDB200_E_SHAPE;
    if (nranks > 1 && (!nccl_unique_id || !nccl().ok)) return SVDB200_E_STATE;
    Dist* d = new (std::nothrow) Dist();
    if (!d) return SVDB200_E_STATE;
    svdb200_handle h = nullptr;
    int st = svdb200_create(&h, device, n, band, dtype);
    if (st != 0) { delete d; return st; }
    d->ctx = reinterpret_cast<Ctx*>(h);
    d->rank = rank; d->nranks = nranks; d->n = n; d->band = band;
    const size_t es = d->ctx->esz;
    d->ncl_max = (n / band + nranks - 1) / nranks * band;
    cudaError_t e = cudaSuccess;
    if (e == cudaSuccess) e = cudaMalloc(&d->rowpanel, es * band * n);
    if (e == cudaSuccess) e = cudaMalloc(&d->gather, es * (size_t)nranks * band * d->ncl_max);
    if (e == cudaSuccess) e = cudaMalloc(&d->sendbuf, es * band * d->ncl_max);
    if (e == cudaSuccess) e = cudaMalloc(&d->ut_loc, es * band * d->ncl_max);
    if (e == cudaSuccess) e = cudaMalloc(&d->u2_loc, es * band * d->ncl_max);
    if (e == cudaSuccess) e = cudaMalloc(&d->vv, es * 2 * (n + 256) * band);
    if (e == cudaSuccess) e = cudaMalloc(&d->bandsend, es * d->ncl_max * (band + 1));
    if (e == cudaSuccess) e = cudaMalloc(&d->bandall, es * (size_t)nranks * d->ncl_max * (band + 1));
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&d->lqbuf), sizeof(double) * (chol_dist_buf_elems((int)band) + 64));
    if (e == cudaSuccess) e = cudaHostAlloc(reinterpret_cast<void**>(&d->h_status), 64, cudaHostAllocDefault);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d->ev_status, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d->ev_qstatus, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d->ev_raw, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d->ev_rawdone, cudaEventDisableTiming);
    if (e == cudaSuccess) {
        int lo = 0, hi = 0;
        e = cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&d->bc_stream, cudaStreamNonBlocking, hi);
    }
    if (e == cudaSuccess) e = cudaMalloc(&d->qsend, es * ((n + 256) * band + 4 * band * band + 64));
    if (e != cudaSuccess) { int s2 = cuda_status(d->ctx, e, "cudaMalloc(dist)"); svdb200_dist_destroy(reinterpret_cast<svdb200_dist_handle>(d)); return s2; }
    if (nranks > 1) {
        ncclUniqueId id;
        std::memcpy(&id, nccl_unique_id, 128);
        ncclResult_t r = nccl().CommInitRank(&d->comm, nranks, id, rank);
        if (r != ncclSuccess) { svdb200_dist_destroy(reinterpret_cast<svdb200_dist_handle>(d)); return SVDB200_NCCL_ERR + (int)r; }
    }
    *out = reinterpret_cast<svdb200_dist_handle>(d);
    return 0;
}

int svdb200_dist_destroy(svdb200_dist_handle h) {
    if (!h) return SVDB200_E_ARG;
    Dist* d = reinterpret_cast<Dist*>(h);
    if (d->ctx) { cudaSetDevice(d->ctx->device); cudaStreamSynchronize(d->ctx->stream); }
    if (d->comm) nccl().CommDestroy(d->comm);
    void* ptrs[] = {d->rowpanel, d->gather, d->sendbuf, d->ut_loc, d->u2_loc, d->vv, d->bandsend, d->bandall, d->lqbuf, d->qsend};
    for (void* p : ptrs) if (p) cudaFree(p);
    if (d->h_status) cudaFreeHost(d->h_status);
    if (d->ev_status) cudaEventDestroy(d->ev_status);
    if (d->ev_qstatus) cudaEventDestroy(d->ev_qstatus);
    if (d->ev_raw) cudaEventDestroy(d->ev_raw);
    if (d->ev_rawdone) cudaEventDestroy(d->ev_rawdone);
    if (d->bc_stream) { cudaStreamSynchronize(d->bc_stream); cudaStreamDestroy(d->bc_stream); }
    if (d->ctx) svdb200_destroy(reinterpret_cast<svdb200_handle>(d->ctx));
    delete d;
    return 0;
}

int svdb200_dist_set_stream(svdb200_dist_handle h, void* stream) {
    if (!h) return SVDB200_E_ARG;
    return svdb200_set_stream(reinterpret_cast<svdb200_handle>(reinterpret_cast<Dist*>(h)->ctx), stream);
}

long long svdb200_dist_launch_count(svdb200_dist_handle h) { return h ? reinterpret_cast<Dist*>(h)->ctx->launches : -1; }
long long svdb200_dist_lq_fallback_count(svdb200_dist_handle h) { return h ? reinterpret_cast<Dist*>(h)->lq_fallbacks + reinterpret_cast<Dist*>(h)->qr_fallbacks : -1; }

int svdb200_dist_dense_to_band_dev_f32(svdb200_dist_handle h, float* a, size_t n, size_t band) {
    if (!h || !a) return SVDB200_E_ARG;
    Dist* d = reinterpret_cast<Dist*>(h);
    if (d->ctx->dtype != SVDB200_F32 || n != d->n || band != d->band) return SVDB200_E_ARG;
    SVDB_CHECK(d->ctx, cudaSetDevice(d->ctx->device));
    return dist_stage1<float>(d, a, n, band);
}
int svdb200_dist_dense_to_band_dev_f64(svdb200_dist_handle h, double* a, size_t n, size_t band) {
    if (!h || !a) return SVDB200_E_ARG;
    Dist* d = reinterpret_cast<Dist*>(h);
    if (d->ctx->dtype != SVDB200_F64 || n != d->n || band != d->band) return SVDB200_E_ARG;
    SVDB_CHECK(d->ctx, cudaSetDevice(d->ctx->device));
    return dist_stage1<double>(d, a, n, band);
}

#define SVDB_DIST_TYPED(T, S, CODE)                                                                                  \
    int svdb200_dist_gather_band_dev_##S(svdb200_dist_handle h, const T* a_local, T* packed) {                       \
        if (!h || !a_local || !packed) return SVDB200_E_ARG;                                                         \
        Dist* d = reinterpret_cast<Dist*>(h);                                                                        \
        if (d->ctx->dtype != CODE) return SVDB200_E_ARG;                                                             \
        SVDB_CHECK(d->ctx, cudaSetDevice(d->ctx->device));                                                           \
        return dist_gather_band<T>(d, a_local, packed);                                                              \
    }                                                                                                                \
    int svdb200_dist_svdvals_dev_##S(svdb200_dist_handle h, T* a_local, T* sigma) {                                  \
        if (!h || !a_local) return SVDB200_E_ARG;                                                                    \
        Dist* d = reinterpret_cast<Dist*>(h);                                                                        \
        if (d->ctx->dtype != CODE || (d->rank == 0 && !sigma)) return SVDB200_E_ARG;                                 \
        SVDB_CHECK(d->ctx, cudaSetDevice(d->ctx->device));                                                           \
        return dist_svdvals<T>(d, a_local, sigma);                                                                   \
    }
SVDB_DIST_TYPED(float, f32, SVDB200_F32)
SVDB_DIST_TYPED(double, f64, SVDB200_F64)
#undef SVDB_DIST_TYPED

int svdb200_dist_configure_panels(svdb200_dist_handle h, int lq_distributed) {
    if (!h || lq_distributed < 0 || lq_distributed > 1) return SVDB200_E_ARG;
    reinterpret_cast<Dist*>(h)->lq_dist = lq_distributed;
    reinterpret_cast<Dist*>(h)->qr_dist = lq_distributed;
    return 0;
}

int svdb200_dist_configure(svdb200_dist_handle h, int stage2_schedule, int qr_method, int tc05_mode) {
    if (!h) return SVDB200_E_ARG;
    Dist* d = reinterpret_cast<Dist*>(h);
    svdb200_handle ch = reinterpret_cast<svdb200_handle>(d->ctx);
    if (stage2_schedule >= 0) SVDB_TRY(svdb200_set_stage2_schedule(ch, stage2_schedule));
    if (qr_method >= 0) SVDB_TRY(svdb200_set_qr_method(ch, qr_method, 0));
    if (tc05_mode >= 0) SVDB_TRY(svdb200_set_tc05(ch, tc05_mode, 0));
    return 0;
}

}  // extern "C"

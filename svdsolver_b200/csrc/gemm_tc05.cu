// FP32 compact-WY trailing update of stage 1 on the 5th-generation tensor cores:
// TMA-fed tcgen05.mma (kind::tf32) with the accumulator in TMEM, error-compensated 3xTF32.
//
// Replaces qr_apply / lq_apply (svd_parallel.h:243-281; GPU: svd_cuda_2.cu:1039-1110) for T = float at
// panel widths 32 / 64.  FP64 cannot take this path: tcgen05.mma has no f64 kind (SURVEY 0.6), it stays
// on the DMMA kernels of gemm_fast.cu.
//
// Every fp32 operand x is used as x = hi + lo with hi = x rounded / truncated to TF32 and lo = x - hi
// (exact in fp32); a product is accumulated as lo*hi + hi*lo + hi*hi in fp32 in TMEM, which keeps
// ~2^-21 relative accuracy through the n/b chained updates (a single TF32 pass, 2^-11, does not hold
// the 1e-4 tolerance).
//
//   rank_update_tc05_kernel : C(MxN) += P(MxK) Q(KxN), K = b.  Persistent, one CTA per SM.  P tile
//       resident, Q tiles streamed, both pre-split in HBM (they are O(n b)); the 128x128 accumulator is
//       double-buffered in TMEM; C moves HBM -> smem -> HBM by TMA through a ring of 128x32 sub-tiles
//       that the epilogue warps update in place (tcgen05.ld + add).  HBM-bound: 8 bytes per 2b flops.
//   gemm_tc05_kernel<NN>    : W(Mxb) = C(MxN) Ut(Nxb)      A = C tile, K-major
//   gemm_tc05_kernel<TN>    : W(bxN) = V(Mxb)^T C(MxN)     A = C^T tile, MN-major (no transpose pass)
//       C is streamed once by TMA; four warps split each landed tile into hi (in place) and lo on
//       chip, one thread issues the three MMAs per k-step into TMEM; four drain warps fold the
//       double-buffered partial accumulators into register sums every 256 k (see gemm_tc05_kernel).
//
// Warp roles: warp 0 TMA producer, warp 1 MMA issuer + TMEM allocator, warps 2-5 epilogue (rank update)
// or split (GEMMs), warps 6-9 drain (GEMMs); warp w owns TMEM lanes 32*(w%4) .. +31.  All waits are
// mbarrier based.
#include <cuda.h>
#include "common.cuh"

namespace svdb200 {

template <typename T> int rank_update_tc05(Ctx*, T*, size_t, int, int, int, const T*, const T*, size_t);
template <typename T> int gemm_tn_tc05(Ctx*, const T*, const T*, size_t, int, int, int, T*);
template <typename T> int gemm_nn_tc05(Ctx*, const T*, size_t, int, int, int, const T*, T*);

namespace tc05 {

constexpr int kThreads = 192;
constexpr unsigned long long kWatchdogNs = 4000000000ull;   // a stuck mbarrier traps instead of hanging the GPU

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    const unsigned long long t0 = gtime();
    uint32_t polls = 0;
    while (!mbar_try_wait(bar, parity)) {
        if ((++polls & 1023u) == 0 && gtime() - t0 > kWatchdogNs) __trap();
    }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int x, int y) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int x, int y) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(src), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void prefetch_map(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem] * B[smem], TF32 inputs, FP32 accumulate; issued by ONE thread for the CTA
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// mbarrier arrives once every tcgen05 operation issued so far by this thread has completed
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives TMEM lane (base lane + t)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t rna_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- descriptors ------------------------------------------------------------------------------------
// Shared-memory matrix descriptor, SWIZZLE_128B (the layout TMA writes with CU_TENSOR_MAP_SWIZZLE_128B):
// bits [0,14) start address >> 4, [16,30) leading byte offset >> 4, [32,46) stride byte offset >> 4,
// [46,48) version = 1 (sm_100), [61,64) layout type = 2.
//   (kind::tf32 reads fp32 words and ignores their low 13 mantissa bits: truncation, not rounding.)
//   K-major operand : rows of 128 B (32 tf32 along K), 8-row groups SBO apart; one MMA (K = 8) reads 32 B
//                     of every row, the k-step advances the start address by 32 B inside the swizzle atom.
//   MN-major operand: see make_desc_mn.
__device__ __forceinline__ uint64_t make_desc_raw(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout << 61;
    return d;
}
// K-major operand, SWIZZLE_128B (16-byte chunks XOR row%8; TMA: CU_TENSOR_MAP_SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return make_desc_raw(saddr, lbo_bytes, sbo_bytes, 2u);
}
// MN-major TF32 operand: the only legal swizzled layout is SWIZZLE_128B_BASE32B (32-byte chunks XOR k-row%4;
// TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B).  Slabs of 32 elements along M/N (128 B) x k rows at a 128 B pitch;
// the K atom is 4 rows (SBO = 512 B), LBO = slab stride; one MMA (K = 8) reads two K atoms, the k-step advances
// the start address by 1024 B.
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t saddr, uint32_t slab_bytes) {
    return make_desc_raw(saddr, slab_bytes, 512u, 1u);
}
// Instruction descriptor (upper 32 bits of the 64-bit idesc): c_format f32 (1 @4), a/b format tf32 (2 @7, 2 @10),
// a_major @15, b_major @16 (1 = MN-major), N >> 3 @17, M >> 4 @24.
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn, int b_mn) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
           ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- operand pre-split (small operands only: O(n b) elements) ----------------------------------------
__global__ void split_tf32_kernel(const float* __restrict__ src, size_t ld_src, int rows, int cols, float* __restrict__ hi,
                                  float* __restrict__ lo, size_t ld_dst) {
    const size_t total = (size_t)rows * cols;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / cols), c = (int)(e - (size_t)r * cols);
        const float x = src[(size_t)r * ld_src + c];
        const uint32_t h = rna_tf32(x);
        const uint32_t l = rna_tf32(x - __uint_as_float(h));
        hi[(size_t)r * ld_dst + c] = __uint_as_float(h);
        lo[(size_t)r * ld_dst + c] = __uint_as_float(l);
    }
}

// =====================================================================================================
// C(MxN) += P(MxK) Q(KxN)
// =====================================================================================================
template <int K> struct RuCfg {
    static constexpr int kPBytes = 128 * K * 4;          // one of {hi, lo}: K/32 blocks of 128 rows x 128 B
    static constexpr int kQBytes = K * 128 * 4;          // one of {hi, lo}: 4 slabs of K rows x 128 B
    static constexpr int kStage = 128 * 32 * 4;          // C sub-tile: 128 rows x 32 columns
    static constexpr int kRing = K == 64 ? 6 : 8;
    static constexpr int kBarBytes = 256;
    static constexpr int kSmem = 1024 + 2 * kPBytes + 2 * kQBytes + kRing * kStage + kBarBytes;
};

template <int K>
__global__ void __launch_bounds__(kThreads, 1)
rank_update_tc05_kernel(const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmPh,
                        const __grid_constant__ CUtensorMap tmPl, const __grid_constant__ CUtensorMap tmQh,
                        const __grid_constant__ CUtensorMap tmQl, int RB, int NT, int chunk_tiles, int NCH) {
    using Cfg = RuCfg<K>;
    constexpr int R = Cfg::kRing;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* gbase = smem_raw + (base - raw);
    const uint32_t sPh = base, sPl = sPh + Cfg::kPBytes, sQh = sPl + Cfg::kPBytes, sQl = sQh + Cfg::kQBytes;
    const uint32_t sC = sQl + Cfg::kQBytes;
    unsigned char* gC = gbase + (sC - base);
    const uint32_t sBar = sC + R * Cfg::kStage;
    const uint32_t bPFull = sBar, bPFree = sBar + 8, bQFull = sBar + 16, bQFree = sBar + 24;
    const uint32_t bTFull = sBar + 32, bTEmpty = sBar + 48, bCFull = sBar + 64;        // [2], [2], [R]
    const uint32_t sSlot = bCFull + 8 * R;
    volatile uint32_t* slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + (sSlot - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nitems = RB * NCH;

    if (threadIdx.x == 0) {
        mbar_init(bPFull, 1); mbar_init(bPFree, 1); mbar_init(bQFull, 1); mbar_init(bQFree, 1);
        mbar_init(bTFull, 1); mbar_init(bTFull + 8, 1);
        mbar_init(bTEmpty, 4); mbar_init(bTEmpty + 8, 4);
        for (int i = 0; i < R; ++i) mbar_init(bCFull + 8 * i, 1);
        fence_barrier_init();
        prefetch_map(&tmC); prefetch_map(&tmPh); prefetch_map(&tmPl); prefetch_map(&tmQh); prefetch_map(&tmQl);
    }
    if (warp == 1) tmem_alloc(sSlot, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *slot_ptr;

    if (warp == 0) {
        // ================= TMA producer: P once per item, Q once per tile =================
        if (lane == 0) {
            int g = 0, it = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
                const int ch = item / RB, rb = item - ch * RB;
                const int t0 = ch * chunk_tiles, t1 = min(NT, t0 + chunk_tiles);
                if (it > 0) mbar_wait(bPFree, (it - 1) & 1);
                mbar_expect_tx(bPFull, 2 * Cfg::kPBytes);
#pragma unroll
                for (int kb = 0; kb < K / 32; ++kb) {
                    tma_load_2d(sPh + kb * 16384, &tmPh, bPFull, kb * 32, rb * 128);
                    tma_load_2d(sPl + kb * 16384, &tmPl, bPFull, kb * 32, rb * 128);
                }
                for (int t = t0; t < t1; ++t, ++g) {
                    if (g > 0) mbar_wait(bQFree, (g - 1) & 1);
                    mbar_expect_tx(bQFull, 2 * Cfg::kQBytes);
#pragma unroll
                    for (int sl = 0; sl < 4; ++sl) {
                        tma_load_2d(sQh + sl * (K * 128), &tmQh, bQFull, t * 128 + sl * 32, 0);
                        tma_load_2d(sQl + sl * (K * 128), &tmQl, bQFull, t * 128 + sl * 32, 0);
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(128, 128, 0, 1);
            int g = 0, it = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++it) {
                const int ch = item / RB;
                const int t0 = ch * chunk_tiles, t1 = min(NT, t0 + chunk_tiles);
                mbar_wait(bPFull, it & 1);
                for (int t = t0; t < t1; ++t, ++g) {
                    const int buf = g & 1;
                    mbar_wait(bQFull, g & 1);
                    if (g >= 2) mbar_wait(bTEmpty + 8 * buf, ((g >> 1) - 1) & 1);
                    tc_fence_after();
                    const uint32_t d = tmem + buf * 128;
                    uint32_t acc = 0;
#pragma unroll
                    for (int pass = 0; pass < 3; ++pass) {
                        const uint32_t pa = pass == 0 ? sPl : sPh;       // lo*hi, hi*lo, hi*hi
                        const uint32_t qb = pass == 1 ? sQl : sQh;
#pragma unroll
                        for (int ks = 0; ks < K / 8; ++ks) {
                            const uint64_t ad = make_desc(pa + (ks >> 2) * 16384 + (ks & 3) * 32, 16, 1024);
                            const uint64_t bd = make_desc_mn(qb + ks * 1024, K * 128);
                            mma_tf32(d, ad, bd, idesc, acc);
                            acc = 1;
                        }
                    }
                    mma_commit(bQFree);
                    mma_commit(bTFull + 8 * buf);
                }
                mma_commit(bPFree);
            }
        }
    } else {
        // ================= epilogue: C sub-tile += accumulator, in place in the staging ring =================
        const int quad = warp & 3;
        const int row = quad * 32 + lane;
        const bool leader = (warp == 2 && lane == 0);
        struct Cur { int item, t, j, rb, t1; };
        auto cur_set = [&](Cur& c) {
            if (c.item < nitems) {
                const int ch = c.item / RB;
                c.rb = c.item - ch * RB;
                c.t = ch * chunk_tiles;
                c.t1 = min(NT, c.t + chunk_tiles);
            }
            c.j = 0;
        };
        auto cur_next = [&](Cur& c) {
            if (++c.j == 4) {
                c.j = 0;
                if (++c.t == c.t1) { c.item += gridDim.x; cur_set(c); }
            }
        };
        Cur pc; pc.item = blockIdx.x; cur_set(pc);
        Cur lc = pc;
        if (leader) {
            for (int k = 0; k < R - 1 && lc.item < nitems; ++k) {
                mbar_expect_tx(bCFull + 8 * k, Cfg::kStage);
                tma_load_2d(sC + k * Cfg::kStage, &tmC, bCFull + 8 * k, lc.t * 128 + lc.j * 32, lc.rb * 128);
                cur_next(lc);
            }
        }
        int s = 0, g = 0;
        while (pc.item < nitems) {
            const int st = s % R;
            mbar_wait(bCFull + 8 * st, (s / R) & 1);
            if (pc.j == 0) {
                mbar_wait(bTFull + 8 * (g & 1), (g >> 1) & 1);
                tc_fence_after();
            }
            uint32_t v[32];
            tmem_ld32(tmem + ((uint32_t)(quad * 32) << 16) + (g & 1) * 128 + pc.j * 32, v);
            tmem_ld_wait();
            float4* rowp = reinterpret_cast<float4*>(gC + st * Cfg::kStage + row * 128);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                float4 x = rowp[c ^ (row & 7)];
                x.x += __uint_as_float(v[4 * c + 0]);
                x.y += __uint_as_float(v[4 * c + 1]);
                x.z += __uint_as_float(v[4 * c + 2]);
                x.w += __uint_as_float(v[4 * c + 3]);
                rowp[c ^ (row & 7)] = x;
            }
            fence_proxy_async();
            if (pc.j == 3) {
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bTEmpty + 8 * (g & 1));
                ++g;
            }
            named_bar_sync(1, 128);
            if (leader) {
                tma_store_2d(&tmC, sC + st * Cfg::kStage, pc.t * 128 + pc.j * 32, pc.rb * 128);
                bulk_commit();
                bulk_wait_read<1>();               // the store issued one sub-tile ago has released its stage
                if (lc.item < nitems) {
                    const int ls = (s + R - 1) % R;
                    mbar_expect_tx(bCFull + 8 * ls, Cfg::kStage);
                    tma_load_2d(sC + ls * Cfg::kStage, &tmC, bCFull + 8 * ls, lc.t * 128 + lc.j * 32, lc.rb * 128);
                    cur_next(lc);
                }
            }
            cur_next(pc);
            ++s;
        }
        if (leader) bulk_wait_all();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 256);
}

// =====================================================================================================
// MODE 0 (NN): W(M x B) = C(M x N) Ut(N x B)      CTA tile = 128 rows of C, k runs over the columns
// MODE 1 (TN): W(B x N) = V(M x B)^T C(M x N)     CTA tile = 128 columns of C, k runs over the rows
// =====================================================================================================
template <int B> struct GemmCfg {
    static constexpr int kABytes = 128 * 32 * 4;         // 16 KB: raw (-> hi in place) and lo
    static constexpr int kXBytes = B * 32 * 4;           // one of {hi, lo}: B/32 slabs of 32 k-rows x 128 B
    static constexpr int kStage = 2 * kABytes + 2 * kXBytes;
    static constexpr int kStages = B == 64 ? 4 : 5;
    static constexpr int kBarBytes = 256;
    static constexpr int kSmem = 1024 + kStages * kStage + kBarBytes;
};

constexpr int kGemmThreads = 320;    // warp 0 TMA, warp 1 MMA, warps 2-5 split, warps 6-9 drain / epilogue
constexpr int kPeriod = 8;           // stages (of 32 k) accumulated in TMEM before the partial sum is drained

// Accumulation: tcgen05.mma adds into the fp32 TMEM accumulator with truncation, so a long chain of MMAs on one
// accumulator drifts by ~2^-24 per instruction (1.2e-4 at k = 16384).  Therefore (1) the two small products
// lo*hi and hi*lo go to their own accumulator, (2) both accumulators are double-buffered and restarted every
// kPeriod stages (32 hi*hi MMAs); four drain warps pull the finished pair out of TMEM (tcgen05.ld) and keep the
// running sum in registers with round-to-nearest fp32 adds while the MMAs of the next period run.
template <int MODE, int B>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc05_kernel(const __grid_constant__ CUtensorMap tmC, const __grid_constant__ CUtensorMap tmXh,
                 const __grid_constant__ CUtensorMap tmXl, float* __restrict__ out, int M, int N, int klen) {
    using Cfg = GemmCfg<B>;
    constexpr int S = Cfg::kStages;
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* gbase = smem_raw + (base - raw);
    const uint32_t sBar = base + S * Cfg::kStage;
    const uint32_t bFull = sBar, bSplit = sBar + 8 * S, bEmpty = sBar + 16 * S;
    const uint32_t bAccFull = sBar + 24 * S, bAccEmpty = bAccFull + 16;                  // [2], [2]
    const uint32_t sSlot = bAccEmpty + 16;
    volatile uint32_t* slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + (sSlot - base));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ktot = MODE == 0 ? N : M;
    const int kbeg = blockIdx.y * klen;
    const int kend = min(ktot, kbeg + klen);
    const int nk = max(0, (kend - kbeg + 31) / 32);
    const int t0 = blockIdx.x * 128;                     // first row (NN) / first column (TN) of the tile

    if (threadIdx.x == 0) {
        for (int i = 0; i < S; ++i) {
            mbar_init(bFull + 8 * i, 1);
            mbar_init(bSplit + 8 * i, 128);
            mbar_init(bEmpty + 8 * i, 1);
        }
        mbar_init(bAccFull, 1); mbar_init(bAccFull + 8, 1);
        mbar_init(bAccEmpty, 4); mbar_init(bAccEmpty + 8, 4);
        fence_barrier_init();
        prefetch_map(&tmC); prefetch_map(&tmXh); prefetch_map(&tmXl);
    }
    if (warp == 1) tmem_alloc(sSlot, 4 * B);             // 2 buffers x {hi*hi, small} x B columns
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *slot_ptr;

    if (warp == 0) {
        if (lane == 0) {
            for (int i = 0; i < nk; ++i) {
                const int st = i % S;
                if (i >= S) mbar_wait(bEmpty + 8 * st, ((i / S) - 1) & 1);
                const uint32_t sA = base + st * Cfg::kStage;
                const uint32_t sXh = sA + 2 * Cfg::kABytes, sXl = sXh + Cfg::kXBytes;
                const int k0 = kbeg + i * 32;
                mbar_expect_tx(bFull + 8 * st, Cfg::kABytes + 2 * Cfg::kXBytes);
                if (MODE == 0) {
                    tma_load_2d(sA, &tmC, bFull + 8 * st, k0, t0);                       // box 32 (k) x 128 rows
                } else {
#pragma unroll
                    for (int sl = 0; sl < 4; ++sl)                                       // box 32 columns x 32 k-rows
                        tma_load_2d(sA + sl * 4096, &tmC, bFull + 8 * st, t0 + sl * 32, k0);
                }
#pragma unroll
                for (int sl = 0; sl < B / 32; ++sl) {
                    tma_load_2d(sXh + sl * 4096, &tmXh, bFull + 8 * st, sl * 32, k0);
                    tma_load_2d(sXl + sl * 4096, &tmXl, bFull + 8 * st, sl * 32, k0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // kind::tf32 ignores the low 13 mantissa bits of an fp32 operand (probed: tools/tc05_selftest.py rounding), so
            // the raw tile IS the hi operand.  [Xh | Xl] are adjacent with one slab stride: A_raw x [Xh | Xl] is one MMA
            // of N = 2B (hi*hi -> columns [0,B), hi*lo -> [B,2B)); A_lo x Xh adds to [B,2B).
            constexpr uint32_t idesc2 = make_idesc(128, 2 * B, MODE, 1);
            constexpr uint32_t idesc1 = make_idesc(128, B, MODE, 1);
            for (int i = 0; i < nk; ++i) {
                const int st = i % S;
                const int p = i / kPeriod, buf = p & 1;
                const bool first = (i % kPeriod) == 0;
                if (first && p >= 2) mbar_wait(bAccEmpty + 8 * buf, ((p >> 1) - 1) & 1);
                mbar_wait(bSplit + 8 * st, (i / S) & 1);
                tc_fence_after();
                const uint32_t dHi = tmem + buf * (2 * B), dLo = dHi + B;
                const uint32_t sA = base + st * Cfg::kStage, sAl = sA + Cfg::kABytes;
                const uint32_t sXh = sA + 2 * Cfg::kABytes;
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                    uint64_t ah, al;
                    if (MODE == 0) {
                        ah = make_desc(sA + ks * 32, 16, 1024);
                        al = make_desc(sAl + ks * 32, 16, 1024);
                    } else {
                        ah = make_desc_mn(sA + ks * 1024, 4096);
                        al = make_desc_mn(sAl + ks * 1024, 4096);
                    }
                    const uint64_t xx = make_desc_mn(sXh + ks * 1024, 4096);
                    mma_tf32(dHi, ah, xx, idesc2, (first && ks == 0) ? 0u : 1u);
                    mma_tf32(dLo, al, xx, idesc1, 1u);
                }
                mma_commit(bEmpty + 8 * st);
                if ((i % kPeriod) == kPeriod - 1 || i == nk - 1) mma_commit(bAccFull + 8 * buf);
            }
        }
    } else if (warp < 6) {
        // ---- split: lo = rna_tf32(x - trunc_tf32(x)) into the second buffer (same layout); the raw tile serves as hi ----
        const int tid = threadIdx.x - 64;
        for (int i = 0; i < nk; ++i) {
            const int st = i % S;
            mbar_wait(bFull + 8 * st, (i / S) & 1);
            const uint4* a = reinterpret_cast<const uint4*>(gbase + st * Cfg::kStage);
            uint4* al = reinterpret_cast<uint4*>(gbase + st * Cfg::kStage + Cfg::kABytes);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const int idx = tid + q * 128;
                const uint4 x = a[idx];
                uint4 l;
                l.x = rna_tf32(__uint_as_float(x.x) - __uint_as_float(x.x & 0xffffe000u));
                l.y = rna_tf32(__uint_as_float(x.y) - __uint_as_float(x.y & 0xffffe000u));
                l.z = rna_tf32(__uint_as_float(x.z) - __uint_as_float(x.z & 0xffffe000u));
                l.w = rna_tf32(__uint_as_float(x.w) - __uint_as_float(x.w & 0xffffe000u));
                al[idx] = l;
            }
            fence_proxy_async();
            mbar_arrive(bSplit + 8 * st);
        }
    } else {
        // ---- drain + epilogue: running sum of the per-period partial accumulators in registers ----
        const int quad = warp & 3;
        const int row = quad * 32 + lane;
        float run[B];
#pragma unroll
        for (int j = 0; j < B; ++j) run[j] = 0.f;
        const int nper = (nk + kPeriod - 1) / kPeriod;
        for (int p = 0; p < nper; ++p) {
            const int buf = p & 1;
            mbar_wait(bAccFull + 8 * buf, (p >> 1) & 1);
            tc_fence_after();
            const uint32_t tb = tmem + ((uint32_t)(quad * 32) << 16) + buf * (2 * B);
#pragma unroll
            for (int cb = 0; cb < B / 32; ++cb) {
                uint32_t v[32], u[32];
                tmem_ld32(tb + cb * 32, v);
                tmem_ld32(tb + B + cb * 32, u);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) run[cb * 32 + j] += __uint_as_float(v[j]) + __uint_as_float(u[j]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bAccEmpty + 8 * buf);
        }
        float* o = out + (size_t)blockIdx.y * (size_t)(MODE == 0 ? (size_t)M * B : (size_t)B * N);
        if (MODE == 0) {
            if (t0 + row < M) {
                float4* dst = reinterpret_cast<float4*>(o + (size_t)(t0 + row) * B);
#pragma unroll
                for (int c = 0; c < B / 4; ++c) dst[c] = make_float4(run[4 * c], run[4 * c + 1], run[4 * c + 2], run[4 * c + 3]);
            }
        } else {
            if (t0 + row < N) {
#pragma unroll
                for (int j = 0; j < B; ++j) o[(size_t)j * N + t0 + row] = run[j];
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, 4 * B);
}

// ---- measured tcgen05 TF32 issue rate (register-free loop over resident smem; no loads) ----------------
__global__ void __launch_bounds__(64, 1) probe_tf32_kernel(int iters) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* gbase = smem_raw + (base - raw);
    const uint32_t sBar = base + 64 * 1024;
    volatile uint32_t* slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + 64 * 1024 + 8);
    for (int i = threadIdx.x; i < 16 * 1024; i += blockDim.x) reinterpret_cast<float*>(gbase)[i] = 0.f;
    if (threadIdx.x == 0) { mbar_init(sBar, 1); fence_barrier_init(); }
    fence_proxy_async();
    if (threadIdx.x < 32) tmem_alloc(sBar + 8, 256);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *slot_ptr;
    if (threadIdx.x == 0) {
        constexpr uint32_t idesc = make_idesc(128, 256, 0, 0);
        const uint64_t ad = make_desc(base, 16, 1024);             // A 128 x 32 (K-major), B 256 x 32 (K-major)
        const uint64_t bd = make_desc(base + 16384, 16, 1024);
        for (int i = 0; i < iters; ++i) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) mma_tf32(tmem, ad + 2 * ks, bd + 2 * ks, idesc, 1);
        }
        mma_commit(sBar);
        mbar_wait(sBar, 0);
    }
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(tmem, 256);
}

// ---- self-test: one TMA-loaded tile pair -> 4 MMAs -> TMEM -> global, plus a dump of the staged shared memory --------
// a_mn = 0: A is 128 x 32 row-major (K-major operand, one 32x128 box);  a_mn = 1: A^T given as 32 x 128 row-major
// (MN-major operand, four 32x32 boxes).  b_mn likewise with N = 64: b_mn = 0: B^T 64 x 32; b_mn = 1: B 32 x 64.
__global__ void __launch_bounds__(128, 1)
selftest_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int a_mn, int b_mn,
                float* __restrict__ out, float* __restrict__ dump) {
    extern __shared__ unsigned char smem_raw[];
    const uint32_t raw = smem_u32(smem_raw);
    const uint32_t base = (raw + 1023u) & ~1023u;
    unsigned char* gbase = smem_raw + (base - raw);
    const uint32_t sA = base, sB = base + 16384, sBar = base + 32768;
    volatile uint32_t* slot_ptr = reinterpret_cast<volatile uint32_t*>(gbase + 32768 + 16);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) { mbar_init(sBar, 1); mbar_init(sBar + 8, 1); fence_barrier_init(); }
    if (warp == 0) tmem_alloc(sBar + 16, 64);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *slot_ptr;
    if (threadIdx.x == 0) {
        mbar_expect_tx(sBar, 16384 + 8192);
        if (a_mn == 0) tma_load_2d(sA, &tmA, sBar, 0, 0);
        else for (int sl = 0; sl < 4; ++sl) tma_load_2d(sA + sl * 4096, &tmA, sBar, sl * 32, 0);
        if (b_mn == 0) tma_load_2d(sB, &tmB, sBar, 0, 0);
        else for (int sl = 0; sl < 2; ++sl) tma_load_2d(sB + sl * 4096, &tmB, sBar, sl * 32, 0);
    }
    mbar_wait(sBar, 0);
    for (int i = threadIdx.x; i < 6144; i += blockDim.x) dump[i] = reinterpret_cast<float*>(gbase)[i];
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t idesc = make_idesc(128, 64, a_mn, b_mn);
        tc_fence_after();
        for (int ks = 0; ks < 4; ++ks) {
            const uint64_t ad = a_mn == 0 ? make_desc(sA + ks * 32, 16, 1024) : make_desc_mn(sA + ks * 1024, 4096);
            const uint64_t bd = b_mn == 0 ? make_desc(sB + ks * 32, 16, 1024) : make_desc_mn(sB + ks * 1024, 4096);
            mma_tf32(tmem, ad, bd, idesc, ks > 0 ? 1u : 0u);
        }
        mma_commit(sBar + 8);
    }
    mbar_wait(sBar + 8, 0);
    tc_fence_after();
    const int row = warp * 32 + lane;
    for (int cb = 0; cb < 2; ++cb) {
        uint32_t v[32];
        tmem_ld32(tmem + ((uint32_t)(warp * 32) << 16) + cb * 32, v);
        tmem_ld_wait();
        for (int j = 0; j < 32; ++j) out[row * 64 + cb * 32 + j] = __uint_as_float(v[j]);
    }
    if (threadIdx.x == 0) out[128 * 64] = __uint_as_float(tmem);
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 64);
}

// ---- host side -------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            cudaGetLastError();
    }
    return fn;
}

// 2-D fp32 row-major view (rows x cols, leading dimension ld elements), boxes of box_rows x 32 columns (128 B),
// 128-byte swizzle (16-byte atoms; 32-byte atoms for tiles that feed an MN-major UMMA operand), out-of-bounds
// elements read as zero / are not written.
static int make_map(Ctx* c, CUtensorMap* m, const float* ptr, size_t rows, size_t cols, size_t ld, unsigned box_rows,
                    bool mn_major = false) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) { c->last_error = "cuTensorMapEncodeTiled unavailable"; return SVDB200_E_STATE; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {32u, box_rows};
    cuuint32_t estr[2] = {1u, 1u};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        c->last_error = "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")";
        return SVDB200_E_STATE;
    }
    return 0;
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static int ensure_scratch(Ctx* c) {
    if (c->tcsplit) return 0;
    c->tcsplit_elems = 4 * (c->max_n + 64) * c->band + 1024;
    SVDB_CHECK(c, cudaMalloc(&c->tcsplit, sizeof(float) * c->tcsplit_elems));
    return 0;
}

static int launch_split(Ctx* c, const float* src, size_t ld_src, int rows, int cols, float* hi, float* lo, size_t ld_dst) {
    const size_t total = (size_t)rows * cols;
    int blocks = (int)((total + 255) / 256);
    if (blocks > 4 * c->num_sms) blocks = 4 * c->num_sms;
    if (blocks < 1) blocks = 1;
    split_tf32_kernel<<<blocks, 256, 0, c->stream>>>(src, ld_src, rows, cols, hi, lo, ld_dst);
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    return 0;
}

static bool wanted(Ctx* c, int M, int N, int B) {
    if (c->cfg.use_tc05 == 0) return false;
    if (B != 32 && B != 64) return false;
    if (c->cfg.use_tc05 >= 2) return true;
    return (long long)M * N >= (long long)c->cfg.tc05_min_elems;
}

}  // namespace tc05

// ---- entry points (return 1: not applicable, the caller falls back to the mma.sync kernels) ------------------
template <>
int rank_update_tc05<double>(Ctx*, double*, size_t, int, int, int, const double*, const double*, size_t) { return 1; }
template <>
int gemm_tn_tc05<double>(Ctx*, const double*, const double*, size_t, int, int, int, double*) { return 1; }
template <>
int gemm_nn_tc05<double>(Ctx*, const double*, size_t, int, int, int, const double*, double*) { return 1; }

template <>
int rank_update_tc05<float>(Ctx* c, float* cm, size_t ldc, int M, int N, int K, const float* p, const float* q, size_t ldq) {
    using namespace tc05;
    if (!wanted(c, M, N, K) || !aligned16(cm) || (ldc & 3)) return 1;
    SVDB_TRY(ensure_scratch(c));
    const size_t ldn = ((size_t)N + 3) & ~(size_t)3;
    float* ph = reinterpret_cast<float*>(c->tcsplit);
    float* pl = ph + (size_t)M * K;
    float* qh = pl + (size_t)M * K;
    float* ql = qh + (size_t)K * ldn;
    if ((size_t)(ql + (size_t)K * ldn - ph) > c->tcsplit_elems) return 1;
    SVDB_TRY(launch_split(c, p, (size_t)K, M, K, ph, pl, (size_t)K));
    SVDB_TRY(launch_split(c, q, ldq, K, N, qh, ql, ldn));
    CUtensorMap tC, tPh, tPl, tQh, tQl;
    SVDB_TRY(make_map(c, &tC, cm, M, N, ldc, 128));
    SVDB_TRY(make_map(c, &tPh, ph, M, K, K, 128));
    SVDB_TRY(make_map(c, &tPl, pl, M, K, K, 128));
    SVDB_TRY(make_map(c, &tQh, qh, K, N, ldn, K, true));
    SVDB_TRY(make_map(c, &tQl, ql, K, N, ldn, K, true));
    const int RB = (M + 127) / 128, NT = (N + 127) / 128;
    int chunk = 8;
    // persistent CTAs, one per SM -- minus the SMs left to a look-ahead panel on the high-priority stream (the panel's
    // kernels need whole SMs: this kernel's CTAs never retire early)
    const int sms = c->reserve_now > 0 && c->num_sms > 2 * c->reserve_now ? c->num_sms - c->reserve_now : c->num_sms;
    while (chunk > 1 && (long long)RB * ((NT + chunk - 1) / chunk) < 2LL * sms) chunk >>= 1;
    const int NCH = (NT + chunk - 1) / chunk;
    int grid = RB * NCH;
    if (grid > sms) grid = sms;
    if (K == 64) {
        auto kern = rank_update_tc05_kernel<64>;
        SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, RuCfg<64>::kSmem));
        kern<<<grid, kThreads, RuCfg<64>::kSmem, c->stream>>>(tC, tPh, tPl, tQh, tQl, RB, NT, chunk, NCH);
    } else {
        auto kern = rank_update_tc05_kernel<32>;
        SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, RuCfg<32>::kSmem));
        kern<<<grid, kThreads, RuCfg<32>::kSmem, c->stream>>>(tC, tPh, tPl, tQh, tQl, RB, NT, chunk, NCH);
    }
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    return 0;
}

namespace tc05 {

template <typename T>
__global__ void reduce_parts_kernel(const T* __restrict__ part, T* __restrict__ w, size_t count, int splits) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    T acc = part[i];
    for (int s = 1; s < splits; ++s) acc += part[(size_t)s * count + i];
    w[i] = acc;
}

// mode 0: NN (x = Ut, N x B), mode 1: TN (x = V, M x B)
static int gemm_common(Ctx* c, int mode, const float* cm, size_t ldc, int M, int N, int B, const float* x, float* w) {
    if (!wanted(c, M, N, B) || !aligned16(cm) || (ldc & 3)) return 1;
    SVDB_TRY(ensure_scratch(c));
    const int xrows = mode == 0 ? N : M;
    float* xh = reinterpret_cast<float*>(c->tcsplit);
    float* xl = xh + (size_t)xrows * B;
    if ((size_t)2 * xrows * B > c->tcsplit_elems) return 1;
    SVDB_TRY(launch_split(c, x, (size_t)B, xrows, B, xh, xl, (size_t)B));
    const int ktot = mode == 0 ? N : M;
    const int tiles = ((mode == 0 ? M : N) + 127) / 128;
    const size_t out_elems = (size_t)(mode == 0 ? M : N) * B;
    // split-K so that tiles x splits fills whole waves of one CTA per SM: minimise ceil(tiles*s / SMs) / s
    const int kiters = (ktot + 31) / 32;
    int smax = kiters / 16;                               // >= 512 k per split
    if (smax > 16) smax = 16;
    if ((size_t)smax * out_elems > c->wpart_elems) smax = (int)(c->wpart_elems / out_elems);
    if (smax < 1) smax = 1;
    int splits = 1;
    double best = 1e30;
    for (int sp = 1; sp <= smax; ++sp) {
        const double cost = (double)((tiles * sp + c->num_sms - 1) / c->num_sms) / sp + 0.004 * sp;
        if (cost < best - 1e-12) { best = cost; splits = sp; }
    }
    int klen = (((ktot + splits - 1) / splits + 31) / 32) * 32;
    splits = (ktot + klen - 1) / klen;
    float* out = splits == 1 ? w : reinterpret_cast<float*>(c->wpart);
    CUtensorMap tC, tXh, tXl;
    SVDB_TRY(make_map(c, &tC, cm, M, N, ldc, mode == 0 ? 128 : 32, mode == 1));
    SVDB_TRY(make_map(c, &tXh, xh, xrows, B, B, 32, true));
    SVDB_TRY(make_map(c, &tXl, xl, xrows, B, B, 32, true));
    dim3 grid(tiles, splits);
#define SVDB_TC05_GEMM(MODEv, Bv)                                                                                  \
    {                                                                                                              \
        auto kern = gemm_tc05_kernel<MODEv, Bv>;                                                                   \
        SVDB_CHECK(c, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<Bv>::kSmem)); \
        kern<<<grid, kGemmThreads, GemmCfg<Bv>::kSmem, c->stream>>>(tC, tXh, tXl, out, M, N, klen);                    \
    }
    if (mode == 0) { if (B == 64) SVDB_TC05_GEMM(0, 64) else SVDB_TC05_GEMM(0, 32) }
    else           { if (B == 64) SVDB_TC05_GEMM(1, 64) else SVDB_TC05_GEMM(1, 32) }
#undef SVDB_TC05_GEMM
    SVDB_CHECK(c, cudaGetLastError());
    c->launches++;
    if (splits > 1) {
        reduce_parts_kernel<float><<<(unsigned)((out_elems + 255) / 256), 256, 0, c->stream>>>(out, w, out_elems, splits);
        SVDB_CHECK(c, cudaGetLastError());
        c->launches++;
    }
    return 0;
}

}  // namespace tc05

template <>
int gemm_tn_tc05<float>(Ctx* c, const float* v, const float* cm, size_t ldc, int M, int N, int B, float* w) {
    return tc05::gemm_common(c, 1, cm, ldc, M, N, B, v, w);
}
template <>
int gemm_nn_tc05<float>(Ctx* c, const float* cm, size_t ldc, int M, int N, int B, const float* ut, float* w) {
    return tc05::gemm_common(c, 0, cm, ldc, M, N, B, ut, w);
}

// self-test entry: a (device, 4096 floats), b (device, 2048 floats), out (device, 128*64+1), dump (device, 6144)
int tc05_selftest(Ctx* c, int a_mn, int b_mn, const float* a, const float* b, float* out, float* dump) {
    using namespace tc05;
    CUtensorMap tA, tB;
    if (a_mn == 0) SVDB_TRY(make_map(c, &tA, a, 128, 32, 32, 128)); else SVDB_TRY(make_map(c, &tA, a, 32, 128, 128, 32, true));
    if (b_mn == 0) SVDB_TRY(make_map(c, &tB, b, 64, 32, 32, 64)); else SVDB_TRY(make_map(c, &tB, b, 32, 64, 64, 32, true));
    const int smem = 1024 + 32768 + 64;
    SVDB_CHECK(c, cudaFuncSetAttribute(selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    selftest_kernel<<<1, 128, smem, c->stream>>>(tA, tB, a_mn, b_mn, out, dump);
    SVDB_CHECK(c, cudaGetLastError());
    SVDB_CHECK(c, cudaStreamSynchronize(c->stream));
    return 0;
}

// tcgen05 kind::tf32 issue rate (M = 128, N = 256, K = 8 per instruction), all SMs
int probe_tc05_tf32(Ctx* c, double* tflops) {
    using namespace tc05;
    const int iters = 4096;
    const int smem = 1024 + 64 * 1024 + 64;
    SVDB_CHECK(c, cudaFuncSetAttribute(probe_tf32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    cudaEvent_t e0, e1;
    SVDB_CHECK(c, cudaEventCreate(&e0));
    SVDB_CHECK(c, cudaEventCreate(&e1));
    probe_tf32_kernel<<<c->num_sms, 64, smem, c->stream>>>(64);
    SVDB_CHECK(c, cudaEventRecord(e0, c->stream));
    probe_tf32_kernel<<<c->num_sms, 64, smem, c->stream>>>(iters);
    SVDB_CHECK(c, cudaEventRecord(e1, c->stream));
    SVDB_CHECK(c, cudaEventSynchronize(e1));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    const double flops = 2.0 * 128 * 256 * 8 * 4.0 * iters * c->num_sms;
    *tflops = flops / (ms * 1e-3) / 1e12;
    return 0;
}

}  // namespace svdb200

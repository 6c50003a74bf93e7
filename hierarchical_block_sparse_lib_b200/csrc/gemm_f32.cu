// gemm_f32.cu -- fp32 leaf GEMM on the 5th-generation tensor cores: C_tile = sum_k op(A_ik) * op(B_kj)  (H:7273 for
// Treal = float, G:92-98 sgemm), persistent and C-stationary like the FP64 kernel, accumulators in TMEM.
//
// tcgen05 has no fp32 kind and single-pass TF32 (10-bit mantissa) misses the 1e-5 parity bar, so every operand x is
// split in shared memory into  hi = x with the 13 low mantissa bits cleared  (exactly a TF32 number; the tensor core
// drops those bits itself -- measured: feeding the raw x gives bit-identical results -- so "hi" is the raw operand left
// in place) and lo = x - hi  (exact in fp32), and each K-step issues three  tcgen05.mma.kind::tf32  with fp32 accumulation:
//   D += A_lo*B_hi ; D += A_hi*B_lo ; D += A_hi*B_hi         (the dropped lo*lo term is ~2^-22 relative)
// The tensor core truncates when it adds into its fp32 accumulator, which biases long chains (measured 1e-5 after 384
// chained MMAs), so the TMEM accumulator only ever holds ONE leaf product (small terms issued first, then the hi*hi
// terms); the epilogue warps add each finished product into the C tile held in registers with ordinary round-to-nearest
// fp32 adds, in k order -- the summation order of the reference's sgemm calls (H:7273, beta = 1).
//
// Warp roles (one CTA per SM, 16 warps):
//   warp 0      TMA producer + dynamic C-tile scheduler: per K-chunk one 128B-swizzled box set for op(A) and op(B)
//   warp 1      TMEM allocator; one elected lane issues the MMAs and tcgen05.commit's
//   warps 4-7   hi/lo split of each landed stage, in place (elementwise, so the swizzled layout is untouched)
//   warps 8-15  epilogue: tcgen05.ld of each finished product, C tile accumulated in registers, coalesced column-major
//               stores when the k-list of the C tile ends
// Pipelines: smem ring  raw(TMA) -> split(converters) -> consumed(tcgen05.commit), and a 2-deep TMEM accumulator ring
// (MMAs of product p+1 overlap the drain of product p).
//
// Operand layouts.  Leaves are column-major (H:715).  An operand whose MN index runs along leaf rows (A as is, B
// transposed) is "MN-major": the K-chunk is a set of leaf columns, staged as slabs [k][32 mn] (128 B per k row).
// An operand whose K index runs along leaf rows (A transposed, B as is) is "K-major": staged as slabs [mn][32 k].
// K-major uses the canonical SWIZZLE_128B layout; MN-major 32-bit operands must use the 128B-swizzle-with-32B-atom
// layout (4 k rows per atom; TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, descriptor layout type 1).  All four (tA,tB)
// combinations therefore only differ in the tensor map and a few descriptor fields -- no transposition pass.
// This kernel serves leaves of 128 and 256 (128-row compute tiles, M = 128: C row i is TMEM lane i); leaves of 32 and 64
// have kernels of their own below.
#include "gemm_common.cuh"

namespace hbsm_b200 {

namespace {

// ---- tcgen05 / TMEM PTX wrappers ----
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %6, %7, %8}, p;\n\t}"
        ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tma_box_g2s(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}

// UMMA shared-memory descriptor (sm_100): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) | version=1 [46,48) |
// layout type [61,64) (2 = SWIZZLE_128B, 1 = SWIZZLE_128B with 32-byte atoms)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
           (1ull << 46) | ((uint64_t)layout_type << 61);
}

template <int BS>
struct F32Cfg {
    static_assert(BS == 128, "128-row compute tiles");
    static constexpr int KC = 32;                           // K-chunk per pipeline stage
    static constexpr int NCHUNK = BS / KC;
    static constexpr int OPER_BYTES = BS * KC * 4;          // one operand chunk (raw == hi), same again for lo
    static constexpr int STAGE_BYTES = 4 * OPER_BYTES;      // A_hi | A_lo | B_hi | B_lo
    static constexpr int NST = (196 * 1024 / STAGE_BYTES) > 8 ? 8 : (196 * 1024 / STAGE_BYTES);
    static constexpr int HEADER_BYTES = 1024;
    static constexpr int SMEM_BYTES = 1024 + HEADER_BYTES + NST * STAGE_BYTES;
    // Independent TMEM accumulators per leaf product.  Back-to-back MMAs into ONE accumulator serialise on its
    // read-modify-write latency (measured ~100 clk per N=64 MMA instead of the 32 clk dispatch floor), so the hi*hi term
    // gets an accumulator of its own and lo*hi, hi*lo share the other (TMEM has 512 columns); the epilogue adds them.
    // x2 for the double-buffered hand-off to the epilogue.
    static constexpr int NACC = 2;
    static constexpr int ACC_COLS = NACC * BS;
    static constexpr int TMEM_COLS = 2 * ACC_COLS;
    static_assert(TMEM_COLS == 512, "TMEM has 512 columns");
    static constexpr int THREADS = 512;
    static constexpr int CVT_WARPS = 4;
    static constexpr int EPI_H = 2;                                 // column halves: two warps share a TMEM lane quadrant
    static constexpr int EPI_CW = BS / EPI_H;                       // columns per epilogue warp
    static constexpr int EPI_WARPS = 4 * EPI_H;
    static constexpr int KSTEPS = KC / 8;
    static_assert(NST >= 2, "pipeline needs two stages");
};

struct F32Header {
    uint64_t full_raw[8], full_cvt[8], empty[8], tmem_full[8], tmem_empty[8];   // the 3-MMA kernel uses 2 accumulator sets
    GemmMeta meta[8];
    int acc_tile[8];
    int acc_flags[8];     // 1 = first product of its C tile, 2 = last product, 4 = no more work
    uint32_t tmem_base;
    // stacked kernel: per-STAGE-SEQUENCE meta written once by the producer and read by every later role (split warps, MMA
    // issuer, epilogue), so that the issuing lane never stores to shared memory: a store would need a fence before the
    // tcgen05.commit that publishes it, and a fence in that lane waits for its MMAs in flight -- the tensor pipe then
    // idles for the whole per-stage hand-off (measured: 135 clk per M=N=64 MMA instead of 47).  The producer leads the
    // epilogue by at most NST + NSETS * CH <= 11 stages, the ring has 16 entries.
    GemmMeta ring[16];
};

// LS = leaf size (H:167 blocksize), BS = the square compute tile one CTA accumulates (BS == LS for 128-leaves; a
// 256-leaf is processed as 2 x 2 C sub-tiles whose k-lists are the leaf's k-list with both 128-wide halves of each
// operand: the tensor-map coordinates address the sub-blocks in place, ld = LS).
template <int LS, int BS, bool TA, bool TB>
__global__ void __launch_bounds__(F32Cfg<BS>::THREADS, 1)
k_gemm_f32_tc(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
              const uint2* __restrict__ ab, const uint64_t* __restrict__ begin, uint32_t n_ctiles,
              const uint32_t* __restrict__ tile_list, unsigned* __restrict__ next_tile, float* __restrict__ Ct) {
    using Cfg = F32Cfg<BS>;
    constexpr int S = LS / BS;            // sub-tiles per leaf side
    static_assert(LS % BS == 0 && (S == 1 || S == 2), "leaf / compute-tile shapes");
    constexpr int NST = Cfg::NST, KC = Cfg::KC;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    F32Header* hd = reinterpret_cast<F32Header*>(smem);
    unsigned char* stages = smem + Cfg::HEADER_BYTES;
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(smem_u32(&hd->full_raw[s]), 1);
            mbar_init(smem_u32(&hd->full_cvt[s]), Cfg::CVT_WARPS);
            mbar_init(smem_u32(&hd->empty[s]), 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(smem_u32(&hd->tmem_full[a]), 1);
            mbar_init(smem_u32(&hd->tmem_empty[a]), Cfg::EPI_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&hd->tmem_base), Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = hd->tmem_base;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
            uint32_t it = 0;
            for (;;) {
                const unsigned unit = atomicAdd(next_tile, 1u);       // work unit = (C tile, sub-tile)
                if (unit >= n_ctiles * (unsigned)(S * S)) break;
                const unsigned sub = unit % (S * S);
                const unsigned tile = tile_list ? tile_list[unit / (S * S)] : unit / (S * S);
                const int cunit = (int)(tile * (S * S) + sub);
                const int si = (int)(sub % S) * BS, sj = (int)(sub / S) * BS;   // row / column offset of the C sub-tile
                const uint64_t p0 = begin[tile], p1 = begin[tile + 1];
                uint2 t = ab[p0];
                for (uint64_t p = p0; p < p1; ++p) {
                    const uint2 tn = (p + 1 < p1) ? ab[p + 1] : t;
#pragma unroll 1
                    for (int kk = 0; kk < S; ++kk) {
#pragma unroll 1
                        for (int ch = 0; ch < Cfg::NCHUNK; ++ch, ++it) {
                            const uint32_t s = it % NST, ph = (it / NST) & 1u;
                            mbar_wait(smem_u32(&hd->empty[s]), ph ^ 1u);
                            const uint32_t fb = smem_u32(&hd->full_raw[s]);
                            int fl = 0;
                            if (p == p0 && kk == 0) fl |= 1;                  // first accumulator of its C (sub-)tile
                            if (p + 1 == p1 && kk == S - 1) fl |= 2;          // ... the last
                            if (ch == 0) fl |= 8;                             // first K-chunk of this accumulator
                            if (ch == Cfg::NCHUNK - 1) fl |= 16;              // last K-chunk
                            hd->meta[s].ctile = cunit;
                            hd->meta[s].flags = fl;
                            mbar_arrive_expect_tx(fb, 2 * Cfg::OPER_BYTES);
                            const uint32_t sa = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES);
                            const uint32_t sb = sa + 2 * Cfg::OPER_BYTES;
                            const int k0 = kk * BS + ch * KC;
                            // tensor map: dim0 = leaf row (contiguous), dim1 = leaf column + LS * tile
                            if (TA) {   // K-major: slabs [BS mn][32 k], box {32 rows (k), BS columns (mn)}
#pragma unroll
                                for (int j = 0; j < KC / 32; ++j) tma_box_g2s(sa + j * (BS * 128), &mapA, k0 + 32 * j, (int)t.x * LS + si, fb);
                            } else {    // MN-major: slabs [KC k][32 mn], box {32 rows (mn), KC columns (k)}
#pragma unroll
                                for (int j = 0; j < BS / 32; ++j) tma_box_g2s(sa + j * (KC * 128), &mapA, si + 32 * j, (int)t.x * LS + k0, fb);
                            }
                            if (TB) {   // op(B) = B^T: n runs along leaf rows -> MN-major
#pragma unroll
                                for (int j = 0; j < BS / 32; ++j) tma_box_g2s(sb + j * (KC * 128), &mapB, sj + 32 * j, (int)t.y * LS + k0, fb);
                            } else {    // op(B) = B: k runs along leaf rows -> K-major
#pragma unroll
                                for (int j = 0; j < KC / 32; ++j) tma_box_g2s(sb + j * (BS * 128), &mapB, k0 + 32 * j, (int)t.y * LS + sj, fb);
                            }
                        }
                    }
                    t = tn;
                }
            }
            const uint32_t s = it % NST, ph = (it / NST) & 1u;
            mbar_wait(smem_u32(&hd->empty[s]), ph ^ 1u);
            hd->meta[s].ctile = -1;
            hd->meta[s].flags = 4;
            mbar_arrive(smem_u32(&hd->full_raw[s]));
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            // instruction descriptor: D fp32 [4,6)=1, A/B tf32 [7,10)=[10,13)=2, a_major bit 15, b_major bit 16 (1 = MN-major),
            // N>>3 at [17,23), M>>4 at [24,29)
            constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((TA ? 0u : 1u) << 15) | ((TB ? 1u : 0u) << 16) |
                                       ((uint32_t)(BS >> 3) << 17) | ((uint32_t)(BS >> 4) << 24);
            // K-major: SWIZZLE_128B (type 2), 8-row groups 1024 B apart.  MN-major fp32: 32-byte-atom swizzle (type 1), 4 k rows
            // per atom (SBO = 512 B), 32-element MN chunks one slab (LBO) apart.
            constexpr uint32_t A_LBO = TA ? 16 : KC * 128, B_LBO = TB ? KC * 128 : 16;
            constexpr uint32_t A_SBO = TA ? 1024 : 512, B_SBO = TB ? 512 : 1024;
            constexpr uint32_t A_LT = TA ? 2 : 1, B_LT = TB ? 1 : 2;
            uint32_t it = 0, pc = 0;
            bool open = false;
            for (;; ++it) {
                const uint32_t s = it % NST, ph = (it / NST) & 1u;
                mbar_wait(smem_u32(&hd->full_cvt[s]), ph);
                const GemmMeta m = hd->meta[s];
                const uint32_t as = pc & 1u;
                if (m.flags & 4) {
                    mbar_wait(smem_u32(&hd->tmem_empty[as]), ((pc >> 1) & 1u) ^ 1u);
                    hd->acc_flags[as] = 4;
                    __threadfence_block();
                    mbar_arrive(smem_u32(&hd->tmem_full[as]));
                    break;
                }
                if (m.flags & 8) {
                    mbar_wait(smem_u32(&hd->tmem_empty[as]), ((pc >> 1) & 1u) ^ 1u);   // epilogue drained this accumulator set
                    open = false;
                }
                tc_fence_after();
                const uint32_t d_small = tmem_base + as * Cfg::ACC_COLS;                    // lo*hi + hi*lo
                const uint32_t d_big = d_small + BS;                                        // hi*hi
                const uint32_t sa = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES);
                const uint32_t a_hi = sa, a_lo = sa + Cfg::OPER_BYTES, b_hi = sa + 2 * Cfg::OPER_BYTES, b_lo = sa + 3 * Cfg::OPER_BYTES;
                // MN-major: 8 k rows = 1024 B per step; K-major: 32 B inside the 128-B row, next slab every 4 steps
#pragma unroll
                for (int ks = 0; ks < Cfg::KSTEPS; ++ks) {
                    const uint32_t ao = TA ? (uint32_t)((ks >> 2) * (BS * 128) + (ks & 3) * 32) : (uint32_t)(ks * 1024);
                    const uint32_t bo = TB ? (uint32_t)(ks * 1024) : (uint32_t)((ks >> 2) * (BS * 128) + (ks & 3) * 32);
                    const uint64_t dah = umma_desc(a_hi + ao, A_LBO, A_SBO, A_LT), dal = umma_desc(a_lo + ao, A_LBO, A_SBO, A_LT);
                    const uint64_t dbh = umma_desc(b_hi + bo, B_LBO, B_SBO, B_LT), dbl = umma_desc(b_lo + bo, B_LBO, B_SBO, B_LT);
                    mma_tf32(d_small, dal, dbh, IDESC, open ? 1u : 0u);
                    mma_tf32(d_small, dah, dbl, IDESC, 1u);
                    mma_tf32(d_big, dah, dbh, IDESC, open ? 1u : 0u);
                    open = true;
                }
                tc_commit(smem_u32(&hd->empty[s]));             // stage free when these MMAs have read it
                if (m.flags & 16) {                             // product complete: hand the accumulator to the epilogue
                    hd->acc_tile[as] = m.ctile;
                    hd->acc_flags[as] = m.flags & 3;
                    __threadfence_block();
                    tc_commit(smem_u32(&hd->tmem_full[as]));
                    ++pc;
                }
            }
        }
    } else if (warp >= 4 && warp < 4 + Cfg::CVT_WARPS) {
        // ===== hi/lo split: raw fp32 (A at +0, B at +2*OPER) stays in place as hi, lo at +OPER =====
        const unsigned tid = threadIdx.x - 128;
        for (uint32_t it = 0;; ++it) {
            const uint32_t s = it % NST, ph = (it / NST) & 1u;
            mbar_wait(smem_u32(&hd->full_raw[s]), ph);
            const int flags = hd->meta[s].flags;
            if (!(flags & 4)) {
                unsigned char* st = stages + (size_t)s * Cfg::STAGE_BYTES;
#pragma unroll
                for (int op = 0; op < 2; ++op) {
                    const float4* hi = reinterpret_cast<const float4*>(st + op * 2 * Cfg::OPER_BYTES);
                    float4* lo = reinterpret_cast<float4*>(st + op * 2 * Cfg::OPER_BYTES + Cfg::OPER_BYTES);
#pragma unroll 4
                    for (int i = (int)tid; i < Cfg::OPER_BYTES / 16; i += Cfg::CVT_WARPS * 32) {
                        const float4 x = hi[i];
                        float4 l;
                        l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                        l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                        l.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                        l.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                        lo[i] = l;
                    }
                }
                fence_proxy_async();   // generic-proxy writes -> visible to the tensor core's async-proxy reads
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&hd->full_cvt[s]));
            if (flags & 4) break;
        }
    } else if (warp >= 8 && (warp - 8) < Cfg::EPI_WARPS) {
        // ===== epilogue: warp (q,h) owns TMEM lanes [32q, 32q+32) = C rows, columns [h*CW, (h+1)*CW) =====
        const unsigned q = (warp - 8) & 3, h = (warp - 8) >> 2;
        constexpr int CW = Cfg::EPI_CW;
        const int row = (int)(q * 32 + lane);
        float acc[CW];
        for (uint32_t pc = 0;; ++pc) {
            const uint32_t as = pc & 1u;
            mbar_wait(smem_u32(&hd->tmem_full[as]), (pc >> 1) & 1u);
            const int flags = hd->acc_flags[as];
            if (flags & 4) break;
            const int ctile = hd->acc_tile[as];
            tc_fence_after();
#pragma unroll
            for (int c0 = 0; c0 < CW; c0 += 32) {
#pragma unroll
                for (int a = 0; a < Cfg::NACC; ++a) {      // small terms first, the hi*hi accumulator last
                    uint32_t r[32];
                    tmem_ld32(tmem_base + ((q * 32u) << 16) + as * Cfg::ACC_COLS + a * BS + h * CW + c0, r);
                    tmem_ld_wait();
                    if (a == 0 && (flags & 1)) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[c0 + j] = __uint_as_float(r[j]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[c0 + j] = __fadd_rn(acc[c0 + j], __uint_as_float(r[j]));
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&hd->tmem_empty[as]));
            if (flags & 2) {
                const unsigned tile = (unsigned)ctile / (S * S), sub = (unsigned)ctile % (S * S);
                float* C = Ct + (size_t)tile * LS * LS + (size_t)((sub / S) * BS + h * CW) * LS + (sub % S) * BS + row;
#pragma unroll
                for (int j = 0; j < CW; ++j) C[(size_t)j * LS] = acc[j];   // 32 lanes = 32 consecutive rows: 128 B per store
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------------
// Leaves of 32 / 64: ONE MMA per K-step computes all four hi/lo cross terms.
//
// Measured on B200: a kind::tf32 MMA is paced by the shared-memory fetch of its operands (~64 B/clk/SM), not by the
// 32-clk dispatch floor.  Stacking  [A_hi ; A_lo]  along M and  [B_hi | B_lo]  along N turns the three MMAs of a K-step
// (18 KiB of operand reads at BS = 64) into one M = N = 2*BS MMA (8 KiB) whose accumulator quadrants are
//     D[0:BS, 0:BS] = hi*hi   D[0:BS, BS:2BS] = hi*lo   D[BS:2BS, 0:BS] = lo*hi   D[BS:2BS, BS:2BS] = lo*lo
// (the lo*lo term comes for free).  The stacked operands are plain descriptors over the hi/lo buffers: MN-major
// operands keep "hi slabs then lo slabs" (consecutive 32-element chunks, LBO apart), K-major operands interleave
// "hi slab j, lo slab j" so that the 8-row groups of hi and lo are consecutive (SBO apart).
// Epilogue: warps of TMEM lane quadrants 0,1 own the hi rows, quadrants 2,3 the lo rows of the SAME C rows; each keeps
// its partial C tile in registers (round-to-nearest adds, one leaf product at a time) and the two halves are combined
// through shared memory once per C tile.
// ---------------------------------------------------------------------------------------------------
template <int BS>
struct Q4Cfg {
    static constexpr int KC = BS;                            // whole leaf products per pipeline stage
    static constexpr int OPER_BYTES = BS * KC * 4;
    static constexpr int PROD_BYTES = 4 * OPER_BYTES;        // one product: A (hi+lo) | B (hi+lo)
    // Products per pipeline stage.  The producer lane, the MMA-issuing lane and the hand-offs between the roles cost several
    // hundred clocks PER STAGE whatever its size (measured, profiles/r02_f32_small_leaves.md: at one 32-leaf product per stage
    // the issuing lane was busy 656 clk per product for 188 clk of MMAs), so a stage carries up to GP consecutive products of
    // one C tile: 64 KiB of operands per stage at both leaf sizes.  The GP products are chained into ONE TMEM accumulator set (16 MMAs at
    // 32-leaves, 8 at 64; the tensor core truncates when it adds into the accumulator, so chains stay short: bias ~16 * 2^-24
    // relative, inside the 1e-5 bar); the epilogue adds the chains in k order with round-to-nearest fp32 adds.
    static constexpr int GP = BS == 32 ? 4 : 1;
    static constexpr int CH = BS == 32 ? 1 : 2;              // stages chained into one accumulator set (16 MMAs either way)
    static constexpr int STAGE_BYTES = GP * PROD_BYTES;
    static constexpr int NST = (192 * 1024 / STAGE_BYTES) > 8 ? 8 : (192 * 1024 / STAGE_BYTES);
    static constexpr int MM = 2 * BS, NN = 2 * BS;           // stacked MMA shape
    static constexpr int SLAB_MN = KC * 128, SLAB_K = BS * 128;
    static constexpr int EPI_H = BS / 32;                    // 32-column groups of C
    static constexpr int EPI_WARPS = 4 * EPI_H;
    static constexpr int STG_BYTES = 2 * EPI_H * 32 * 32 * 4;   // lo-row partial tiles handed to the hi-row warps
    static constexpr int HEADER_BYTES = 1024;
    static constexpr int SMEM_BYTES = 1024 + HEADER_BYTES + NST * STAGE_BYTES + STG_BYTES;
    // Accumulator ring: every leaf product gets its own TMEM accumulator set (NN columns); all 512 columns are used (8 sets
    // at 32-leaves, 4 at 64) so that the issue -> commit -> drain -> release round trip of one product (several hundred
    // clocks, longer than a 32-leaf product's MMAs) overlaps with the MMAs of the next ones.
    static constexpr int NSETS = 512 / NN;
    static constexpr int TMEM_COLS = NSETS * NN;
    static constexpr int THREADS = 512;
    // hi/lo split warps (warps 2..7) in CVT_GROUPS groups of CVT_WPG warps: group g owns the pipeline stages of iterations
    // g, g + CVT_GROUPS, ..., so CVT_GROUPS products are being split at once -- one product's split is a dependent chain
    // (load, subtract, store, proxy fence, arrive) of several hundred clocks.  Never more groups than stages: a group's first
    // wait would otherwise alias the parity of a phase that has not started.
    static constexpr int CVT_WARPS = 6;
    static constexpr int CVT_GROUPS = NST >= 6 ? 6 : (NST >= 3 ? 3 : 2);
    static constexpr int CVT_WPG = CVT_WARPS / CVT_GROUPS;
    static constexpr int KSTEPS = KC / 8;
};

template <int BS, bool TA, bool TB>
__global__ void __launch_bounds__(Q4Cfg<BS>::THREADS, 1)
k_gemm_f32_q4(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
              const uint2* __restrict__ ab, const uint64_t* __restrict__ begin, uint32_t n_ctiles,
              const uint32_t* __restrict__ tile_list, unsigned* __restrict__ next_tile, float* __restrict__ Ct) {
    using Cfg = Q4Cfg<BS>;
    constexpr int NST = Cfg::NST, KC = Cfg::KC;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    F32Header* hd = reinterpret_cast<F32Header*>(smem);
    unsigned char* stages = smem + Cfg::HEADER_BYTES;
    float* stg = reinterpret_cast<float*>(stages + (size_t)NST * Cfg::STAGE_BYTES);
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(smem_u32(&hd->full_raw[s]), 1);
            mbar_init(smem_u32(&hd->full_cvt[s]), Cfg::CVT_WPG);   // the split warps of the group that owns the stage
            mbar_init(smem_u32(&hd->empty[s]), 1);
        }
        for (int a = 0; a < Cfg::NSETS; ++a) {
            mbar_init(smem_u32(&hd->tmem_full[a]), 1);
            mbar_init(smem_u32(&hd->tmem_empty[a]), Cfg::EPI_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&hd->tmem_base), Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = hd->tmem_base;

    if (warp == 0) {
        // ===== TMA producer: raw operand slabs land in the "hi" positions of the stacked layout.  The warp walks the task
        // list together (next C tile claimed one tile ahead, 32 (A tile, B tile) pairs per coalesced load): a 32-leaf
        // product lasts a few hundred clocks, less than one dependent index fetch; lane 0 issues the copies =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
        }
        uint32_t it = 0;
        unsigned claimed = 0;
        if (lane == 0) claimed = atomicAdd(next_tile, 1u);
        for (;;) {
            unsigned tile = __shfl_sync(0xffffffffu, claimed, 0);
            if (tile >= n_ctiles) break;
            if (lane == 0) claimed = atomicAdd(next_tile, 1u);   // consumed at the top of the next round
            if (tile_list) tile = tile_list[tile];
            const uint64_t bnd = begin[tile + (lane & 1u)];
            const uint64_t p0 = __shfl_sync(0xffffffffu, bnd, 0), p1 = __shfl_sync(0xffffffffu, bnd, 1);
            for (uint64_t pb = p0; pb < p1; pb += 32) {
                const uint2 mine = (pb + lane < p1) ? ab[pb + lane] : make_uint2(0u, 0u);   // lane l: operands of product pb + l
                const int cnt = (int)((p1 - pb) < 32 ? (p1 - pb) : 32);
                for (int j0 = 0; j0 < cnt; j0 += Cfg::GP, ++it) {      // one stage = products [pb + j0, pb + j0 + n)
                    const int n = cnt - j0 < Cfg::GP ? cnt - j0 : Cfg::GP;
                    const uint32_t s = it % NST, ph = (it / NST) & 1u;
                    const uint32_t fb = smem_u32(&hd->full_raw[s]);
                    // (operand indices are fetched BEFORE the wait: with three 64 KiB stages the time from "stage freed" to
                    // "copies issued" is on the critical path)
                    const uint2 tj = Cfg::GP > 1 ? mine : make_uint2(__shfl_sync(0xffffffffu, mine.x, j0), __shfl_sync(0xffffffffu, mine.y, j0));
                    if (lane == 0) {
                        mbar_wait(smem_u32(&hd->empty[s]), ph ^ 1u);
                        hd->ring[it & 15u].ctile = (int)tile;
                        hd->ring[it & 15u].flags = (pb + j0 == p0 ? 1 : 0) | (pb + j0 + n == p1 ? 2 : 0) | (n << 8);
                        mbar_arrive_expect_tx(fb, (uint32_t)n * 2u * Cfg::OPER_BYTES);
                    }
                    if (Cfg::GP > 1) __syncwarp();
                    // lanes j0 .. j0 + n - 1 issue one product's copies each (GP = 1: lane 0 issues for lane j0)
                    const int l = Cfg::GP > 1 ? (int)lane - j0 : (lane == 0 ? 0 : -1);
                    if (l >= 0 && l < n) {
                        const uint2 t = tj;
                        const uint32_t sa = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES + (size_t)l * Cfg::PROD_BYTES);
                        const uint32_t sb = sa + 2 * Cfg::OPER_BYTES;
                        if (TA) {   // K-major: [BS mn][32 k] slabs, hi slab j at 2j * SLAB_K
#pragma unroll
                            for (int jj = 0; jj < KC / 32; ++jj) tma_box_g2s(sa + 2 * jj * Cfg::SLAB_K, &mapA, 32 * jj, (int)t.x * BS, fb);
                        } else {    // MN-major: [KC k][32 mn] slabs, hi slabs first
#pragma unroll
                            for (int jj = 0; jj < BS / 32; ++jj) tma_box_g2s(sa + jj * Cfg::SLAB_MN, &mapA, 32 * jj, (int)t.x * BS, fb);
                        }
                        if (TB) {
#pragma unroll
                            for (int jj = 0; jj < BS / 32; ++jj) tma_box_g2s(sb + jj * Cfg::SLAB_MN, &mapB, 32 * jj, (int)t.y * BS, fb);
                        } else {
#pragma unroll
                            for (int jj = 0; jj < KC / 32; ++jj) tma_box_g2s(sb + 2 * jj * Cfg::SLAB_K, &mapB, 32 * jj, (int)t.y * BS, fb);
                        }
                    }
                    __syncwarp();
                }
            }
        }
        if (lane == 0) {   // one terminal stage per split group (each of them watches only its own stages)
            for (int e = 0; e < Cfg::CVT_GROUPS; ++e, ++it) {
                const uint32_t s = it % NST, ph = (it / NST) & 1u;
                mbar_wait(smem_u32(&hd->empty[s]), ph ^ 1u);
                hd->ring[it & 15u].ctile = -1;
                hd->ring[it & 15u].flags = 4;
                mbar_arrive(smem_u32(&hd->full_raw[s]));
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one stacked MMA per K-step =====
        if (lane == 0) {
            constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((TA ? 0u : 1u) << 15) | ((TB ? 1u : 0u) << 16) |
                                       ((uint32_t)(Cfg::NN >> 3) << 17) | ((uint32_t)(Cfg::MM >> 4) << 24);
            constexpr uint32_t A_LBO = TA ? 16 : Cfg::SLAB_MN, B_LBO = TB ? Cfg::SLAB_MN : 16;
            constexpr uint32_t A_SBO = TA ? 1024 : 512, B_SBO = TB ? 512 : 1024;
            constexpr uint32_t A_LT = TA ? 2 : 1, B_LT = TB ? 1 : 2;
            // (Interleaving the K-steps of consecutive products over their accumulator sets was tried and is SLOWER:
            // 100 -> 72 TF/s at 64-leaves, 23.6 -> 20.8 at 32 -- the issuer then waits for whole batches of stages.)
            uint32_t chain = 0;       // accumulator-set uses so far
            int in_chain = 0;
            for (uint32_t it = 0;; ++it) {
                const uint32_t s = it % NST, ph = (it / NST) & 1u;
                mbar_wait(smem_u32(&hd->full_cvt[s]), ph);
                const GemmMeta m = hd->ring[it & 15u];
                const uint32_t as = chain % Cfg::NSETS;
                if (in_chain == 0) mbar_wait(smem_u32(&hd->tmem_empty[as]), ((chain / Cfg::NSETS) & 1u) ^ 1u);   // epilogue drained this set
                if (m.flags & 4) {   // (a chain never spans C tiles, so none is open here)
                    mbar_arrive(smem_u32(&hd->tmem_full[as]));   // the epilogue finds the terminal entry in the ring itself
                    break;
                }
                tc_fence_after();
                const uint32_t d = tmem_base + as * Cfg::NN;
                const int n = Cfg::GP == 1 ? 1 : (m.flags >> 8);
                const uint32_t s0 = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES);
                // descriptors of the stage's first product, first K-step; the others differ in the start-address field only
                const uint64_t da0 = umma_desc(s0, A_LBO, A_SBO, A_LT), db0 = umma_desc(s0 + 2 * Cfg::OPER_BYTES, B_LBO, B_SBO, B_LT);
                for (int j = 0; j < n; ++j) {
#pragma unroll
                    for (int ks = 0; ks < Cfg::KSTEPS; ++ks) {
                        const uint32_t ao = TA ? (uint32_t)((ks >> 2) * 2 * Cfg::SLAB_K + (ks & 3) * 32) : (uint32_t)(ks * 1024);
                        const uint32_t bo = TB ? (uint32_t)(ks * 1024) : (uint32_t)((ks >> 2) * 2 * Cfg::SLAB_K + (ks & 3) * 32);
                        mma_tf32(d, da0 + (uint64_t)((j * Cfg::PROD_BYTES + ao) >> 4), db0 + (uint64_t)((j * Cfg::PROD_BYTES + bo) >> 4), IDESC,
                                 (ks || j || in_chain) ? 1u : 0u);
                    }
                }
                tc_commit(smem_u32(&hd->empty[s]));
                if ((m.flags & 2) || ++in_chain == Cfg::CH) {   // hand the set to the epilogue (which reads the same ring entries)
                    tc_commit(smem_u32(&hd->tmem_full[as]));
                    ++chain;
                    in_chain = 0;
                }
            }
        }
    } else if (warp >= 2 && warp < 2 + Cfg::CVT_WARPS) {
        // ===== lo = x - trunc_tf32(x) next to every raw slab (the raw slab itself serves as hi); group g owns iterations g, g+G, ... =====
        const unsigned tid = ((warp - 2) % Cfg::CVT_WPG) * 32 + lane;
        for (uint32_t it = (warp - 2) / Cfg::CVT_WPG;; it += Cfg::CVT_GROUPS) {
            const uint32_t s = it % NST, ph = (it / NST) & 1u;
            mbar_wait(smem_u32(&hd->full_raw[s]), ph);
            const int flags = hd->ring[it & 15u].flags;
            if (!(flags & 4))
            for (int pj = 0; pj < (Cfg::GP == 1 ? 1 : (flags >> 8)); ++pj) {
                unsigned char* st = stages + (size_t)s * Cfg::STAGE_BYTES + (size_t)pj * Cfg::PROD_BYTES;
#pragma unroll
                for (int op = 0; op < 2; ++op) {
                    const bool kmajor = op == 0 ? TA : !TB;
                    // K-major: KC/32 raw ranges of SLAB_K bytes, 2*SLAB_K apart, lo right behind each; MN-major: one range, lo at +OPER
                    const int n_ranges = kmajor ? KC / 32 : 1;
                    const int range_bytes = kmajor ? Cfg::SLAB_K : Cfg::OPER_BYTES;
                    const int lo_off = kmajor ? Cfg::SLAB_K : Cfg::OPER_BYTES;
                    for (int rg = 0; rg < n_ranges; ++rg) {
                        const float4* hi = reinterpret_cast<const float4*>(st + op * 2 * Cfg::OPER_BYTES + rg * 2 * range_bytes);
                        float4* lo = reinterpret_cast<float4*>(st + op * 2 * Cfg::OPER_BYTES + rg * 2 * range_bytes + lo_off);
#pragma unroll 4
                        for (int i = (int)tid; i < range_bytes / 16; i += Cfg::CVT_WPG * 32) {
                            const float4 x = hi[i];
                            float4 l;
                            l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                            l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                            l.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                            l.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                            lo[i] = l;
                        }
                    }
                }
            }
            if (!(flags & 4)) fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&hd->full_cvt[s]));
            if (flags & 4) break;
        }
    } else if (warp >= 8 && (warp - 8) < Cfg::EPI_WARPS) {
        // ===== epilogue: warp (q,h): TMEM lane quadrant q (0,1 = hi rows, 2,3 = lo rows), C columns [32h, 32h+32) =====
        const unsigned q = (warp - 8) & 3, h = (warp - 8) >> 2;
        const bool lo_rows = q >= 2;
        // M = 128 (BS = 64): D row = lane index; M = 64 (BS = 32): D row i sits in lane 32*(i/16) + i%16
        const int crow = BS == 64 ? (int)((q & 1) * 32 + lane) : (lane < 16 ? (int)((q & 1) * 16 + lane) : BS);
        float* my_stg = stg + (size_t)(((q & 1) * Cfg::EPI_H + h) * 32 * 32);
        float acc[32];
        uint32_t it_e = 0;            // stage sequence number of the next ring entry this warp consumes
        for (uint32_t pc = 0;; ++pc) {
            const uint32_t as = pc % Cfg::NSETS;
            mbar_wait(smem_u32(&hd->tmem_full[as]), (pc / Cfg::NSETS) & 1u);
            // the accumulator set holds the stages [it_e, ...) of one chain: up to CH stages, closed early by the end of the C tile
            GemmMeta m = hd->ring[it_e & 15u];
            int flags = m.flags & 7;
            if (flags & 4) break;
            ++it_e;
#pragma unroll
            for (int c = 1; c < Cfg::CH; ++c) {
                if (flags & 2) break;
                m = hd->ring[it_e & 15u];
                flags |= m.flags & 3;
                ++it_e;
            }
            const int ctile = m.ctile;
            tc_fence_after();
            uint32_t r1[32], r2[32];
            tmem_ld32(tmem_base + ((q * 32u) << 16) + as * Cfg::NN + BS + h * 32, r2);   // x * B_lo
            tmem_ld32(tmem_base + ((q * 32u) << 16) + as * Cfg::NN + h * 32, r1);        // x * B_hi
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&hd->tmem_empty[as]));
            if (flags & 1) {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = __fadd_rn(__uint_as_float(r2[j]), __uint_as_float(r1[j]));
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = __fadd_rn(__fadd_rn(acc[j], __uint_as_float(r2[j])), __uint_as_float(r1[j]));
            }
            if (flags & 2) {   // k-list of this C tile done: lo-row partial sums -> hi-row warps -> global
                if (lo_rows) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) my_stg[j * 32 + lane] = acc[j];
                }
                asm volatile("bar.sync 1, %0;" ::"r"(Cfg::EPI_WARPS * 32) : "memory");
                if (!lo_rows && crow < BS) {
                    float* C = Ct + (size_t)ctile * BS * BS + (size_t)(h * 32) * BS + crow;
#pragma unroll
                    for (int j = 0; j < 32; ++j) C[(size_t)j * BS] = __fadd_rn(acc[j], my_stg[j * 32 + lane]);
                }
                asm volatile("bar.sync 1, %0;" ::"r"(Cfg::EPI_WARPS * 32) : "memory");
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// 2-D fp32 view of a tile pool: dim0 = leaf row (contiguous), dim1 = leaf column + BS * tile; 128-B swizzled boxes
void make_f32_map(CUtensorMap* map, const void* tiles, size_t n_tiles, int LS, int box_rows, int box_cols, bool mn_major) {
    EncodeTiledFn enc = encode_tiled_fn();
    cuuint64_t gdim[2] = {(cuuint64_t)LS, (cuuint64_t)LS * n_tiles};
    cuuint64_t gstr[1] = {(cuuint64_t)LS * 4};
    cuuint32_t box[2] = {(cuuint32_t)box_rows, (cuuint32_t)box_cols};
    cuuint32_t estr[2] = {1, 1};
    if (!enc || enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(tiles), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        throw Error(HBSM_E_CUDA, "hbsm_b200: the driver refused the tensor map of an fp32 leaf operand");
}


constexpr uint32_t P32_NONE = 0xFFFFFFFFu;   // "no tile here": the member / operand reads the zero leaf

const float* zero_leaf_f32() {   // one zero leaf (32 x 32 fp32) for the group members that have no product at some k
    static float* z = nullptr;
    if (!z) {
        HB_CUDA(cudaMalloc((void**)&z, 32 * 32 * sizeof(float)));
        HB_CUDA(cudaMemset(z, 0, 32 * 32 * sizeof(float)));
    }
    return z;
}

// ---------------------------------------------------------------------------------------------------
// 32-leaves, 2 x 2 groups: four C tiles per MMA.
//
// The Morton-aligned 2 x 2 block of C tiles (ci0 + r, cj0 + c), r, c in {0, 1}, is up to four CONSECUTIVE entries of C's table
// (keys 4q + 2c + r).  Per contraction index k its products read A(ci0 + r, k) and B(k, cj0 + c): one M = N = 128 MMA per K-step,
//        [A0_hi ; A0_lo ; A1_hi ; A1_lo] (128 x 32)  x  [B0_hi | B0_lo | B1_hi | B1_lo] (32 x 128),
// computes all four.  Measured (tools/mma_probe.cu, profiles/r02_mma_probe.json): a kind::tf32 MMA with fresh operands costs
// ~66 clk whatever its shape up to M = N = 128, so this is the shape at which it runs at the full tensor rate (the M = N = 64
// MMA of the single-tile kernel uses a quarter of it), and a leaf product moves 20 KiB through shared memory instead of 40
// (single tiles) -- small leaves are shared-memory-bound (profiles/r02_f32_small_leaves.md).  Vertical pairs only (M = 128,
// N = 64, 30 KiB per product) were measured on the way: 51 TF/s, against 35 (single tiles) and 74 (this kernel).
// Exactness: a group-k whose EXECUTED combinations W form a rectangle R x S is one super-product with the operands of the
// rows not in R / columns not in S replaced by the zero tile (exact +0 for those members); any other W (three of four, or a
// diagonal pair -- SpAMM prunes per leaf pair) is issued as two super-products, one per row, each a rectangle.  So every member
// accumulates exactly its own k-list, in k order, plus exact zeros: the executed-product set and the partial sums are those of
// the single-tile kernel.  TMEM lane quadrant q = 2r + (0 hi rows | 1 lo rows); accumulator columns [64c, 64c + 32) = x * Bc_hi,
// [64c + 32, 64c + 64) = x * Bc_lo.
// ---------------------------------------------------------------------------------------------------
struct G32Cfg {
    static constexpr int BS = 32;
    static constexpr int SLAB = 32 * 128;
    static constexpr int SP_BYTES = 8 * SLAB;                // A: hi0 lo0 hi1 lo1 | B: hi0 lo0 hi1 lo1  (32 KiB)
    static constexpr int GP = 2;                             // super-products per stage = chained into one accumulator set (8 MMAs)
    static constexpr int STAGE_BYTES = GP * SP_BYTES;        // 64 KiB
    static constexpr int NST = 3;
    static constexpr int MM = 128, NN = 128;
    static constexpr int NSETS = 512 / NN;
    static constexpr int TMEM_COLS = 512;
    static constexpr int THREADS = 512;
    static constexpr int CVT_WARPS = 6, CVT_GROUPS = 3, CVT_WPG = 2;
    static constexpr int EPI_WARPS = 8;
    static constexpr int KSTEPS = 4;
    static constexpr int STG_BYTES = 4 * 32 * 32 * 4;        // lo-row partial tiles of the four members
    static constexpr int HEADER_BYTES = 1024;
    static constexpr int SMEM_BYTES = 1024 + HEADER_BYTES + NST * STAGE_BYTES + STG_BYTES;
};
struct G32Header {
    uint64_t full_raw[8], full_cvt[8], empty[8], tmem_full[8], tmem_empty[8];
    uint32_t tmem_base;
    uint32_t pad_[3];
    int4 ring_tiles[16];                                     // C tile of member m = 2c + r, or -1
    int ring_flags[16];                                      // 1 first stage of the group, 2 last, 4 end; n << 8
};
static_assert(sizeof(G32Header) <= G32Cfg::HEADER_BYTES, "header");

template <bool TA, bool TB>
__global__ void __launch_bounds__(G32Cfg::THREADS, 1)
k_gemm_f32_g32(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapZ,
               const uint4* __restrict__ gops /* {A row 0, A row 1, B col 0, B col 1} tiles per super-product; P32_NONE = zero tile */,
               const uint64_t* __restrict__ gbegin, const int4* __restrict__ gtiles, const uint64_t* __restrict__ n_groups_dev,
               unsigned* __restrict__ next_group, float* __restrict__ Ct) {
    using Cfg = G32Cfg;
    constexpr int NST = Cfg::NST, BS = Cfg::BS;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    G32Header* hd = reinterpret_cast<G32Header*>(smem);
    unsigned char* stages = smem + Cfg::HEADER_BYTES;
    float* stg = reinterpret_cast<float*>(stages + (size_t)NST * Cfg::STAGE_BYTES);
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned n_groups = (unsigned)*n_groups_dev;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(smem_u32(&hd->full_raw[s]), 1);
            mbar_init(smem_u32(&hd->full_cvt[s]), Cfg::CVT_WPG);
            mbar_init(smem_u32(&hd->empty[s]), 1);
        }
        for (int a = 0; a < Cfg::NSETS; ++a) {
            mbar_init(smem_u32(&hd->tmem_full[a]), 1);
            mbar_init(smem_u32(&hd->tmem_empty[a]), Cfg::EPI_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&hd->tmem_base), Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = hd->tmem_base;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapZ) : "memory");
        }
        uint32_t it = 0;
        unsigned claimed = 0;
        if (lane == 0) claimed = atomicAdd(next_group, 1u);
        for (;;) {
            const unsigned g = __shfl_sync(0xffffffffu, claimed, 0);
            if (g >= n_groups) break;
            if (lane == 0) claimed = atomicAdd(next_group, 1u);
            const uint64_t bnd = gbegin[g + (lane & 1u)];
            const uint64_t p0 = __shfl_sync(0xffffffffu, bnd, 0), p1 = __shfl_sync(0xffffffffu, bnd, 1);
            const int4 ct = gtiles[g];
            for (uint64_t pb = p0; pb < p1; pb += 32) {
                const uint4 mine = (pb + lane < p1) ? gops[pb + lane] : make_uint4(0u, 0u, 0u, 0u);
                const int cnt = (int)((p1 - pb) < 32 ? (p1 - pb) : 32);
                for (int j0 = 0; j0 < cnt; j0 += Cfg::GP, ++it) {
                    const int n = cnt - j0 < Cfg::GP ? cnt - j0 : Cfg::GP;
                    const uint32_t s = it % NST, ph = (it / NST) & 1u;
                    const uint32_t fb = smem_u32(&hd->full_raw[s]);
                    if (lane == 0) {
                        mbar_wait(smem_u32(&hd->empty[s]), ph ^ 1u);
                        hd->ring_tiles[it & 15u] = ct;
                        hd->ring_flags[it & 15u] = (pb + j0 == p0 ? 1 : 0) | (pb + j0 + n == p1 ? 2 : 0) | (n << 8);
                        mbar_arrive_expect_tx(fb, (uint32_t)n * 4u * Cfg::SLAB);
                    }
                    __syncwarp();
                    const int l = (int)lane - j0;
                    if (l >= 0 && l < n) {   // raw tiles land in the "hi" slabs 0, 2 (A rows) and 4, 6 (B columns)
                        const uint32_t sa = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES + (size_t)l * Cfg::SP_BYTES);
                        if (mine.x != P32_NONE) tma_box_g2s(sa, &mapA, 0, (int)mine.x * BS, fb);
                        else tma_box_g2s(sa, &mapZ, 0, 0, fb);
                        if (mine.y != P32_NONE) tma_box_g2s(sa + 2 * Cfg::SLAB, &mapA, 0, (int)mine.y * BS, fb);
                        else tma_box_g2s(sa + 2 * Cfg::SLAB, &mapZ, 0, 0, fb);
                        if (mine.z != P32_NONE) tma_box_g2s(sa + 4 * Cfg::SLAB, &mapB, 0, (int)mine.z * BS, fb);
                        else tma_box_g2s(sa + 4 * Cfg::SLAB, &mapZ, 0, 0, fb);
                        if (mine.w != P32_NONE) tma_box_g2s(sa + 6 * Cfg::SLAB, &mapB, 0, (int)mine.w * BS, fb);
                        else tma_box_g2s(sa + 6 * Cfg::SLAB, &mapZ, 0, 0, fb);
                    }
                    __syncwarp();
                }
            }
        }
        if (lane == 0) {
            for (int e = 0; e < Cfg::CVT_GROUPS; ++e, ++it) {
                const uint32_t s = it % NST, ph = (it / NST) & 1u;
                mbar_wait(smem_u32(&hd->empty[s]), ph ^ 1u);
                hd->ring_flags[it & 15u] = 4;
                mbar_arrive(smem_u32(&hd->full_raw[s]));
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            constexpr uint32_t IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((TA ? 0u : 1u) << 15) | ((TB ? 1u : 0u) << 16) |
                                       ((uint32_t)(Cfg::NN >> 3) << 17) | ((uint32_t)(Cfg::MM >> 4) << 24);
            constexpr uint32_t A_LBO = TA ? 16 : Cfg::SLAB, B_LBO = TB ? Cfg::SLAB : 16;
            constexpr uint32_t A_SBO = TA ? 1024 : 512, B_SBO = TB ? 512 : 1024;
            constexpr uint32_t A_LT = TA ? 2 : 1, B_LT = TB ? 1 : 2;
            for (uint32_t it = 0;; ++it) {
                const uint32_t s = it % NST, ph = (it / NST) & 1u;
                mbar_wait(smem_u32(&hd->full_cvt[s]), ph);
                const int flags = hd->ring_flags[it & 15u];
                const uint32_t as = it % Cfg::NSETS;
                mbar_wait(smem_u32(&hd->tmem_empty[as]), ((it / Cfg::NSETS) & 1u) ^ 1u);
                if (flags & 4) {
                    mbar_arrive(smem_u32(&hd->tmem_full[as]));
                    break;
                }
                tc_fence_after();
                const uint32_t d = tmem_base + as * Cfg::NN;
                const int n = flags >> 8;
                const uint32_t s0 = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES);
                const uint64_t da0 = umma_desc(s0, A_LBO, A_SBO, A_LT), db0 = umma_desc(s0 + 4 * Cfg::SLAB, B_LBO, B_SBO, B_LT);
                for (int j = 0; j < n; ++j) {
#pragma unroll
                    for (int ks = 0; ks < Cfg::KSTEPS; ++ks) {
                        const uint32_t ao = TA ? (uint32_t)(ks * 32) : (uint32_t)(ks * 1024);
                        const uint32_t bo = TB ? (uint32_t)(ks * 1024) : (uint32_t)(ks * 32);
                        mma_tf32(d, da0 + (uint64_t)((j * Cfg::SP_BYTES + ao) >> 4), db0 + (uint64_t)((j * Cfg::SP_BYTES + bo) >> 4), IDESC,
                                 (ks || j) ? 1u : 0u);
                    }
                }
                tc_commit(smem_u32(&hd->empty[s]));
                tc_commit(smem_u32(&hd->tmem_full[as]));
            }
        }
    } else if (warp >= 2 && warp < 2 + Cfg::CVT_WARPS) {
        // ===== lo = x - trunc_tf32(x): slabs 1, 3, 5, 7 of every super-product from the raw slabs 0, 2, 4, 6 =====
        const unsigned tid = ((warp - 2) % Cfg::CVT_WPG) * 32 + lane;
        for (uint32_t it = (warp - 2) / Cfg::CVT_WPG;; it += Cfg::CVT_GROUPS) {
            const uint32_t s = it % NST, ph = (it / NST) & 1u;
            mbar_wait(smem_u32(&hd->full_raw[s]), ph);
            const int flags = hd->ring_flags[it & 15u];
            if (!(flags & 4)) {
                for (int pj = 0; pj < (flags >> 8); ++pj) {
                    unsigned char* st = stages + (size_t)s * Cfg::STAGE_BYTES + (size_t)pj * Cfg::SP_BYTES;
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
                        const float4* hi = reinterpret_cast<const float4*>(st + r * 2 * Cfg::SLAB);
                        float4* lo = reinterpret_cast<float4*>(st + r * 2 * Cfg::SLAB + Cfg::SLAB);
#pragma unroll 4
                        for (int i = (int)tid; i < Cfg::SLAB / 16; i += Cfg::CVT_WPG * 32) {
                            const float4 x = hi[i];
                            float4 l;
                            l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                            l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                            l.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                            l.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                            lo[i] = l;
                        }
                    }
                }
                fence_proxy_async();
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&hd->full_cvt[s]));
            if (flags & 4) break;
        }
    } else if (warp >= 8 && (warp - 8) < Cfg::EPI_WARPS) {
        // ===== epilogue: warp (q, c): TMEM lane quadrant q (member row r = q >> 1, hi rows if q even else lo rows), member column c =====
        const unsigned q = (warp - 8) & 3, c = (warp - 8) >> 2;
        const bool lo_rows = (q & 1u) != 0;
        const unsigned member = 2 * c + (q >> 1);
        float* my_stg = stg + (size_t)(member * 32 * 32);
        float acc[32];
        for (uint32_t pc = 0;; ++pc) {
            const uint32_t as = pc % Cfg::NSETS;
            mbar_wait(smem_u32(&hd->tmem_full[as]), (pc / Cfg::NSETS) & 1u);
            const int flags = hd->ring_flags[pc & 15u];
            if (flags & 4) break;
            const int4 tiles = hd->ring_tiles[pc & 15u];
            tc_fence_after();
            uint32_t r1[32], r2[32];
            tmem_ld32(tmem_base + ((q * 32u) << 16) + as * Cfg::NN + c * 64 + BS, r2);   // x * Bc_lo
            tmem_ld32(tmem_base + ((q * 32u) << 16) + as * Cfg::NN + c * 64, r1);        // x * Bc_hi
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&hd->tmem_empty[as]));
            if (flags & 1) {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = __fadd_rn(__uint_as_float(r2[j]), __uint_as_float(r1[j]));
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = __fadd_rn(__fadd_rn(acc[j], __uint_as_float(r2[j])), __uint_as_float(r1[j]));
            }
            if (flags & 2) {   // the group's k-list is done: lo-row partial sums -> hi-row warps -> global
                if (lo_rows) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) my_stg[j * 32 + lane] = acc[j];
                }
                asm volatile("bar.sync 1, %0;" ::"r"(Cfg::EPI_WARPS * 32) : "memory");
                const int ctile = member == 0 ? tiles.x : (member == 1 ? tiles.y : (member == 2 ? tiles.z : tiles.w));
                if (!lo_rows && ctile >= 0) {
                    float* C = Ct + (size_t)ctile * BS * BS + lane;
#pragma unroll
                    for (int j = 0; j < 32; ++j) C[(size_t)j * BS] = __fadd_rn(acc[j], my_stg[j * 32 + lane]);
                }
                asm volatile("bar.sync 1, %0;" ::"r"(Cfg::EPI_WARPS * 32) : "memory");
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

// ---- 2 x 2 groups and their super-product lists, built from the task list on the device ----
// (tile_list, if given, is an ascending subset of C's table -- e.g. the C tiles of a sharded product that read no halo tile:
// position i stands for tile tile_list[i], and a group only takes the members that are in the list)
__device__ __forceinline__ uint32_t g32_tile(const uint32_t* __restrict__ tile_list, uint32_t i) { return tile_list ? tile_list[i] : i; }
__global__ void k_g32_heads(const uint64_t* __restrict__ ckeys, const uint32_t* __restrict__ tile_list, uint32_t n, uint32_t* __restrict__ head) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    head[t] = (t == 0 || (ckeys[g32_tile(tile_list, t - 1)] >> 2) != (ckeys[g32_tile(tile_list, t)] >> 2)) ? 1u : 0u;
}
// four sorted k-lists -> super-products in k order (one thread per group): count pass and fill pass
template <bool FILL>
__global__ void k_g32_merge(const uint64_t* __restrict__ ckeys, const uint32_t* __restrict__ tile_list, uint32_t n, const uint32_t* __restrict__ head, const uint64_t* __restrict__ gpos,
                            const uint64_t* __restrict__ begin, const uint2* __restrict__ ab, const uint32_t* __restrict__ task_k,
                            uint32_t* __restrict__ cnt, const uint64_t* __restrict__ gbegin, int4* __restrict__ gtiles, uint4* __restrict__ gops) {
    const uint32_t t0 = blockIdx.x * blockDim.x + threadIdx.x;
    if (t0 >= n || !head[t0]) return;
    const uint64_t quad = ckeys[g32_tile(tile_list, t0)] >> 2;
    int tile[4] = {-1, -1, -1, -1};
    uint64_t p[4] = {0, 0, 0, 0}, pe[4] = {0, 0, 0, 0};
    for (uint32_t i = t0; i < n && i < t0 + 4; ++i) {
        const uint32_t t = g32_tile(tile_list, i);
        if ((ckeys[t] >> 2) != quad) break;
        const int m = (int)(ckeys[t] & 3ull);   // member 2c + r
        tile[m] = (int)t;
        p[m] = begin[t];
        pe[m] = begin[t + 1];
    }
    const uint64_t g = gpos[t0];
    uint64_t out = FILL ? gbegin[g] : 0;
    uint32_t c = 0;
    for (;;) {
        uint32_t kmin = 0xFFFFFFFFu;
#pragma unroll
        for (int m = 0; m < 4; ++m)
            if (p[m] < pe[m]) kmin = min(kmin, task_k[p[m]]);
        if (kmin == 0xFFFFFFFFu) break;
        bool w[4];
        uint32_t a[2] = {P32_NONE, P32_NONE}, b[2] = {P32_NONE, P32_NONE};
        int nw = 0;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            w[m] = p[m] < pe[m] && task_k[p[m]] == kmin;
            if (w[m]) {
                ++nw;
                if (FILL) {
                    const uint2 o = ab[p[m]];
                    a[m & 1] = o.x;       // row r = m & 1
                    b[m >> 1] = o.y;      // column c = m >> 1
                }
                ++p[m];
            }
        }
        const int rows = ((w[0] || w[2]) ? 1 : 0) + ((w[1] || w[3]) ? 1 : 0);
        const int cols = ((w[0] || w[1]) ? 1 : 0) + ((w[2] || w[3]) ? 1 : 0);
        if (nw == rows * cols) {   // a rectangle: one super-product
            if (FILL) gops[out++] = make_uint4(a[0], a[1], b[0], b[1]);
            ++c;
        } else {                   // three of four, or a diagonal: one super-product per row
            if (FILL) {
                gops[out++] = make_uint4(a[0], P32_NONE, w[0] ? b[0] : P32_NONE, w[2] ? b[1] : P32_NONE);
                gops[out++] = make_uint4(P32_NONE, a[1], w[1] ? b[0] : P32_NONE, w[3] ? b[1] : P32_NONE);
            }
            c += 2;
        }
    }
    if (!FILL) cnt[g] = c;
    else gtiles[g] = make_int4(tile[0], tile[1], tile[2], tile[3]);
}

template <bool TA, bool TB>
void launch_g32_inst(const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, const uint64_t* ckeys, const uint32_t* task_k,
                     const uint32_t* tile_list, uint32_t n_ctiles, size_t n_products, float* Ct) {
    using Cfg = G32Cfg;
    CUtensorMap mapA, mapB, mapZ;
    make_f32_map(&mapA, A.tiles.p, A.L, 32, 32, 32, !TA);
    make_f32_map(&mapB, B.tiles.p, B.n_ext(), 32, 32, 32, TB);
    make_f32_map(&mapZ, zero_leaf_f32(), 1, 32, 32, 32, !TA);
    // (one zero map serves both operands: the swizzle mode only permutes where the zeros land)
    DevBuf<uint32_t> head(n_ctiles), cnt(n_ctiles);
    DevBuf<uint64_t> gpos((size_t)n_ctiles + 1), gbegin((size_t)n_ctiles + 1);
    DevBuf<int4> gtiles(n_ctiles);
    DevBuf<uint4> gops(std::max<size_t>(n_products, 1));
    cnt.zero();
    const unsigned gb = (n_ctiles + 255) / 256;
    HB_LAUNCH(k_g32_heads, gb, 256, 0, ckeys, tile_list, n_ctiles, head.p);
    exclusive_scan_u32(head.p, gpos.p, n_ctiles);
    HB_LAUNCH((k_g32_merge<false>), gb, 256, 0, ckeys, tile_list, n_ctiles, head.p, gpos.p, begin, ab, task_k, cnt.p, (const uint64_t*)nullptr,
              (int4*)nullptr, (uint4*)nullptr);
    exclusive_scan_u32(cnt.p, gbegin.p, n_ctiles);
    HB_LAUNCH((k_g32_merge<true>), gb, 256, 0, ckeys, tile_list, n_ctiles, head.p, gpos.p, begin, ab, task_k, (uint32_t*)nullptr, gbegin.p, gtiles.p,
              gops.p);
    DevBuf<unsigned> counter(1);
    counter.zero();
    auto kfn = k_gemm_f32_g32<TA, TB>;
    static bool configured = false;
    if (!configured) {
        HB_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        configured = true;
    }
    const unsigned grid = std::min<unsigned>(n_ctiles, (unsigned)engine().sm_count);
    HB_LAUNCH(kfn, grid, Cfg::THREADS, Cfg::SMEM_BYTES, mapA, mapB, mapZ, gops.p, gbegin.p, gtiles.p, gpos.p + n_ctiles, counter.p, Ct);
}

void launch_g32(bool tA, bool tB, const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, const uint64_t* ckeys,
                const uint32_t* task_k, const uint32_t* tile_list, uint32_t n, size_t n_products, float* Ct) {
    if (!tA && !tB) launch_g32_inst<false, false>(A, B, ab, begin, ckeys, task_k, tile_list, n, n_products, Ct);
    else if (!tA && tB) launch_g32_inst<false, true>(A, B, ab, begin, ckeys, task_k, tile_list, n, n_products, Ct);
    else if (tA && !tB) launch_g32_inst<true, false>(A, B, ab, begin, ckeys, task_k, tile_list, n, n_products, Ct);
    else launch_g32_inst<true, true>(A, B, ab, begin, ckeys, task_k, tile_list, n, n_products, Ct);
}


// ---------------------------------------------------------------------------------------------------
// 64-leaves, 2 x 2 groups.  Same groups and super-product lists as the 32-leaf kernel above (k_g32_heads / k_g32_merge work on
// C's table whatever the leaf size), different operand stacking: M = 128 is TWO row tiles, and the hi/lo split is spread over
// two MMAs per K-step instead of being stacked along M,
//     D[128 x 256]  = [A0_hi ; A1_hi] x [B0_hi | B1_hi | B0_lo | B1_lo]        (N = 256: hi*hi and hi*lo of all four members)
//     D[:, 0:128]  += [A0_lo ; A1_lo] x [B0_hi | B1_hi]                        (N = 128: lo*hi into the hi*hi columns)
// i.e. 194 clk and 20 KiB of operand fetch per K-step for FOUR products (single-tile kernel: 66 clk and 8 KiB for one): 88 KiB
// through shared memory per leaf product instead of 160.  One pipeline stage = one K-half (32 k) of a super-product = 64 KiB
// (hi and lo stacks of A and B, 16 KiB each); an accumulator set (256 TMEM columns, two sets) holds one super-product = two
// stages = 16 MMAs.  There are no "lo rows": every accumulator lane is a C row, so the epilogue is 8 warps of 32 rows x 64
// columns adding  D[:, hi cols] + D[:, lo cols]  into registers -- no staging, no CTA-level barrier.
// ---------------------------------------------------------------------------------------------------
struct G64Cfg {
    static constexpr int BS = 64, KC = 32;
    static constexpr int STACK = 128 * KC * 4;               // one stack: two tiles' K-half, 16 KiB
    static constexpr int STAGE_BYTES = 4 * STACK;            // A_hi | A_lo | B_hi | B_lo
    static constexpr int NST = 3;
    static constexpr int NSETS = 2;                          // 256 columns each
    static constexpr int TMEM_COLS = 512;
    static constexpr int THREADS = 512;
    static constexpr int CVT_WARPS = 6, CVT_GROUPS = 3, CVT_WPG = 2;
    static constexpr int EPI_WARPS = 8;
    static constexpr int KSTEPS = KC / 8;
    static constexpr int HEADER_BYTES = 1024;
    static constexpr int SMEM_BYTES = 1024 + HEADER_BYTES + NST * STAGE_BYTES;
};

const float* zero_leaf_f32_64() {
    static float* z = nullptr;
    if (!z) {
        HB_CUDA(cudaMalloc((void**)&z, 64 * 64 * sizeof(float)));
        HB_CUDA(cudaMemset(z, 0, 64 * 64 * sizeof(float)));
    }
    return z;
}

template <bool TA, bool TB>
__global__ void __launch_bounds__(G64Cfg::THREADS, 1)
k_gemm_f32_g64(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapZa,
               const __grid_constant__ CUtensorMap mapZb, const uint4* __restrict__ gops, const uint64_t* __restrict__ gbegin,
               const int4* __restrict__ gtiles, const uint64_t* __restrict__ n_groups_dev, unsigned* __restrict__ next_group,
               float* __restrict__ Ct) {
    using Cfg = G64Cfg;
    constexpr int NST = Cfg::NST, BS = Cfg::BS, KC = Cfg::KC;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    G32Header* hd = reinterpret_cast<G32Header*>(smem);
    unsigned char* stages = smem + Cfg::HEADER_BYTES;
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const unsigned n_groups = (unsigned)*n_groups_dev;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(smem_u32(&hd->full_raw[s]), 1);
            mbar_init(smem_u32(&hd->full_cvt[s]), Cfg::CVT_WPG);
            mbar_init(smem_u32(&hd->empty[s]), 1);
        }
        for (int a = 0; a < Cfg::NSETS; ++a) {
            mbar_init(smem_u32(&hd->tmem_full[a]), 1);
            mbar_init(smem_u32(&hd->tmem_empty[a]), Cfg::EPI_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(smem_u32(&hd->tmem_base), Cfg::TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = hd->tmem_base;

    if (warp == 0) {
        // ===== TMA producer: per super-product two stages (K halves); lanes 0..3 copy one tile's K-half each =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapZa) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapZb) : "memory");
        }
        uint32_t it = 0;
        unsigned claimed = 0;
        if (lane == 0) claimed = atomicAdd(next_group, 1u);
        for (;;) {
            const unsigned g = __shfl_sync(0xffffffffu, claimed, 0);
            if (g >= n_groups) break;
            if (lane == 0) claimed = atomicAdd(next_group, 1u);
            const uint64_t bnd = gbegin[g + (lane & 1u)];
            const uint64_t p0 = __shfl_sync(0xffffffffu, bnd, 0), p1 = __shfl_sync(0xffffffffu, bnd, 1);
            const int4 ct = gtiles[g];
            for (uint64_t pb = p0; pb < p1; pb += 32) {
                const uint4 mine = (pb + lane < p1) ? gops[pb + lane] : make_uint4(0u, 0u, 0u, 0u);
                const int cnt = (int)((p1 - pb) < 32 ? (p1 - pb) : 32);
                for (int j = 0; j < cnt; ++j) {
                    // this super-product's four tiles: lane l (0..3) takes tile l = {A row 0, A row 1, B col 0, B col 1}
                    const uint32_t tx = __shfl_sync(0xffffffffu, mine.x, j), ty = __shfl_sync(0xffffffffu, mine.y, j);
                    const uint32_t tz = __shfl_sync(0xffffffffu, mine.z, j), tw = __shfl_sync(0xffffffffu, mine.w, j);
                    const uint32_t my_tile = lane == 0 ? tx : (lane == 1 ? ty : (lane == 2 ? tz : tw));
#pragma unroll 1
                    for (int half = 0; half < 2; ++half, ++it) {
                        const uint32_t s = it % NST, ph = (it / NST) & 1u;
                        const uint32_t fb = smem_u32(&hd->full_raw[s]);
                        if (lane == 0) {
                            mbar_wait(smem_u32(&hd->empty[s]), ph ^ 1u);
                            hd->ring_tiles[it & 15u] = ct;
                            hd->ring_flags[it & 15u] = ((pb + j == p0 && half == 0) ? 1 : 0) | ((pb + j + 1 == p1 && half == 1) ? 2 : 0);
                            mbar_arrive_expect_tx(fb, 2u * Cfg::STACK);
                        }
                        __syncwarp();
                        if (lane < 4) {
                            const bool is_a = lane < 2;
                            const bool kmajor = is_a ? TA : !TB;
                            const CUtensorMap* map = my_tile != P32_NONE ? (is_a ? &mapA : &mapB) : (is_a ? &mapZa : &mapZb);
                            const int tcol = my_tile != P32_NONE ? (int)my_tile * BS : 0;
                            const int k0 = half * KC;
                            // hi stack of the operand; inside it tile (lane & 1) is rows / chunks [64 (lane & 1), 64 (lane & 1) + 64)
                            const uint32_t dst = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES) + (is_a ? 0u : 2u * Cfg::STACK);
                            if (kmajor) {   // [mn][32 k] rows of 128 B: one box {32 k, 64 mn}
                                tma_box_g2s(dst + (lane & 1u) * (64 * 128), map, k0, tcol, fb);
                            } else {        // 32-mn chunks of [32 k][32 mn]: two boxes {32 mn, 32 k}
                                tma_box_g2s(dst + (2 * (lane & 1u) + 0) * (KC * 128), map, 0, tcol + k0, fb);
                                tma_box_g2s(dst + (2 * (lane & 1u) + 1) * (KC * 128), map, 32, tcol + k0, fb);
                            }
                        }
                        __syncwarp();
                    }
                }
            }
        }
        if (lane == 0) {
            for (int e = 0; e < Cfg::CVT_GROUPS; ++e, ++it) {
                const uint32_t s = it % NST, ph = (it / NST) & 1u;
                mbar_wait(smem_u32(&hd->empty[s]), ph ^ 1u);
                hd->ring_flags[it & 15u] = 4;
                mbar_arrive(smem_u32(&hd->full_raw[s]));
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: per K-step one N = 256 MMA (hi rows x all of B) and one N = 128 MMA (lo rows x B_hi) =====
        if (lane == 0) {
            constexpr uint32_t IDESC_BASE = (1u << 4) | (2u << 7) | (2u << 10) | ((TA ? 0u : 1u) << 15) | ((TB ? 1u : 0u) << 16) | ((uint32_t)(128 >> 4) << 24);
            constexpr uint32_t IDESC1 = IDESC_BASE | ((uint32_t)(256 >> 3) << 17), IDESC2 = IDESC_BASE | ((uint32_t)(128 >> 3) << 17);
            constexpr uint32_t CHUNK = KC * 128;
            constexpr uint32_t A_LBO = TA ? 16 : CHUNK, B_LBO = TB ? CHUNK : 16;
            constexpr uint32_t A_SBO = TA ? 1024 : 512, B_SBO = TB ? 512 : 1024;
            constexpr uint32_t A_LT = TA ? 2 : 1, B_LT = TB ? 1 : 2;
            for (uint32_t it = 0;; ++it) {
                const uint32_t s = it % NST, ph = (it / NST) & 1u;
                mbar_wait(smem_u32(&hd->full_cvt[s]), ph);
                const int flags = hd->ring_flags[it & 15u];
                const uint32_t chain = it >> 1, as = chain % Cfg::NSETS;
                const bool second = (it & 1u) != 0;
                if (!second || (flags & 4)) mbar_wait(smem_u32(&hd->tmem_empty[as]), ((chain / Cfg::NSETS) & 1u) ^ 1u);
                if (flags & 4) {   // (always at an even stage: super-products are two stages)
                    mbar_arrive(smem_u32(&hd->tmem_full[as]));
                    break;
                }
                tc_fence_after();
                const uint32_t d = tmem_base + as * 256;
                const uint32_t s0 = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES);
                const uint64_t dah = umma_desc(s0, A_LBO, A_SBO, A_LT), dal = umma_desc(s0 + Cfg::STACK, A_LBO, A_SBO, A_LT);
                const uint64_t dbh = umma_desc(s0 + 2 * Cfg::STACK, B_LBO, B_SBO, B_LT);
#pragma unroll
                for (int ks = 0; ks < Cfg::KSTEPS; ++ks) {
                    const uint64_t ao = (uint64_t)((TA ? ks * 32 : ks * 1024) >> 4), bo = (uint64_t)((TB ? ks * 1024 : ks * 32) >> 4);
                    mma_tf32(d, dah + ao, dbh + bo, IDESC1, (ks || second) ? 1u : 0u);   // hi x [B_hi | B_lo]
                    mma_tf32(d, dal + ao, dbh + bo, IDESC2, 1u);                          // lo x B_hi, into the hi*hi columns
                }
                tc_commit(smem_u32(&hd->empty[s]));
                if (second) tc_commit(smem_u32(&hd->tmem_full[as]));
            }
        }
    } else if (warp >= 2 && warp < 2 + Cfg::CVT_WARPS) {
        // ===== lo stacks from the raw (= hi) stacks =====
        const unsigned tid = ((warp - 2) % Cfg::CVT_WPG) * 32 + lane;
        for (uint32_t it = (warp - 2) / Cfg::CVT_WPG;; it += Cfg::CVT_GROUPS) {
            const uint32_t s = it % NST, ph = (it / NST) & 1u;
            mbar_wait(smem_u32(&hd->full_raw[s]), ph);
            const int flags = hd->ring_flags[it & 15u];
            if (!(flags & 4)) {
                unsigned char* st = stages + (size_t)s * Cfg::STAGE_BYTES;
#pragma unroll
                for (int op = 0; op < 2; ++op) {
                    const float4* hi = reinterpret_cast<const float4*>(st + op * 2 * Cfg::STACK);
                    float4* lo = reinterpret_cast<float4*>(st + op * 2 * Cfg::STACK + Cfg::STACK);
#pragma unroll 4
                    for (int i = (int)tid; i < Cfg::STACK / 16; i += Cfg::CVT_WPG * 32) {
                        const float4 x = hi[i];
                        float4 l;
                        l.x = x.x - __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u);
                        l.y = x.y - __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u);
                        l.z = x.z - __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u);
                        l.w = x.w - __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u);
                        lo[i] = l;
                    }
                }
                fence_proxy_async();
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&hd->full_cvt[s]));
            if (flags & 4) break;
        }
    } else if (warp >= 8 && (warp - 8) < Cfg::EPI_WARPS) {
        // ===== epilogue: warp (q, c): TMEM lanes [32q, 32q + 32) = rows 32 (q & 1) + lane of member row r = q >> 1; member column c =====
        const unsigned q = (warp - 8) & 3, c = (warp - 8) >> 2;
        const unsigned member = 2 * c + (q >> 1);
        const int crow = (int)((q & 1u) * 32 + lane);
        float acc[64];
        uint32_t it_e = 0;
        for (uint32_t pc = 0;; ++pc) {
            const uint32_t as = pc % Cfg::NSETS;
            mbar_wait(smem_u32(&hd->tmem_full[as]), (pc / Cfg::NSETS) & 1u);
            const int f0 = hd->ring_flags[it_e & 15u];
            if (f0 & 4) break;
            const int flags = (f0 | hd->ring_flags[(it_e + 1) & 15u]) & 3;
            const int4 tiles = hd->ring_tiles[it_e & 15u];
            it_e += 2;
            tc_fence_after();
            const uint32_t tbase = tmem_base + ((q * 32u) << 16) + as * 256;
#pragma unroll
            for (int hcol = 0; hcol < 2; ++hcol) {   // (one 32-column load in flight at a time: 64 accumulators + 32 loaded values per lane)
                uint32_t r[32];
                tmem_ld32(tbase + 128 + c * 64 + hcol * 32, r);    // x_hi * Bc_lo
                tmem_ld_wait();
                if (flags & 1) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[hcol * 32 + j] = __uint_as_float(r[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[hcol * 32 + j] = __fadd_rn(acc[hcol * 32 + j], __uint_as_float(r[j]));
                }
                tmem_ld32(tbase + c * 64 + hcol * 32, r);          // x_hi * Bc_hi + x_lo * Bc_hi
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[hcol * 32 + j] = __fadd_rn(acc[hcol * 32 + j], __uint_as_float(r[j]));
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&hd->tmem_empty[as]));
            if (flags & 2) {
                const int ctile = member == 0 ? tiles.x : (member == 1 ? tiles.y : (member == 2 ? tiles.z : tiles.w));
                if (ctile >= 0) {
                    float* C = Ct + (size_t)ctile * BS * BS + crow;
#pragma unroll
                    for (int j = 0; j < 64; ++j) C[(size_t)j * BS] = acc[j];
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (warp == 1) tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
}

template <bool TA, bool TB>
void launch_g64_inst(const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, const uint64_t* ckeys, const uint32_t* task_k,
                     const uint32_t* tile_list, uint32_t n_ctiles, size_t n_products, float* Ct) {
    using Cfg = G64Cfg;
    CUtensorMap mapA, mapB, mapZa, mapZb;
    // K-major operand (k along leaf rows): box {32 k, 64 mn};  MN-major: box {32 mn, 32 k}
    make_f32_map(&mapA, A.tiles.p, A.L, 64, 32, TA ? 64 : 32, !TA);
    make_f32_map(&mapB, B.tiles.p, B.n_ext(), 64, 32, TB ? 32 : 64, TB);
    make_f32_map(&mapZa, zero_leaf_f32_64(), 1, 64, 32, TA ? 64 : 32, !TA);
    make_f32_map(&mapZb, zero_leaf_f32_64(), 1, 64, 32, TB ? 32 : 64, TB);
    DevBuf<uint32_t> head(n_ctiles), cnt(n_ctiles);
    DevBuf<uint64_t> gpos((size_t)n_ctiles + 1), gbegin((size_t)n_ctiles + 1);
    DevBuf<int4> gtiles(n_ctiles);
    DevBuf<uint4> gops(std::max<size_t>(n_products, 1));
    cnt.zero();
    const unsigned gb = (n_ctiles + 255) / 256;
    HB_LAUNCH(k_g32_heads, gb, 256, 0, ckeys, tile_list, n_ctiles, head.p);
    exclusive_scan_u32(head.p, gpos.p, n_ctiles);
    HB_LAUNCH((k_g32_merge<false>), gb, 256, 0, ckeys, tile_list, n_ctiles, head.p, gpos.p, begin, ab, task_k, cnt.p, (const uint64_t*)nullptr,
              (int4*)nullptr, (uint4*)nullptr);
    exclusive_scan_u32(cnt.p, gbegin.p, n_ctiles);
    HB_LAUNCH((k_g32_merge<true>), gb, 256, 0, ckeys, tile_list, n_ctiles, head.p, gpos.p, begin, ab, task_k, (uint32_t*)nullptr, gbegin.p, gtiles.p,
              gops.p);
    DevBuf<unsigned> counter(1);
    counter.zero();
    auto kfn = k_gemm_f32_g64<TA, TB>;
    static bool configured = false;
    if (!configured) {
        HB_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        configured = true;
    }
    const unsigned grid = std::min<unsigned>(n_ctiles, (unsigned)engine().sm_count);
    HB_LAUNCH(kfn, grid, Cfg::THREADS, Cfg::SMEM_BYTES, mapA, mapB, mapZa, mapZb, gops.p, gbegin.p, gtiles.p, gpos.p + n_ctiles, counter.p, Ct);
}

void launch_g64(bool tA, bool tB, const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, const uint64_t* ckeys,
                const uint32_t* task_k, const uint32_t* tile_list, uint32_t n, size_t n_products, float* Ct) {
    if (!tA && !tB) launch_g64_inst<false, false>(A, B, ab, begin, ckeys, task_k, tile_list, n, n_products, Ct);
    else if (!tA && tB) launch_g64_inst<false, true>(A, B, ab, begin, ckeys, task_k, tile_list, n, n_products, Ct);
    else if (tA && !tB) launch_g64_inst<true, false>(A, B, ab, begin, ckeys, task_k, tile_list, n, n_products, Ct);
    else launch_g64_inst<true, true>(A, B, ab, begin, ckeys, task_k, tile_list, n, n_products, Ct);
}

template <int LS, int BS, bool TA, bool TB>
void launch_inst(const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, uint32_t n_ctiles,
                 const uint32_t* tile_list, unsigned* counter, float* Ct) {
    using Cfg = F32Cfg<BS>;
    CUtensorMap mapA, mapB;
    // K-major operand (k along leaf rows): box {32 k, BS mn};  MN-major: box {32 mn, KC k}
    make_f32_map(&mapA, A.tiles.p, A.L, LS, 32, TA ? BS : Cfg::KC, !TA);
    make_f32_map(&mapB, B.tiles.p, B.n_ext(), LS, 32, TB ? Cfg::KC : BS, TB);
    auto kfn = k_gemm_f32_tc<LS, BS, TA, TB>;
    static bool configured = false;
    if (!configured) {
        HB_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        configured = true;
    }
    const uint64_t units = (uint64_t)n_ctiles * (LS / BS) * (LS / BS);
    if (units >= 0x7fffffffull) throw Error(HBSM_E_CUDA, "hbsm_b200: too many C sub-tiles for one fp32 leaf-GEMM launch");
    unsigned grid = (unsigned)std::min<uint64_t>(units, (uint64_t)engine().sm_count);
    HB_LAUNCH(kfn, grid, Cfg::THREADS, Cfg::SMEM_BYTES, mapA, mapB, ab, begin, n_ctiles, tile_list, counter, Ct);
}

template <int LS, int BS>
void launch_bs(bool tA, bool tB, const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, uint32_t n,
               const uint32_t* tile_list, unsigned* counter, float* Ct) {
    if (!tA && !tB) launch_inst<LS, BS, false, false>(A, B, ab, begin, n, tile_list, counter, Ct);
    else if (!tA && tB) launch_inst<LS, BS, false, true>(A, B, ab, begin, n, tile_list, counter, Ct);
    else if (tA && !tB) launch_inst<LS, BS, true, false>(A, B, ab, begin, n, tile_list, counter, Ct);
    else launch_inst<LS, BS, true, true>(A, B, ab, begin, n, tile_list, counter, Ct);
}

template <int BS, bool TA, bool TB>
void launch_q4_inst(const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, uint32_t n_ctiles,
                    const uint32_t* tile_list, unsigned* counter, float* Ct) {
    using Cfg = Q4Cfg<BS>;
    CUtensorMap mapA, mapB;
    make_f32_map(&mapA, A.tiles.p, A.L, BS, 32, BS, !TA);
    make_f32_map(&mapB, B.tiles.p, B.n_ext(), BS, 32, BS, TB);
    auto kfn = k_gemm_f32_q4<BS, TA, TB>;
    static bool configured = false;
    if (!configured) {
        HB_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        configured = true;
    }
    unsigned grid = std::min<unsigned>(n_ctiles, (unsigned)engine().sm_count);
    HB_LAUNCH(kfn, grid, Cfg::THREADS, Cfg::SMEM_BYTES, mapA, mapB, ab, begin, n_ctiles, tile_list, counter, Ct);
}

template <int BS>
void launch_q4(bool tA, bool tB, const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, uint32_t n,
               const uint32_t* tile_list, unsigned* counter, float* Ct) {
    if (!tA && !tB) launch_q4_inst<BS, false, false>(A, B, ab, begin, n, tile_list, counter, Ct);
    else if (!tA && tB) launch_q4_inst<BS, false, true>(A, B, ab, begin, n, tile_list, counter, Ct);
    else if (tA && !tB) launch_q4_inst<BS, true, false>(A, B, ab, begin, n, tile_list, counter, Ct);
    else launch_q4_inst<BS, true, true>(A, B, ab, begin, n, tile_list, counter, Ct);
}

}  // namespace

void launch_gemm_f32_tc(const Matrix& A, bool tA, const Matrix& B, bool tB, const uint2* ab, const uint64_t* begin,
                        uint32_t n_ctiles, const uint32_t* tile_list, unsigned* counter, float* Ct, const uint64_t* ckeys,
                        const uint32_t* task_k, size_t n_products, bool single_tile) {
    switch (A.b) {
        case 32:
            if (single_tile) launch_q4<32>(tA, tB, A, B, ab, begin, n_ctiles, tile_list, counter, Ct);
            else launch_g32(tA, tB, A, B, ab, begin, ckeys, task_k, tile_list, n_ctiles, n_products, Ct);
            break;
        case 64:
            if (single_tile) launch_q4<64>(tA, tB, A, B, ab, begin, n_ctiles, tile_list, counter, Ct);
            else launch_g64(tA, tB, A, B, ab, begin, ckeys, task_k, tile_list, n_ctiles, n_products, Ct);
            break;
        case 128: launch_bs<128, 128>(tA, tB, A, B, ab, begin, n_ctiles, tile_list, counter, Ct); break;
        case 256: launch_bs<256, 128>(tA, tB, A, B, ab, begin, n_ctiles, tile_list, counter, Ct); break;
        default: throw Error(HBSM_E_ARG, "hbsm_b200: no fp32 tensor-core leaf kernel for this blocksize");
    }
}

}  // namespace hbsm_b200

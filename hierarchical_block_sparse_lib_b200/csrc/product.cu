// product.cu -- multiply / SpAMM on the flat block table.
//
// Replaces the reference's two phases (SURVEY 3.1):
//   symbolic  get_batches_multiply H:5478 / get_batches_spamm H:6291  -> task-list builder (count, scan, fill, sort by
//             (Morton key of the C tile, k), segment heads = C's block table)
//   numeric   multiply_batches H:7240 (+ BLAS gemm H:7273)            -> one persistent grouped leaf-GEMM kernel,
//             C-stationary (a CTA owns a C tile for its whole k-list, no atomics on data), A/B tiles staged by TMA tensor
//             copies into shared memory behind an mbarrier ring, FP64 DMMA (mma.sync m8n8k4) accumulation.
//
// Executed set (SURVEY 0.3, 9): exact = every (ci,k,cj) with both tiles present; SpAMM additionally requires
// fl(nsq(A_tile) * nsq(B_tile)) > fl(tau*tau) evaluated in Treal with a strict '>' (H:2008, H:6651).  The hierarchical
// test of the reference collapses to this flat leaf-pair rule because node norms are sums of non-negative child norms.
#include "matrix.cuh"
#include "gemm_common.cuh"
#include <chrono>

namespace hbsm_b200 {

namespace {

inline unsigned blocks_for(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// ---------------------------------------------------------------------------------------------------
// task-list builder
// ---------------------------------------------------------------------------------------------------
struct JoinArgs {
    const uint32_t* a_ptr; const uint32_t* a_other; const uint32_t* a_tile; uint32_t a_lines;   // op(A): line = ci, other = k
    const uint32_t* b_ptr; const uint32_t* b_other; const uint32_t* b_tile; uint32_t b_lines;   // op(B): line = k, other = cj
    const void* a_norms; const void* b_norms;
    int spamm; int upper_only;
    double tau2_d; float tau2_f;
    size_t a_entries;      // number of op(A) entries joined by this launch ...
    size_t a_entry_lo;     // ... starting at this entry of the line index (a block-row range of C; 0 = all of op(A))
};

template <typename T> __device__ __forceinline__ bool spamm_keep(T na, T nb, const JoinArgs& g);
template <> __device__ __forceinline__ bool spamm_keep<double>(double na, double nb, const JoinArgs& g) {
    return __dmul_rn(na, nb) > g.tau2_d;
}
template <> __device__ __forceinline__ bool spamm_keep<float>(float na, float nb, const JoinArgs& g) {
    return __fmul_rn(na, nb) > g.tau2_f;
}

// one warp per tile of op(A): walks row k of op(B).  FILL=false counts survivors, FILL=true writes them.
template <typename T, bool FILL>
__global__ void __launch_bounds__(256) k_join(JoinArgs g, const uint32_t* __restrict__ a_line_of_entry,
                                               uint32_t* __restrict__ counts, const uint64_t* __restrict__ offsets,
                                               int kbits, uint64_t* __restrict__ keys, uint32_t* __restrict__ pa,
                                               uint32_t* __restrict__ pb, unsigned long long* __restrict__ n_cand) {
    const unsigned lane = threadIdx.x & 31;
    const size_t w = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // counts / offsets are indexed by w
    if (w >= g.a_entries) return;
    const size_t e = g.a_entry_lo + w;
    const uint32_t ci = a_line_of_entry[e];
    const uint32_t k = g.a_other[e];
    const uint32_t ta = g.a_tile[e];
    uint32_t beg = 0, end = 0;
    if (k < g.b_lines) { beg = g.b_ptr[k]; end = g.b_ptr[k + 1]; }
    T na = g.spamm ? reinterpret_cast<const T*>(g.a_norms)[ta] : (T)0;
    uint32_t total = 0;
    uint64_t base = FILL ? offsets[w] : 0;
    for (uint32_t f0 = beg; f0 < end; f0 += 32) {
        uint32_t f = f0 + lane;
        bool keep = false;
        uint32_t cj = 0, tb = 0;
        if (f < end) {
            cj = g.b_other[f];
            tb = g.b_tile[f];
            keep = true;
            if (g.spamm) keep = spamm_keep<T>(na, reinterpret_cast<const T*>(g.b_norms)[tb], g);
            if (g.upper_only && ci > cj) keep = false;
        }
        unsigned bal = __ballot_sync(0xffffffffu, keep);
        if (FILL && keep) {
            uint64_t p = base + total + __popc(bal & ((1u << lane) - 1u));
            keys[p] = (morton_encode(ci, cj) << kbits) | (uint64_t)k;
            pa[p] = ta;
            pb[p] = tb;
        }
        total += __popc(bal);
    }
    if (!FILL && lane == 0) {
        counts[w] = total;
        if (n_cand && end > beg) atomicAdd(n_cand, (unsigned long long)(end - beg));
    }
}

// line number of every entry of a line index (inverse of ptr)
__global__ void k_entry_lines(const uint32_t* __restrict__ ptr, uint32_t n_lines, uint32_t* __restrict__ line_of) {
    uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_lines) return;
    for (uint32_t e = ptr[l]; e < ptr[l + 1]; ++e) line_of[e] = l;
}

__global__ void k_row_counts(const uint32_t* __restrict__ ptr, uint32_t n_lines, const uint64_t* __restrict__ offs, size_t entry_lo,
                             size_t n_e, uint64_t* __restrict__ out) {
    const uint32_t l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= n_lines) return;
    const size_t a = min(max((size_t)ptr[l], entry_lo), entry_lo + n_e) - entry_lo;
    const size_t b = min(max((size_t)ptr[l + 1], entry_lo), entry_lo + n_e) - entry_lo;
    out[l] = offs[b] - offs[a];
}

__global__ void k_iota(uint32_t* __restrict__ v, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (uint32_t)i;
}

__global__ void k_task_heads(const uint64_t* __restrict__ keys, size_t n, int kbits, uint32_t* __restrict__ head) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    head[i] = (i == 0 || (keys[i - 1] >> kbits) != (keys[i] >> kbits)) ? 1u : 0u;
}

// sorted keys -> C block table, segment starts, gathered operand indices, k per task
__global__ void k_task_finish(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ perm, size_t n, int kbits,
                              const uint32_t* __restrict__ head, const uint64_t* __restrict__ pos,
                              const uint32_t* __restrict__ pa, const uint32_t* __restrict__ pb,
                              uint64_t* __restrict__ ckeys, uint64_t* __restrict__ begin, uint2* __restrict__ ab,
                              uint32_t* __restrict__ task_k, size_t n_ctiles) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t key = keys[i];
    if (head[i]) { ckeys[pos[i]] = key >> kbits; begin[pos[i]] = i; }
    uint32_t src = perm[i];
    ab[i] = make_uint2(pa[src], pb[src]);
    task_k[i] = (uint32_t)(key & ((1ull << kbits) - 1ull));
    if (i == n - 1) begin[n_ctiles] = n;
}

// ---------------------------------------------------------------------------------------------------
// generic leaf GEMM (any blocksize, both dtypes): one CTA per C tile, plain FMA from global/L2.  Used for the
// blocksizes without a tensor-pipe kernel and as the debug/parity variant (hbsm_set_gemm_variant(1)).
// ---------------------------------------------------------------------------------------------------
template <typename T, bool ACC>
__global__ void __launch_bounds__(256) k_gemm_generic(const T* __restrict__ At, const T* __restrict__ Bt,
                                                       const uint2* __restrict__ ab, const uint64_t* __restrict__ begin,
                                                       const uint32_t* __restrict__ tile_list, int b, int tA, int tB,
                                                       T* __restrict__ Ct, AccEpi<T> epi) {
    const size_t bb = (size_t)b * b;
    const size_t ctile = tile_list ? tile_list[blockIdx.x] : blockIdx.x;   // optional indirection: a subset of C's tiles
    const uint64_t p0 = begin[ctile], p1 = begin[ctile + 1];
    T* C = Ct + ctile * bb;
    const T* O = nullptr;
    if constexpr (ACC) O = epi.old_at(ctile, bb, 0);
    for (size_t idx = threadIdx.x; idx < bb; idx += blockDim.x) {
        const int i = (int)(idx % b), j = (int)(idx / b);
        T acc = 0;
        for (uint64_t p = p0; p < p1; ++p) {
            const T* A = At + (size_t)ab[p].x * bb;
            const T* B = Bt + (size_t)ab[p].y * bb;
            for (int l = 0; l < b; ++l) {
                T a = tA ? A[(size_t)i * b + l] : A[(size_t)l * b + i];
                T bv = tB ? B[(size_t)l * b + j] : B[(size_t)j * b + l];
                acc = fma(a, bv, acc);
            }
        }
        if constexpr (ACC) C[idx] = epi.apply(acc, O, idx);
        else C[idx] = acc;
    }
}

// ---------------------------------------------------------------------------------------------------
// FP64 leaf GEMM: persistent, warp-specialised, one cp.async.bulk.tensor per operand chunk + mbarrier ring + DMMA.
//
// A leaf (column-major, ld = BS) is described to TMA as the 4-D tensor  [tile][r/4][c][r%4]  (innermost last), i.e.
//   dim0 = r % 4 (stride 8 B), dim1 = c (stride BS*8 B), dim2 = r / 4 (stride 32 B), dim3 = tile (stride BS*BS*8 B).
// A box {4, NC, NR4, 1} therefore lands in shared memory as  smem[(r/4)][c][r%4]: every group of 4 consecutive rows
// of 4 consecutive columns is 16 consecutive doubles = 128 contiguous bytes.  A DMMA m8n8k4 fragment is exactly
// "4 consecutive indices along one leaf axis x 4 along the other" per half-warp, for the plain AND the transposed
// operand, so every fragment load is one conflict-free 128-byte wavefront per half-warp -- no padding, no swizzle,
// and a whole operand chunk is ONE TMA instruction issued by one thread.
//   k along leaf columns (A as is, B transposed): box {4, KC, BS/4}, element (x, k) at  x%4 + 4*k + 4*KC*(x/4)
//   k along leaf rows    (A transposed, B as is): box {4, BS, KC/4}, element (x, k) at  k%4 + 4*x + 4*BS*(k/4)
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_tile_g2s(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                             uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
        ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
        : "memory");
}

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

template <int BS, int KC>
struct TmaCfg {
    static constexpr int CHUNK_ELEMS = BS * KC;
    static constexpr int STAGE_BYTES = 2 * CHUNK_ELEMS * 8;
    static constexpr int NCHUNK = BS / KC;
    static constexpr int SMEM_BUDGET = 216 * 1024;
    static constexpr int NST_RAW = SMEM_BUDGET / STAGE_BYTES;
    static constexpr int NST = NST_RAW > 8 ? 8 : NST_RAW;
    static constexpr int CONSUMER_WARPS = 8;
    static constexpr int THREADS = (CONSUMER_WARPS + 1) * 32;
    static constexpr int WM = BS / 2, WN = BS / 4;
    static constexpr int MB = WM / 8, NB = WN / 8;
    static constexpr int HEADER_BYTES = 1024;
    static constexpr int SMEM_BYTES = HEADER_BYTES + NST * STAGE_BYTES + 1024;   // +1024: manual 1 KiB alignment
    static_assert(NST >= 2, "pipeline needs two stages");
};

// LS = leaf size, BS = compute tile of one CTA (BS == LS up to 128; a 256-leaf is 2 x 2 sub-tiles addressed in place)
template <int LS, int BS, int KC, bool TA, bool TB, bool ACC>
__global__ void __launch_bounds__(TmaCfg<BS, KC>::THREADS, 1)
k_gemm_f64_tma(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
               const uint2* __restrict__ ab, const uint64_t* __restrict__ begin, uint32_t n_ctiles,
               const uint32_t* __restrict__ tile_list, unsigned* __restrict__ next_tile, double* __restrict__ Ct,
               AccEpi<double> epi) {
    using Cfg = TmaCfg<BS, KC>;
    constexpr int NST = Cfg::NST;
    constexpr int S = LS / BS;
    static_assert(LS % BS == 0 && (S == 1 || S == 2), "leaf / compute-tile shapes");
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem);
    uint64_t* empty_bar = full_bar + NST;
    GemmMeta* meta = reinterpret_cast<GemmMeta*>(empty_bar + NST);
    unsigned char* stages = smem + Cfg::HEADER_BYTES;
    const unsigned warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; ++s) {
            mbar_init(smem_u32(&full_bar[s]), 1);
            mbar_init(smem_u32(&empty_bar[s]), Cfg::CONSUMER_WARPS);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == Cfg::CONSUMER_WARPS) {
        // ===== producer: the warp walks the task list together -- the next work unit is claimed one unit ahead and 32
        // (A tile, B tile) pairs arrive per coalesced load, so no index fetch latency sits between two TMA issues (at
        // 32-leaves a product lasts ~500 clk, less than one dependent L2 round trip) -- and lane 0 issues the copies =====
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&mapB) : "memory");
        }
        uint32_t it = 0;
        const unsigned n_units = n_ctiles * (unsigned)(S * S);
        unsigned claimed = 0;
        if (lane == 0) claimed = atomicAdd(next_tile, 1u);       // work unit = (C tile, sub-tile)
        for (;;) {
            const unsigned unit = __shfl_sync(0xffffffffu, claimed, 0);
            if (unit >= n_units) break;
            if (lane == 0) claimed = atomicAdd(next_tile, 1u);   // consumed at the top of the next round
            const unsigned sub = unit % (S * S);
            const unsigned tile = tile_list ? tile_list[unit / (S * S)] : unit / (S * S);
            const int cunit = (int)(tile * (S * S) + sub);
            const int si = (int)(sub % S) * BS, sj = (int)(sub / S) * BS;
            const uint64_t bnd = begin[tile + (lane & 1u)];
            const uint64_t p0 = __shfl_sync(0xffffffffu, bnd, 0), p1 = __shfl_sync(0xffffffffu, bnd, 1);
            for (uint64_t pb = p0; pb < p1; pb += 32) {
                const uint2 mine = (pb + lane < p1) ? ab[pb + lane] : make_uint2(0u, 0u);
                const int cnt = (int)((p1 - pb) < 32 ? (p1 - pb) : 32);
                for (int j = 0; j < cnt; ++j) {
                    uint2 t;
                    t.x = __shfl_sync(0xffffffffu, mine.x, j);
                    t.y = __shfl_sync(0xffffffffu, mine.y, j);
                    if (lane == 0) {
                        const uint64_t p = pb + j;
#pragma unroll 1
                        for (int kc = 0; kc < S * Cfg::NCHUNK; ++kc, ++it) {
                            const uint32_t s = it % NST, ph = (it / NST) & 1u;
                            mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1u);
                            const uint32_t fb = smem_u32(&full_bar[s]);
                            int fl = 0;
                            if (p == p0 && kc == 0) fl |= 1;
                            if (p + 1 == p1 && kc == S * Cfg::NCHUNK - 1) fl |= 2;
                            meta[s].ctile = cunit;
                            meta[s].flags = fl;
                            mbar_arrive_expect_tx(fb, Cfg::STAGE_BYTES);
                            const uint32_t sa = smem_u32(stages + (size_t)s * Cfg::STAGE_BYTES);
                            const uint32_t sb = sa + Cfg::CHUNK_ELEMS * 8;
                            const int k0 = kc * KC;   // position along the leaf's full contraction dimension
                            if (TA) tma_tile_g2s(sa, &mapA, 0, si, k0 / 4, (int)t.x, fb);   // k along leaf rows
                            else    tma_tile_g2s(sa, &mapA, 0, k0, si / 4, (int)t.x, fb);   // k along leaf columns
                            if (TB) tma_tile_g2s(sb, &mapB, 0, k0, sj / 4, (int)t.y, fb);
                            else    tma_tile_g2s(sb, &mapB, 0, sj, k0 / 4, (int)t.y, fb);
                        }
                    }
                    __syncwarp();
                }
            }
        }
        if (lane == 0) {
            const uint32_t s = it % NST, ph = (it / NST) & 1u;
            mbar_wait(smem_u32(&empty_bar[s]), ph ^ 1u);
            meta[s].ctile = -1;
            meta[s].flags = 4;
            mbar_arrive(smem_u32(&full_bar[s]));
        }
        return;
    }

    // ===== consumers: 2 x 4 warp grid, DMMA m8n8k4, accumulators in registers =====
    const int wm0 = (int)(warp >> 2) * Cfg::WM, wn0 = (int)(warp & 3) * Cfg::WN;
    const int g = (int)(lane >> 2), t = (int)(lane & 3);
    double acc[Cfg::MB][Cfg::NB][2];
    // A: x = row of op(A) = wm0 + 8*mb + g ; B: x = column of op(B) = wn0 + 8*nb + g ; k = 4*ks + t
    const int a_off = TA ? (t + 4 * (wm0 + g)) : ((g & 3) + 4 * t + 4 * KC * ((wm0 >> 2) + (g >> 2)));
    const int b_off = TB ? ((g & 3) + 4 * t + 4 * KC * ((wn0 >> 2) + (g >> 2))) : (t + 4 * (wn0 + g));
    constexpr int A_BLK = TA ? 32 : 8 * KC;
    constexpr int A_KS = TA ? 4 * BS : 16;
    constexpr int B_BLK = TB ? 8 * KC : 32;
    constexpr int B_KS = TB ? 16 : 4 * BS;
    uint32_t it = 0;
    for (;; ++it) {
        const uint32_t s = it % NST, ph = (it / NST) & 1u;
        mbar_wait(smem_u32(&full_bar[s]), ph);
        const GemmMeta m = meta[s];
        if (m.flags & 4) break;
        if (m.flags & 1) {
#pragma unroll
            for (int i = 0; i < Cfg::MB; ++i)
#pragma unroll
                for (int j = 0; j < Cfg::NB; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
        }
        const double* As = reinterpret_cast<const double*>(stages + (size_t)s * Cfg::STAGE_BYTES) + a_off;
        const double* Bs = reinterpret_cast<const double*>(stages + (size_t)s * Cfg::STAGE_BYTES) + Cfg::CHUNK_ELEMS + b_off;
#pragma unroll
        for (int ks = 0; ks < KC / 4; ++ks) {
            double a[Cfg::MB], b[Cfg::NB];
#pragma unroll
            for (int i = 0; i < Cfg::MB; ++i) a[i] = As[i * A_BLK + ks * A_KS];
#pragma unroll
            for (int j = 0; j < Cfg::NB; ++j) b[j] = Bs[j * B_BLK + ks * B_KS];
#pragma unroll
            for (int i = 0; i < Cfg::MB; ++i)
#pragma unroll
                for (int j = 0; j < Cfg::NB; ++j) dmma884(acc[i][j][0], acc[i][j][1], a[i], b[j]);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&empty_bar[s]));
        if (m.flags & 2) {
            const unsigned tile = (unsigned)m.ctile / (S * S), sub = (unsigned)m.ctile % (S * S);
            double* C = Ct + (size_t)tile * LS * LS + (size_t)((sub / S) * BS) * LS + (sub % S) * BS;
            const double* O = nullptr;
            if constexpr (ACC) O = epi.old_at(tile, (size_t)LS * LS, (size_t)((sub / S) * BS) * LS + (sub % S) * BS);
#pragma unroll
            for (int i = 0; i < Cfg::MB; ++i)
#pragma unroll
                for (int j = 0; j < Cfg::NB; ++j) {
                    const int row = wm0 + i * 8 + g, col = wn0 + j * 8 + 2 * t;
                    if constexpr (ACC) {   // the old values in the store's own pattern
                        C[(size_t)col * LS + row] = epi.apply(acc[i][j][0], O, (size_t)col * LS + row);
                        C[(size_t)(col + 1) * LS + row] = epi.apply(acc[i][j][1], O, (size_t)(col + 1) * LS + row);
                    } else {
                        C[(size_t)col * LS + row] = acc[i][j][0];
                        C[(size_t)(col + 1) * LS + row] = acc[i][j][1];
                    }
                }
        }
    }
}

// tensor map of a tile pool in the interleaved-by-4-rows view; k_rows: the K-chunk runs along leaf rows
void make_tile_map(CUtensorMap* map, const void* tiles, size_t n_tiles, int LS, int BS, int KC, bool k_rows, int esize,
                   CUtensorMapDataType dt) {
    EncodeTiledFn enc = encode_tiled_fn();
    const int grp = 32 / esize;   // rows per 32-byte group (4 doubles / 8 floats)
    cuuint64_t gdim[4] = {(cuuint64_t)grp, (cuuint64_t)LS, (cuuint64_t)(LS / grp), (cuuint64_t)n_tiles};
    cuuint64_t gstr[3] = {(cuuint64_t)LS * esize, 32ull, (cuuint64_t)LS * LS * esize};
    cuuint32_t box[4] = {(cuuint32_t)grp, (cuuint32_t)(k_rows ? BS : KC), (cuuint32_t)(k_rows ? KC / grp : BS / grp), 1u};
    cuuint32_t estr[4] = {1, 1, 1, 1};
    if (!enc || enc(map, dt, 4, const_cast<void*>(tiles), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        throw Error(HBSM_E_CUDA, "hbsm_b200: the driver refused the tensor map of an fp64 leaf operand");
}

template <int LS, int BS, int KC, bool TA, bool TB, bool ACC>
void launch_gemm_f64_tma_inst(const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin, uint32_t n_ctiles,
                              const uint32_t* tile_list, unsigned* counter, double* Ct, const AccEpi<double>& epi) {
    using Cfg = TmaCfg<BS, KC>;
    CUtensorMap mapA, mapB;
    make_tile_map(&mapA, A.tiles.p, A.L, LS, BS, KC, TA, 8, CU_TENSOR_MAP_DATA_TYPE_FLOAT64);
    make_tile_map(&mapB, B.tiles.p, B.n_ext(), LS, BS, KC, !TB, 8, CU_TENSOR_MAP_DATA_TYPE_FLOAT64);
    auto kfn = k_gemm_f64_tma<LS, BS, KC, TA, TB, ACC>;
    static bool configured = false;
    if (!configured) {
        HB_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
        configured = true;
    }
    const uint64_t units = (uint64_t)n_ctiles * (LS / BS) * (LS / BS);
    if (units >= 0x7fffffffull) throw Error(HBSM_E_CUDA, "hbsm_b200: too many C sub-tiles for one fp64 leaf-GEMM launch");
    unsigned grid = (unsigned)std::min<uint64_t>(units, (uint64_t)engine().sm_count);
    HB_LAUNCH(kfn, grid, Cfg::THREADS, Cfg::SMEM_BYTES, mapA, mapB, ab, begin, n_ctiles, tile_list, counter, Ct, epi);
}

template <int LS, int BS, int KC, bool ACC>
void launch_gemm_f64_tma(bool tA, bool tB, const Matrix& A, const Matrix& B, const uint2* ab, const uint64_t* begin,
                         uint32_t n_ctiles, const uint32_t* tile_list, unsigned* counter, double* Ct, const AccEpi<double>& e) {
    if (!tA && !tB) launch_gemm_f64_tma_inst<LS, BS, KC, false, false, ACC>(A, B, ab, begin, n_ctiles, tile_list, counter, Ct, e);
    else if (!tA && tB) launch_gemm_f64_tma_inst<LS, BS, KC, false, true, ACC>(A, B, ab, begin, n_ctiles, tile_list, counter, Ct, e);
    else if (tA && !tB) launch_gemm_f64_tma_inst<LS, BS, KC, true, false, ACC>(A, B, ab, begin, n_ctiles, tile_list, counter, Ct, e);
    else launch_gemm_f64_tma_inst<LS, BS, KC, true, true, ACC>(A, B, ab, begin, n_ctiles, tile_list, counter, Ct, e);
}

struct TaskList {
    size_t n_products = 0, n_ctiles = 0;
    unsigned long long n_candidates = 0;
    DevBuf<uint64_t> ckeys;    // [n_ctiles] ascending Morton keys of C's tiles
    DevBuf<uint64_t> begin;    // [n_ctiles + 1]
    DevBuf<uint2> ab;          // [P] (A tile, B tile), grouped by C tile, k ascending inside a group
    DevBuf<uint32_t> task_k;   // [P]
};

// builds the executed-product list; returns with the stream synchronised
// entry_lo/entry_hi: range of op(A)'s line-index entries to join (= a block-row range of C), default all
// a_norms / b_norms: leaf norm^2 arrays to test against instead of the operands' cached ones (spamm(updated=false))
void build_tasks(const Matrix& A, bool tA, const Matrix& B, bool tB, const ProductOpts& o, int kbits, TaskList& tl,
                 bool count_only, size_t entry_lo = 0, size_t entry_hi = (size_t)-1, const void* a_norms = nullptr,
                 const void* b_norms = nullptr, uint64_t* d_row_counts = nullptr) {
    const LineIndex& la = line_index(A, tA);   // op(A): lines are C rows
    const LineIndex& lb = line_index(B, tB, true);   // op(B): lines are k; includes the halo tail if one is committed
    tl.n_products = tl.n_ctiles = 0;
    tl.n_candidates = 0;
    if (A.L == 0 || B.n_ext() == 0) return;
    entry_hi = std::min(entry_hi, A.L);
    if (entry_lo >= entry_hi) return;
    const size_t n_e = entry_hi - entry_lo;
    JoinArgs g{};
    g.a_ptr = la.ptr.p; g.a_other = la.other.p; g.a_tile = la.tile.p; g.a_lines = la.n_lines;
    g.b_ptr = lb.ptr.p; g.b_other = lb.other.p; g.b_tile = lb.tile.p; g.b_lines = lb.n_lines;
    g.a_norms = a_norms ? a_norms : A.norms.p; g.b_norms = b_norms ? b_norms : B.norms.p;
    g.spamm = o.spamm ? 1 : 0;
    g.upper_only = o.upper_only ? 1 : 0;
    g.tau2_d = o.tau * o.tau;                       // fl(tau*tau) in Treal, H:2008
    { float tf = (float)o.tau; g.tau2_f = tf * tf; }
    g.a_entries = n_e;
    g.a_entry_lo = entry_lo;
    DevBuf<uint32_t> line_of(A.L), counts(n_e);
    HB_LAUNCH(k_entry_lines, blocks_for(la.n_lines, 256), 256, 0, la.ptr.p, la.n_lines, line_of.p);
    DevBuf<unsigned long long> ncand(1);
    ncand.zero();
    const unsigned jgrid = blocks_for(n_e * 32, 256);
    if (A.dtype == HBSM_F64) {
        auto kfn = k_join<double, false>;
        HB_LAUNCH(kfn, jgrid, 256, 0, g, line_of.p, counts.p, (const uint64_t*)nullptr, kbits, (uint64_t*)nullptr,
                  (uint32_t*)nullptr, (uint32_t*)nullptr, ncand.p);
    } else {
        auto kfn = k_join<float, false>;
        HB_LAUNCH(kfn, jgrid, 256, 0, g, line_of.p, counts.p, (const uint64_t*)nullptr, kbits, (uint64_t*)nullptr,
                  (uint32_t*)nullptr, (uint32_t*)nullptr, ncand.p);
    }
    DevBuf<uint64_t> offs(n_e + 1);
    exclusive_scan_u32(counts.p, offs.p, n_e);
    if (d_row_counts)   // products per line of op(A) (= per C block row): differences of the scan at the line boundaries
        HB_LAUNCH(k_row_counts, blocks_for(la.n_lines, 256), 256, 0, la.ptr.p, la.n_lines, offs.p, entry_lo, n_e, d_row_counts);
    const auto pc = read_scalars(offs.p + n_e, (const uint64_t*)ncand.p);
    const uint64_t P = pc.first;
    tl.n_candidates = pc.second;
    tl.n_products = (size_t)P;
    if (P == 0 || count_only) return;
    if (P >= 0xffffffffull) throw Error(HBSM_E_ARG, "hbsm_b200: more than 2^32-1 leaf products in one call");
    DevBuf<uint64_t> keys(P);
    DevBuf<uint32_t> pa(P), pb(P), perm(P);
    if (A.dtype == HBSM_F64) {
        auto kfn = k_join<double, true>;
        HB_LAUNCH(kfn, jgrid, 256, 0, g, line_of.p, (uint32_t*)nullptr, offs.p, kbits, keys.p, pa.p, pb.p,
                  (unsigned long long*)nullptr);
    } else {
        auto kfn = k_join<float, true>;
        HB_LAUNCH(kfn, jgrid, 256, 0, g, line_of.p, (uint32_t*)nullptr, offs.p, kbits, keys.p, pa.p, pb.p,
                  (unsigned long long*)nullptr);
    }
    HB_LAUNCH(k_iota, blocks_for(P, 256), 256, 0, perm.p, (size_t)P);
    // Stable sort on the C-tile bits only: products are emitted per op(A) tile in (ci, k) order (the row index is sorted
    // by k inside a row), so inside one C tile they already appear with k ascending and a stable sort keeps that order.
    radix_sort_pairs_bits(keys.p, perm.p, P, kbits, 3 * kbits);
    DevBuf<uint32_t> head(P);
    HB_LAUNCH(k_task_heads, blocks_for(P, 256), 256, 0, keys.p, (size_t)P, kbits, head.p);
    DevBuf<uint64_t> pos(P + 1);
    exclusive_scan_u32(head.p, pos.p, P);
    const uint64_t nct = read_scalars(pos.p + P, nullptr).first;
    tl.n_ctiles = (size_t)nct;
    tl.ckeys.alloc(nct);
    tl.begin.alloc(nct + 1);
    tl.ab.alloc(P);
    tl.task_k.alloc(P);
    HB_LAUNCH(k_task_finish, blocks_for(P, 256), 256, 0, keys.p, perm.p, (size_t)P, kbits, head.p, pos.p, pa.p, pb.p,
              tl.ckeys.p, tl.begin.p, tl.ab.p, tl.task_k.p, (size_t)nct);
}

int coord_bits(const Matrix& A, const Matrix& B, int cm, int cn, int b) {
    int d = std::max(A.vdepth(), B.vdepth());
    d = std::max(d, Matrix::depth_for(cm, cn, b));
    return std::max(d, 1);
}

// accumulate: C may be sized, with the product's shape, dtype and leaf size
void check_operands(const Matrix& A, bool tA, const Matrix& B, bool tB, const Matrix& C, bool spamm, bool accumulate, int& AM, int& BN) {
    const char* fn = spamm ? "get_batches_spamm" : "get_batches_multiply";
    char msg[200];
    if (!accumulate && !C.empty()) {   // H:5681 / H:6493
        snprintf(msg, sizeof msg, "Error in HierarchicalBlockSparseMatrix::%s(): non-empty matrix to write result!%s", fn,
                 spamm ? "" : " wow");
        throw_ref(msg);
    }
    if (A.empty() || B.empty()) throw Error(HBSM_E_ARG, "hbsm_b200: product of an empty (unsized) matrix");
    if (A.dtype != B.dtype || A.b != B.b) throw Error(HBSM_E_ARG, "hbsm_b200: operands differ in dtype or blocksize");
    AM = tA ? A.N : A.M;
    const int AN = tA ? A.M : A.N, BM = tB ? B.N : B.M;
    BN = tB ? B.M : B.N;
    if (AN != BM) {   // H:5703, H:5730, H:5756, H:5781
        snprintf(msg, sizeof msg, "Error in HierarchicalBlockSparseMatrix::%s(): matrices have bad sizes!", fn);
        throw_ref(msg);
    }
    if (accumulate && !C.empty() && (C.M != AM || C.N != BN || C.dtype != A.dtype || C.b != A.b))
        throw Error(HBSM_E_ARG, "hbsm_b200: multiply_accumulate: C differs from op(A)*op(B) in shape, dtype or blocksize");
}

}  // namespace

// leaf products per line of op(A) (C block row) that op(A)*op(B) would execute: the count pass of the task-list builder only.
// B may be a structure-only matrix (keys + norms, no tiles: e.g. a published table).  d_out has op(A)'s grid side entries.
void product_row_counts(const Matrix& A, bool tA, const Matrix& B, bool tB, const ProductOpts& o, uint64_t* d_out) {
    ensure_engine();
    const uint32_t lines = A.grid_side();
    HB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)lines * sizeof(uint64_t), engine().stream));
    if (A.empty() || B.empty() || A.L == 0 || B.n_ext() == 0) return;
    TaskList tl;
    const int kb = coord_bits(A, B, 1, 1, A.b);
    build_tasks(A, tA, B, tB, o, kb, tl, true, 0, (size_t)-1, nullptr, nullptr, d_out);
}

void check_spamm_operands(const Matrix& A, bool tA, const Matrix& B, bool tB, bool updated) {
    const Matrix none;
    int AM = 0, BN = 0;
    check_operands(A, tA, B, tB, none, true, false, AM, BN);
    if (3 * coord_bits(A, B, AM, BN, A.b) > 64) throw Error(HBSM_E_ARG, "hbsm_b200: block grid too deep for 64-bit task keys (depth > 21)");
    if (!updated && B.n_halo > 0) throw Error(HBSM_E_ARG, "hbsm_b200: spamm(updated=false) on an operand with a committed halo");
}

size_t product_candidates(const Matrix& A, bool tA, const Matrix& B, bool tB, bool upper_only, DevBuf<uint64_t>& begin,
                          DevBuf<uint2>& ab, size_t* n_ctiles) {
    ensure_engine();
    ProductOpts o;
    o.upper_only = upper_only;
    TaskList tl;
    build_tasks(A, tA, B, tB, o, coord_bits(A, B, tA ? A.N : A.M, tB ? B.M : B.N, A.b), tl, false);
    begin = std::move(tl.begin);
    ab = std::move(tl.ab);
    *n_ctiles = tl.n_ctiles;
    return tl.n_products;
}

bool worth_product(const Matrix& A, bool tA, const Matrix& B, bool tB, bool spamm, double tau) {
    if (A.empty() || B.empty()) return false;
    ensure_engine();
    ProductOpts o;
    o.spamm = spamm;
    o.tau = tau;
    TaskList tl;
    int kb = coord_bits(A, B, 1, 1, A.b);
    build_tasks(A, tA, B, tB, o, kb, tl, true);
    return tl.n_products > 0;
}

namespace {

// per C tile: does any of its products read a halo tile of B (tile index >= n_own)?
__global__ void k_classify_ctiles(const uint2* __restrict__ ab, const uint64_t* __restrict__ begin, size_t nct, uint32_t n_own,
                                  uint32_t* __restrict__ own_only) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nct) return;
    bool halo = false;
    for (uint64_t p = begin[t]; p < begin[t + 1] && !halo; ++p) halo = ab[p].y >= n_own;
    own_only[t] = halo ? 0u : 1u;
}
// both lists from ONE scan of the own-only flags: own tiles go to first[pos], the others to later[t - pos]
__global__ void k_split_lists(const uint32_t* __restrict__ own_only, const uint64_t* __restrict__ pos, size_t n,
                              uint32_t* __restrict__ first, uint32_t* __restrict__ later) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (own_only[i]) first[pos[i]] = (uint32_t)i;
    else later[i - pos[i]] = (uint32_t)i;
}

// accumulating product, per tile u of the union of P's C tiles (ckeys, begin) and C_old's tiles: its product range (empty
// for a tile only in C_old: it starts where the next P tile starts) and whether it has products
__global__ void k_union_ranges(const uint64_t* __restrict__ ukeys, const uint32_t* __restrict__ src_p, size_t nu,
                               const uint64_t* __restrict__ ckeys, size_t nct, const uint64_t* __restrict__ begin,
                               uint64_t* __restrict__ ubegin, uint32_t* __restrict__ has_products) {
    size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nu) return;
    size_t j = src_p[u];
    if (j == ACC_NONE) {
        size_t lo = 0, hi = nct;
        while (lo < hi) { size_t mid = (lo + hi) >> 1; if (ckeys[mid] < ukeys[u]) lo = mid + 1; else hi = mid; }
        j = lo;
    }
    ubegin[u] = begin[j];
    has_products[u] = src_p[u] != ACC_NONE ? 1u : 0u;
    if (u == nu - 1) ubegin[nu] = begin[nct];
}

// one leaf-GEMM launch over `n` C tiles: all of them (tile_list == nullptr) or the listed subset.
// One kernel per (dtype, leaf size); hbsm_set_gemm_variant only swaps in the parity references of the tests:
//   dtype, leaf                        kernel                                                last_gemm_kernel
//   fp64, 32 / 64 / 128 / 256          k_gemm_f64_tma                                        1
//   fp32, 32 / 64                      k_gemm_f32_g32 / _g64 (2 x 2 groups of C tiles);      3
//                                      variant 3: k_gemm_f32_q4<32 / 64> (single C tiles)
//   fp32, 128 / 256                    k_gemm_f32_tc                                         3
//   any other leaf size, or variant 1  k_gemm_generic (plain FMA)                            0
//   a task list without products       k_gemm_generic (the only kernel that takes empty k-lists: the zero leaf of a
//                                      single-leaf accumulate whose one leaf product SpAMM skips)  0
// acc (may be null): the accumulating epilogue, in every kernel
void launch_leaf_gemm(const Matrix& A, bool tA, const Matrix& B, bool tB, const TaskList& tl, const uint32_t* tile_list, size_t n,
                      char* ct, const AccArgs* acc = nullptr) {
    if (n == 0) return;
    Engine& e = engine();
    const int variant = shared().gemm_variant.load();
    const uint32_t nn = (uint32_t)n;
    const bool tensor_leaf = A.b == 32 || A.b == 64 || A.b == 128 || A.b == 256;
    const AccArgs plain;
    const AccArgs& ea = acc ? *acc : plain;
    if (variant == 1 || !tensor_leaf || tl.n_products == 0) {
        with_acc(acc, [&](auto on) {
            constexpr bool ACC = decltype(on)::value;
            if (A.dtype == HBSM_F64) {
                auto kfn = k_gemm_generic<double, ACC>;
                HB_LAUNCH(kfn, nn, 256, 0, (const double*)A.tiles.p, (const double*)B.tiles.p, tl.ab.p, tl.begin.p, tile_list, A.b,
                          tA ? 1 : 0, tB ? 1 : 0, (double*)ct, ea.epi<double>());
            } else {
                auto kfn = k_gemm_generic<float, ACC>;
                HB_LAUNCH(kfn, nn, 256, 0, (const float*)A.tiles.p, (const float*)B.tiles.p, tl.ab.p, tl.begin.p, tile_list, A.b,
                          tA ? 1 : 0, tB ? 1 : 0, (float*)ct, ea.epi<float>());
            }
        });
        e.last_gemm_kernel = 0;
        return;
    }
    DevBuf<unsigned> counter(1);   // the persistent kernels' C-tile scheduler; released in stream order
    counter.zero();
    if (A.dtype == HBSM_F64) {
        double* Ct = (double*)ct;
        const AccEpi<double> ep = ea.epi<double>();
        with_acc(acc, [&](auto on) {
            constexpr bool ACC = decltype(on)::value;
            switch (A.b) {
                case 32: launch_gemm_f64_tma<32, 32, 32, ACC>(tA, tB, A, B, tl.ab.p, tl.begin.p, nn, tile_list, counter.p, Ct, ep); break;
                case 64: launch_gemm_f64_tma<64, 64, 64, ACC>(tA, tB, A, B, tl.ab.p, tl.begin.p, nn, tile_list, counter.p, Ct, ep); break;
                case 128: launch_gemm_f64_tma<128, 128, 32, ACC>(tA, tB, A, B, tl.ab.p, tl.begin.p, nn, tile_list, counter.p, Ct, ep); break;
                default: launch_gemm_f64_tma<256, 128, 32, ACC>(tA, tB, A, B, tl.ab.p, tl.begin.p, nn, tile_list, counter.p, Ct, ep); break;
            }
        });
        e.last_gemm_kernel = 1;
    } else {   // split-TF32 on tcgen05 (gemm_f32.cu)
        launch_gemm_f32_tc(A, tA, B, tB, tl.ab.p, tl.begin.p, nn, tile_list, counter.p, (float*)ct, tl.ckeys.p, tl.task_k.p,
                           tl.n_products, variant == 3, acc);
        e.last_gemm_kernel = 3;
    }
}

// a product between op_product_begin and op_product_finish (one at a time per host thread)
struct PendingProduct {
    bool active = false;
    const Matrix* A = nullptr; const Matrix* B = nullptr; Matrix* C = nullptr;
    bool tA = false, tB = false;
    TaskList tl;
    DevBuf<char> ct;
    DevBuf<uint32_t> later;      // C tiles whose products read halo tiles: computed by finish
    size_t n_later = 0;
    DevBuf<uint32_t> first;      // the other C tiles, when their launch was left to finish as well (launch_in_finish)
    size_t n_first = 0;
    bool first_pending = false, first_is_list = false;
    bool upper_only = false;     // finish zeroes the strict lower part of C's diagonal tiles (H:3563 via triu)
    bool replace_table = false;  // finish installs the planned table even without products (accumulate into a sized C)
    size_t old_mults = 0;        // C_old's n_mults when it takes part (accumulate, beta != 0)
    bool c_was_empty = false;    // begin sized C: an abort returns it to the empty state (dtype and leaf size as they were)
    int c_dtype = 0, c_b = -1;
    uint64_t launches0 = 0;
    EventTimer t_total, t_norm, t_index, t_task, t_gemm, t_gemm2;
};
PendingProduct& pending() {
    thread_local PendingProduct p;   // per host thread: products of different threads do not meet
    return p;
}

// drops the planned product's buffers; a C that begin sized goes back to the empty state it was in
void drop_pending(PendingProduct& P) {
    P.tl = TaskList(); P.ct.release(); P.later.release(); P.first.release(); P.first_pending = false;
    P.replace_table = false;
    P.old_mults = 0;
    if (P.c_was_empty && P.C) {
        P.C->clear();
        P.C->dtype = P.c_dtype;
        P.C->b = P.c_b;
    }
    P.c_was_empty = false;
}

}  // namespace

void op_product_begin(const Matrix& A, bool tA, const Matrix& B, bool tB, Matrix& C, const ProductOpts& o, bool defer_halo_tiles,
                      bool launch, bool launch_in_finish) {
    ensure_engine();   // before pending(): its event timers must be created on the engine's device
    PendingProduct& P = pending();
    if (P.active) throw Error(HBSM_E_ARG, "hbsm_b200: a product is already in flight (finish it first)");
    int AM = 0, BN = 0;
    const bool accumulate = o.c_old != nullptr;
    if (accumulate && (o.c_old != &C || defer_halo_tiles || !launch || o.upper_only))
        throw Error(HBSM_E_ARG, "hbsm_b200: an accumulating product runs in one call, on C's own table");
    check_operands(A, tA, B, tB, C, o.spamm, accumulate, AM, BN);
    // every other rejection comes before C is touched, too
    const int kbits = coord_bits(A, B, AM, BN, A.b);
    if (3 * kbits > 64) throw Error(HBSM_E_ARG, "hbsm_b200: block grid too deep for 64-bit task keys (depth > 21)");
    if (o.spamm && !o.updated && B.n_halo > 0)
        throw Error(HBSM_E_ARG, "hbsm_b200: spamm(updated=false) on an operand with a committed halo");
    Engine& e = engine();
    P.launches0 = e.launches;
    P.t_total.start();
    // accumulate into a sized C: its table (C_old) stays in place -- C may be A or B -- until finish installs the new one
    const bool sized_old = accumulate && C.sized;
    const bool use_old = sized_old && o.beta != 0.0 && C.L > 0;   // beta == 0: C_old is not read (BLAS)
    P.replace_table = sized_old;
    P.old_mults = sized_old && o.beta != 0.0 ? C.n_mults : 0;
    P.C = &C;
    P.c_was_empty = !sized_old;   // (a product that is not accumulating requires an empty C)
    P.c_dtype = C.dtype;
    P.c_b = C.b;
    struct Undo {   // anything below that throws leaves C as it was at the call
        PendingProduct& P;
        bool armed;
        ~Undo() { if (armed) drop_pending(P); }
    } undo{P, true};
    if (!sized_old) {
        C.dtype = A.dtype;
        C.b = A.b;
        C.resize(AM, BN);
    }

    P.t_norm.start();
    // updated=false: the reference copies A and B, refreshes the COPIES and leaves the operands' caches alone (H:3990-4005;
    // its batched build then reads freed memory, H:6294-6307).  Same contract here: fresh leaf norms into temporaries.
    DevBuf<char> fresh_a, fresh_b;
    const void* an = nullptr;
    const void* bn = nullptr;
    if (o.spamm && !o.updated) {
        fresh_a.alloc(std::max<size_t>(A.L, 1) * A.esize());
        compute_leaf_norms(A, fresh_a.p);
        an = fresh_a.p;
        if (&B != &A) {
            fresh_b.alloc(std::max<size_t>(B.L, 1) * B.esize());
            compute_leaf_norms(B, fresh_b.p);
            bn = fresh_b.p;
        } else {
            bn = an;
        }
    }
    P.t_norm.stop();
    P.t_index.start();
    line_index(A, tA);
    line_index(B, tB, true);
    P.t_index.stop();

    P.t_task.start();
    P.tl = TaskList();
    build_tasks(A, tA, B, tB, o, kbits, P.tl, false, 0, (size_t)-1, an, bn);
    P.n_later = 0;
    DevBuf<uint32_t>& first = P.first;
    first.release();
    size_t n_first = P.tl.n_ctiles;
    P.first_pending = false;
    const bool split = defer_halo_tiles && B.n_halo > 0 && P.tl.n_products > 0;
    if (split) {   // C tiles that only read B's own tiles can start now; the others wait for the halo tiles
        const size_t nct = P.tl.n_ctiles;
        DevBuf<uint32_t> own(nct);
        DevBuf<uint64_t> pos(nct + 1);
        HB_LAUNCH(k_classify_ctiles, blocks_for(nct, 256), 256, 0, P.tl.ab.p, P.tl.begin.p, nct, (uint32_t)B.L, own.p);
        exclusive_scan_u32(own.p, pos.p, nct);
        first.alloc(nct);       // sized for the worst case: no read-back before the kernels are queued
        P.later.alloc(nct);
        HB_LAUNCH(k_split_lists, blocks_for(nct, 256), 256, 0, own.p, pos.p, nct, first.p, P.later.p);
        n_first = (size_t)read_scalars(pos.p + nct, nullptr).first;
        P.n_later = nct - n_first;
    }
    // a single-leaf product always has its leaf: when SpAMM skips the one leaf product, P is the zero leaf of resize(), and an
    // accumulating product runs it as a C tile with an empty k-list, so its epilogue gives fl(fl(alpha * 0) + fl(beta * c))
    const bool zero_leaf = accumulate && P.tl.n_products == 0 && Matrix::depth_for(AM, BN, A.b) == 0;
    if (zero_leaf) {
        P.tl.ckeys.alloc(1);
        P.tl.ckeys.zero();
        P.tl.begin.alloc(2);
        P.tl.begin.zero();
        P.tl.n_ctiles = 1;
        n_first = 1;
        P.replace_table = true;
    }
    P.t_task.stop();

    // accumulate, beta != 0: C's table becomes the union of P's tiles and C_old's; the leaf GEMMs run over the union tiles with
    // products (gemm_list, ascending) and read their old values through old_of, the C_old-only tiles get fl(beta * c)
    AccArgs acc;
    DevBuf<uint32_t> old_of, gemm_list, old_only;
    size_t n_old_only = 0;
    if (use_old) {
        const size_t nct = P.tl.n_ctiles;
        DevBuf<uint64_t> ukeys;
        DevBuf<uint32_t> src_p;
        const size_t nu = key_union(P.tl.ckeys.p, nct, C.keys.p, C.L, ukeys, src_p, old_of);
        DevBuf<uint64_t> ubegin(nu + 1), pos(nu + 1);
        DevBuf<uint32_t> has(nu);
        if (nct == 0) {   // no C tile from the product: an empty task table to range over
            P.tl.begin.alloc(1);
            P.tl.begin.zero();
        }
        HB_LAUNCH(k_union_ranges, blocks_for(nu, 256), 256, 0, ukeys.p, src_p.p, nu, P.tl.ckeys.p, nct, P.tl.begin.p, ubegin.p, has.p);
        exclusive_scan_u32(has.p, pos.p, nu);
        gemm_list.alloc(std::max<size_t>(nct, 1));
        n_old_only = nu - nct;
        old_only.alloc(std::max<size_t>(n_old_only, 1));
        HB_LAUNCH(k_split_lists, blocks_for(nu, 256), 256, 0, has.p, pos.p, nu, gemm_list.p, old_only.p);
        P.tl.ckeys = std::move(ukeys);
        P.tl.begin = std::move(ubegin);
        P.tl.n_ctiles = nu;
        first.release();
        n_first = nct;
        acc.idx = old_of.p;
    }
    if (accumulate) {
        acc.old = C.tiles.p;
        acc.alpha = o.alpha;
        acc.beta = o.beta;
    }
    const bool fill = P.tl.n_products > 0 || zero_leaf || (use_old && P.tl.n_ctiles > 0);
    if (fill) P.ct.alloc(P.tl.n_ctiles * C.tile_bytes());   // before the timer: a growing pool stalls the host here
    P.t_gemm.start();
    if (P.tl.n_products > 0 || zero_leaf) {
        if (accumulate) launch_leaf_gemm(A, tA, B, tB, P.tl, use_old ? gemm_list.p : nullptr, n_first, P.ct.p, &acc);
        else if (launch) launch_leaf_gemm(A, tA, B, tB, P.tl, split ? first.p : nullptr, n_first, P.ct.p);
        else if (launch_in_finish) { P.first_pending = true; P.first_is_list = split; P.n_first = n_first; }
    }
    if (use_old) scale_tiles_into(C, old_of.p, old_only.p, n_old_only, o.beta, P.ct.p);
    P.t_gemm.stop();
    P.A = &A; P.B = &B; P.tA = tA; P.tB = tB;
    P.upper_only = o.upper_only;
    undo.armed = false;
    P.active = true;
}

void op_product_finish(Matrix& C, cudaEvent_t wait_for, size_t* n_mults, size_t* n_blocks) {
    PendingProduct& P = pending();
    if (!P.active || P.C != &C) throw Error(HBSM_E_ARG, "hbsm_b200: product_finish without a matching product_begin");
    Engine& e = engine();
    P.active = false;
    P.c_was_empty = false;
    if (P.first_pending) {   // begin left every launch to us: own-only tiles now, the halo readers once `wait_for` has fired
        P.t_gemm.start();
        launch_leaf_gemm(*P.A, P.tA, *P.B, P.tB, P.tl, P.first_is_list ? P.first.p : nullptr, P.n_first, P.ct.p);
        P.t_gemm.stop();
        P.first_pending = false;
    }
    if (wait_for) HB_CUDA(cudaStreamWaitEvent(e.stream, wait_for, 0));   // e.g. the NCCL transfer of the halo tiles
    P.t_gemm2.start();
    if (P.n_later > 0) launch_leaf_gemm(*P.A, P.tA, *P.B, P.tB, P.tl, P.later.p, P.n_later, P.ct.p);
    P.t_gemm2.stop();
    if (P.tl.n_products > 0 || P.replace_table) {
        // (an accumulating product releases C_old's buffers here, in stream order behind the kernels that read them)
        const size_t nct = P.tl.n_ctiles;
        C.drop_tasks();
        C.set_table(std::move(P.tl.ckeys), std::move(P.ct), nct);
        C.root_norm_cached = 0.0;   // stale with the leaf norms, as after resize()
        if (nct > 0) {
            C.task_begin = std::move(P.tl.begin);
            C.task_k = std::move(P.tl.task_k);
            C.n_tasks = P.tl.n_products;
        }
        if (P.upper_only) mask_diag_upper(C);   // triu of the diagonal tiles (the off-diagonal ones were never planned)
    }
    P.t_total.stop();
    sync_stream();
    P.later.release();
    P.first.release();
    C.n_mults = P.tl.n_products + P.old_mults;   // H:2194 / H:3984; accumulate: + C_old's as add does (H:1719)
    P.replace_table = false;
    P.old_mults = 0;
    if (n_mults) *n_mults = P.tl.n_products;
    if (n_blocks) *n_blocks = C.L;   // get_n_blocks(), H:7311
    hbsm_stage_times st{};
    st.norms_ms = P.t_norm.ms();
    st.index_ms = P.t_index.ms();
    st.tasklist_ms = P.t_task.ms();
    st.gemm_ms = P.t_gemm.ms() + P.t_gemm2.ms();
    st.total_ms = P.t_total.ms();
    st.n_candidates = P.tl.n_candidates;
    st.n_products = P.tl.n_products;
    st.n_ctiles = P.tl.n_ctiles;
    st.gpu_launches = e.launches - P.launches0;
    st.gemm_kernel = (uint64_t)e.last_gemm_kernel;
    e.last = st;
    P.tl = TaskList();
}

void op_product_abort() {
    PendingProduct& P = pending();
    if (!P.active) return;
    P.active = false;
    cudaStreamSynchronize(engine().stream);
    drop_pending(P);
}

// product whose C tiles stream to HOST memory while later tiles are still being computed: the leaf GEMM is launched in
// `n_chunks` ranges of the (Morton-ordered) C tile list; a copy stream ships each finished range (PCIe D2H overlaps the
// remaining GEMMs).  `host_tiles` should be pinned; it receives all C tiles in table order.  C is completed as usual.
void op_product_to_host(const Matrix& A, bool tA, const Matrix& B, bool tB, Matrix& C, const ProductOpts& o, void* host_tiles,
                        size_t cap_tiles, int n_chunks, size_t* n_mults, size_t* n_blocks) {
    ensure_engine();
    Engine& e = engine();
    thread_local cudaStream_t copy_stream = nullptr;
    if (!copy_stream) HB_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
    op_product_begin(A, tA, B, tB, C, o, /*defer_halo_tiles=*/false, /*launch=*/false, /*launch_in_finish=*/false);
    PendingProduct& P = pending();
    const size_t nct = P.tl.n_ctiles;
    bool streamed = false;
    if (nct > 0 && host_tiles && cap_tiles >= nct) {
        streamed = true;
        n_chunks = std::max(1, std::min<int>(n_chunks, (int)((nct + 1023) / 1024)));
        DevBuf<uint32_t> order(nct);
        HB_LAUNCH(k_iota, blocks_for(nct, 256), 256, 0, order.p, nct);
        std::vector<cudaEvent_t> done((size_t)n_chunks);
        P.t_gemm.start();
        for (int c = 0; c < n_chunks; ++c) {
            const size_t lo = nct * (size_t)c / n_chunks, hi = nct * (size_t)(c + 1) / n_chunks;
            launch_leaf_gemm(A, tA, B, tB, P.tl, order.p + lo, hi - lo, P.ct.p);
            HB_CUDA(cudaEventCreateWithFlags(&done[c], cudaEventDisableTiming));
            HB_CUDA(cudaEventRecord(done[c], e.stream));
            HB_CUDA(cudaStreamWaitEvent(copy_stream, done[c], 0));
            HB_CUDA(cudaMemcpyAsync((char*)host_tiles + lo * C.tile_bytes(), P.ct.p + lo * C.tile_bytes(), (hi - lo) * C.tile_bytes(),
                                    cudaMemcpyDeviceToHost, copy_stream));
        }
        P.t_gemm.stop();
        HB_CUDA(cudaStreamSynchronize(copy_stream));
        for (cudaEvent_t ev : done) cudaEventDestroy(ev);
    } else if (nct > 0) {
        P.t_gemm.start();
        launch_leaf_gemm(A, tA, B, tB, P.tl, nullptr, nct, P.ct.p);
        P.t_gemm.stop();
    }
    op_product_finish(C, nullptr, n_mults, n_blocks);
    if (!streamed && host_tiles && C.L && cap_tiles < C.L) throw Error(HBSM_E_ARG, "hbsm_b200: host buffer too small for the tiles of C");
    if (!streamed && host_tiles && C.L) {   // no product ran: C is the zero leaf resize() gives a single-leaf C
        HB_CUDA(cudaMemcpyAsync(host_tiles, C.tiles.p, C.L * C.tile_bytes(), cudaMemcpyDeviceToHost, e.stream));
        sync_stream();
    }
}

// ---------------------------------------------------------------------------------------------------
// host-to-host product: uploads, norms, task lists, leaf GEMMs and downloads pipelined over block-row slabs of C
// ---------------------------------------------------------------------------------------------------
namespace {

struct HostPlan {   // one operand: its tiles sorted by Morton key, cut into upload runs per slab
    struct Run { size_t dst, src, cnt; };   // sorted positions [dst, dst+cnt) <- host tiles [src, src+cnt)
    std::vector<uint64_t> keys;             // ascending
    std::vector<uint32_t> src;              // host tile of sorted position i
    std::vector<std::vector<Run>> runs;     // [slab]
    size_t n_runs = 0;
};

// slab coordinate of a tile: block row (by_col = false) or block column (by_col = true), >> shift
void plan_operand(const Matrix& X, const HostTiles& h, bool by_col, int shift, int S, HostPlan& pl) {
    const uint32_t g = X.grid_side();
    const size_t n = h.n;
    pl.keys.resize(n);
    pl.src.resize(n);
    bool sorted = true;
    for (size_t i = 0; i < n; ++i) {
        const int bi = h.bi[i], bj = h.bj[i];
        if (bi < 0 || bj < 0 || (uint32_t)bi >= g || (uint32_t)bj >= g || (long long)bi * X.b >= std::max(X.M, 1) ||
            (long long)bj * X.b >= std::max(X.N, 1))
            throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: index outside matrix boundaries.");
        pl.keys[i] = morton_encode((uint32_t)bi, (uint32_t)bj);
        pl.src[i] = (uint32_t)i;
        if (i && pl.keys[i] <= pl.keys[i - 1]) sorted = false;
    }
    if (!sorted) {
        std::sort(pl.src.begin(), pl.src.end(), [&](uint32_t a, uint32_t b) { return pl.keys[a] < pl.keys[b]; });
        std::vector<uint64_t> k2(n);
        for (size_t i = 0; i < n; ++i) k2[i] = pl.keys[pl.src[i]];
        pl.keys.swap(k2);
        for (size_t i = 1; i < n; ++i)
            if (pl.keys[i] == pl.keys[i - 1]) throw Error(HBSM_E_ARG, "hbsm_b200: assign_tiles: tile coordinates are not unique");
    }
    pl.runs.assign((size_t)S, {});
    int cur = -1;
    for (size_t i = 0; i < n; ++i) {
        const uint32_t coord = by_col ? morton_col(pl.keys[i]) : morton_row(pl.keys[i]);
        const int sl = std::min<int>((int)(coord >> shift), S - 1);
        if (sl == cur && pl.src[i] == pl.src[i - 1] + 1) {
            pl.runs[sl].back().cnt++;
        } else {
            pl.runs[sl].push_back({i, pl.src[i], 1});
            pl.n_runs++;
            cur = sl;
        }
    }
}

// dst tile j = tile idx[j] of the concatenation of the per-slab tile buffers (16-byte vectors)
__global__ void __launch_bounds__(256) k_gather_slab_tiles(const uint32_t* __restrict__ idx, const uint64_t* __restrict__ slab_off,
                                                           const uint4* const* __restrict__ slab_ptr, int n_slabs,
                                                           size_t vec_per_tile, uint4* __restrict__ dst) {
    const size_t j = blockIdx.x;
    const uint32_t src = idx[j];
    int lo = 0, hi = n_slabs - 1;   // last slab with slab_off[s] <= src
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (slab_off[mid] <= src) lo = mid; else hi = mid - 1;
    }
    const uint4* from = slab_ptr[lo] + (size_t)(src - slab_off[lo]) * vec_per_tile;
    uint4* to = dst + j * vec_per_tile;
    for (size_t v = (size_t)blockIdx.y * blockDim.x + threadIdx.x; v < vec_per_tile; v += (size_t)gridDim.y * blockDim.x) to[v] = from[v];
}

struct SideStreams {
    cudaStream_t h2d = nullptr, d2h = nullptr;
};
SideStreams& side_streams() {
    thread_local SideStreams s;
    if (!s.h2d) {
        HB_CUDA(cudaStreamCreateWithFlags(&s.h2d, cudaStreamNonBlocking));
        HB_CUDA(cudaStreamCreateWithFlags(&s.d2h, cudaStreamNonBlocking));
    }
    return s;
}

}  // namespace

void op_product_from_host(Matrix& A, const HostTiles& ha, bool tA, Matrix& B, const HostTiles& hb, bool tB, Matrix& C,
                          const ProductOpts& o, int n_slabs, void* host_c_tiles, size_t cap_tiles, int* c_bi, int* c_bj,
                          size_t* n_mults, size_t* n_blocks) {
    ensure_engine();
    Engine& e = engine();
    const auto wall0 = std::chrono::steady_clock::now();
    std::vector<std::pair<const char*, double>> marks;
    auto mark = [&](const char* what) {
        marks.emplace_back(what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count());
    };
    if (&A == &B) throw Error(HBSM_E_ARG, "hbsm_b200: product_from_host needs two distinct operand handles");
    int AM = 0, BN = 0;
    check_operands(A, tA, B, tB, C, o.spamm, false, AM, BN);
    if ((ha.n && (!ha.bi || !ha.bj || !ha.tiles)) || (hb.n && (!hb.bi || !hb.bj || !hb.tiles)))
        throw Error(HBSM_E_ARG, "hbsm_b200: product_from_host: null tile arrays");
    const uint64_t launches0 = e.launches;
    const size_t tb = A.tile_bytes();
    // degenerate (single-leaf operand) or unordered input: bulk upload + device gather, then the ordinary product whose
    // C tiles stream to the host
    auto classic = [&]() {
        assign_tiles_host(A, ha.n, ha.bi, ha.bj, ha.tiles);
        assign_tiles_host(B, hb.n, hb.bi, hb.bj, hb.tiles);
        update_norms(A);
        update_norms(B);
        size_t nb = 0;
        try {
            op_product_to_host(A, tA, B, tB, C, o, host_c_tiles, cap_tiles, 8, n_mults, &nb);
        } catch (...) {   // too small a host buffer is reported after C is complete: the caller still learns its size
            if (n_blocks) *n_blocks = nb;
            throw;
        }
        if (n_blocks) *n_blocks = nb;
        if (nb && c_bi && c_bj) {
            std::vector<uint64_t> hk = C.keys.to_host();
            for (size_t i = 0; i < nb && i < hk.size(); ++i) { c_bi[i] = (int)morton_row(hk[i]); c_bj[i] = (int)morton_col(hk[i]); }
        }
    };
    if (A.vdepth() == 0 || B.vdepth() == 0) { classic(); return; }
    if (A.L != 0 || B.L != 0)
        throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: non-null child0 matrix occured.");

    // slab geometry: 2^shift block rows of C per slab, aligned to Morton squares so that a slab is a few contiguous runs
    const uint32_t g = std::max(A.grid_side(), B.grid_side());
    int gbits = 0;
    while ((1u << gbits) < g) ++gbits;
    int S = n_slabs;
    if (S <= 0) S = (ha.n + hb.n) * tb >= ((size_t)64 << 20) ? 16 : 1;
    int sbits = 0;
    while ((2 << sbits) <= S && sbits < gbits) ++sbits;
    S = 1 << sbits;
    const int shift = gbits - sbits;

    HostPlan pa, pb;
    plan_operand(A, ha, tA, shift, S, pa);    // op(A): slab by ci (block column of A if tA)
    plan_operand(B, hb, tB, shift, S, pb);    // op(B): slab by k  (block column of B if tB)
    if (pa.n_runs + pb.n_runs > 4096) { classic(); return; }
    mark("planned");

    // line-entry ranges of op(A) per slab, and the upload order: chunk c = op(A)'s slab c plus every slab of op(B) that
    // slab c's products read and that is not on its way yet, so that C's slab c is computable as soon as chunk c has landed;
    // op(B) slabs nobody asked for travel in a last chunk S
    const uint32_t ga = A.grid_side();
    std::vector<size_t> hptr((size_t)ga + 2, 0);
    std::vector<int> kmax((size_t)S, -1);
    for (size_t i = 0; i < ha.n; ++i) {
        const uint32_t r = morton_row(pa.keys[i]), c = morton_col(pa.keys[i]);
        const uint32_t ci = tA ? c : r, k = tA ? r : c;
        hptr[ci + 1]++;
        const int sc = std::min<int>((int)(ci >> shift), S - 1), sk = std::min<int>((int)(k >> shift), S - 1);
        kmax[sc] = std::max(kmax[sc], sk);
    }
    for (uint32_t l = 0; l < ga; ++l) hptr[l + 1] += hptr[l];
    std::vector<std::vector<int>> chunk_b((size_t)S + 1);
    {
        int b_up = -1;
        for (int c = 0; c < S; ++c)
            for (; b_up < kmax[c];) chunk_b[c].push_back(++b_up);
        for (; b_up < S - 1;) chunk_b[S].push_back(++b_up);
    }

    // device tables: keys now, tiles as they arrive
    {
        DevBuf<uint64_t> ka(std::max<size_t>(ha.n, 1)), kb(std::max<size_t>(hb.n, 1));
        ka.upload(pa.keys.data(), ha.n);
        kb.upload(pb.keys.data(), hb.n);
        DevBuf<char> ta(std::max<size_t>(ha.n, 1) * tb), tbuf(std::max<size_t>(hb.n, 1) * tb);
        A.set_table(std::move(ka), std::move(ta), ha.n);
        B.set_table(std::move(kb), std::move(tbuf), hb.n);
    }
    mark("tables allocated");
    SideStreams& ss = side_streams();
    const bool trace = getenv("HBSM_TRACE_PIPE") != nullptr;   // per-slab timeline on stderr (development aid)
    std::vector<cudaEvent_t> up((size_t)S + 1, nullptr), done((size_t)S, nullptr), shipped((size_t)S, nullptr);
    for (int c = 0; c <= S; ++c) HB_CUDA(cudaEventCreateWithFlags(&up[c], trace ? cudaEventDefault : cudaEventDisableTiming));
    for (int s2 = 0; s2 < S; ++s2) {
        HB_CUDA(cudaEventCreateWithFlags(&done[s2], trace ? cudaEventDefault : cudaEventDisableTiming));
        if (trace) HB_CUDA(cudaEventCreate(&shipped[s2]));
    }
    struct SlabOut { TaskList tl; DevBuf<char> ct; size_t off = 0; };
    std::vector<SlabOut> outs((size_t)S);
    std::vector<EventTimer> tg((size_t)S);
    std::vector<char> timed((size_t)S, 0);
    EventTimer t_total;
    size_t n_ct = 0, P_total = 0;
    unsigned long long cand = 0;
    bool host_ok = host_c_tiles != nullptr;
    std::vector<uint64_t> hk;   // C's keys in slab-major order (the order of host_c_tiles)
    auto destroy_events = [&]() {
        for (cudaEvent_t ev : up) if (ev) cudaEventDestroy(ev);
        for (cudaEvent_t ev : done) if (ev) cudaEventDestroy(ev);
        for (cudaEvent_t ev : shipped) if (ev) cudaEventDestroy(ev);
    };
    try {
        t_total.start();
        // the tile pools were allocated in engine-stream order: the upload stream may touch them after this event
        HB_CUDA(cudaEventRecord(done[0], e.stream));
        HB_CUDA(cudaStreamWaitEvent(ss.h2d, done[0], 0));
        for (int c = 0; c <= S; ++c) {   // every upload is queued now; PCIe stays busy from here to the last tile
            if (c < S)
                for (const HostPlan::Run& r : pa.runs[c])
                    HB_CUDA(cudaMemcpyAsync(A.tiles.p + r.dst * tb, (const char*)ha.tiles + r.src * tb, r.cnt * tb, cudaMemcpyHostToDevice, ss.h2d));
            for (int j : chunk_b[c])
                for (const HostPlan::Run& r : pb.runs[j])
                    HB_CUDA(cudaMemcpyAsync(B.tiles.p + r.dst * tb, (const char*)hb.tiles + r.src * tb, r.cnt * tb, cudaMemcpyHostToDevice, ss.h2d));
            HB_CUDA(cudaEventRecord(up[c], ss.h2d));
        }
        mark("uploads queued");
        C.dtype = A.dtype;
        C.b = A.b;
        C.resize(AM, BN);
        const int kbits = coord_bits(A, B, AM, BN, A.b);
        if (3 * kbits > 64) throw Error(HBSM_E_ARG, "hbsm_b200: block grid too deep for 64-bit task keys (depth > 21)");
        ProductOpts oo = o;
        oo.updated = true;   // norms are refreshed chunk by chunk below
        int normed = -1;
        auto norms_up_to = [&](int c_hi) {
            for (int c = normed + 1; c <= c_hi; ++c) {
                HB_CUDA(cudaStreamWaitEvent(e.stream, up[c], 0));
                if (c < S)
                    for (const HostPlan::Run& r : pa.runs[c]) compute_leaf_norms_range(A, r.dst, r.cnt, A.norms.p);
                for (int j : chunk_b[c])
                    for (const HostPlan::Run& r : pb.runs[j]) compute_leaf_norms_range(B, r.dst, r.cnt, B.norms.p);
            }
            normed = std::max(normed, c_hi);
        };
        for (int s2 = 0; s2 < S; ++s2) {
            const uint32_t l_lo = std::min<uint32_t>((uint32_t)s2 << shift, ga);
            const uint32_t l_hi = (s2 == S - 1) ? ga : std::min<uint32_t>((uint32_t)(s2 + 1) << shift, ga);
            const size_t e_lo = hptr[l_lo], e_hi = hptr[l_hi];
            if (e_lo == e_hi) continue;
            norms_up_to(s2);
            SlabOut& so = outs[s2];
            build_tasks(A, tA, B, tB, oo, kbits, so.tl, false, e_lo, e_hi);
            cand += so.tl.n_candidates;
            if (so.tl.n_products == 0) continue;
            const size_t nct = so.tl.n_ctiles;
            so.off = n_ct;
            so.ct.alloc(nct * tb);
            tg[s2].start();
            launch_leaf_gemm(A, tA, B, tB, so.tl, nullptr, nct, so.ct.p);
            tg[s2].stop();
            timed[s2] = 1;
            if (host_ok && n_ct + nct <= cap_tiles) {
                HB_CUDA(cudaEventRecord(done[s2], e.stream));
                HB_CUDA(cudaStreamWaitEvent(ss.d2h, done[s2], 0));
                HB_CUDA(cudaMemcpyAsync((char*)host_c_tiles + n_ct * tb, so.ct.p, nct * tb, cudaMemcpyDeviceToHost, ss.d2h));
                if (trace) HB_CUDA(cudaEventRecord(shipped[s2], ss.d2h));
            } else {
                host_ok = false;
            }
            n_ct += nct;
            P_total += so.tl.n_products;
        }
        norms_up_to(S);
        mark("slabs launched");
        // roots of the two norm refreshes (H:3918-3923); this is also where the host joins the engine stream
        A.root_norm_cached = A.L ? hierarchical_norm(A, A.norms.p) : 0.0;
        B.root_norm_cached = B.L ? hierarchical_norm(B, B.norms.p) : 0.0;
        mark("root norms");

        // C's block table: the slabs' tiles merged into one Morton-ordered pool.  Queued behind the last leaf GEMM and NOT
        // waited for: the host results are complete when the download stream drains, the device table when the engine
        // stream does (every later call on C is stream-ordered behind it).
        if (n_ct > 0) {
            int first = -1, n_nonempty = 0;
            for (int s2 = 0; s2 < S; ++s2) if (outs[s2].tl.n_products) { if (first < 0) first = s2; ++n_nonempty; }
            if (c_bi && c_bj) {
                hk.resize(n_ct);
                for (int s2 = 0; s2 < S; ++s2)
                    if (outs[s2].tl.n_products) outs[s2].tl.ckeys.download(hk.data() + outs[s2].off, outs[s2].tl.n_ctiles);
                sync_stream();
            }
            if (n_nonempty == 1) {
                SlabOut& so = outs[first];
                C.set_table(std::move(so.tl.ckeys), std::move(so.ct), n_ct);
                C.task_begin = std::move(so.tl.begin);
                C.task_k = std::move(so.tl.task_k);
                C.n_tasks = so.tl.n_products;
            } else {
                DevBuf<uint64_t> skeys(n_ct);
                DevBuf<uint32_t> idx(n_ct);
                std::vector<uint64_t> h_off((size_t)S);
                std::vector<const uint4*> h_ptr((size_t)S);
                for (int s2 = S - 1, nxt = -1; s2 >= 0; --s2) {   // slabs without tiles must not win the search below
                    if (outs[s2].tl.n_products) {
                        nxt = s2;
                        h_off[s2] = outs[s2].off;
                        HB_CUDA(cudaMemcpyAsync(skeys.p + outs[s2].off, outs[s2].tl.ckeys.p, outs[s2].tl.n_ctiles * sizeof(uint64_t),
                                                cudaMemcpyDeviceToDevice, e.stream));
                    } else {
                        h_off[s2] = nxt >= 0 ? outs[nxt].off : n_ct;
                    }
                    h_ptr[s2] = (const uint4*)outs[s2].ct.p;
                }
                HB_LAUNCH(k_iota, blocks_for(n_ct, 256), 256, 0, idx.p, n_ct);
                radix_sort_pairs(skeys.p, idx.p, n_ct, 2 * std::max(C.vdepth(), 1));
                DevBuf<uint64_t> d_off((size_t)S);
                DevBuf<const uint4*> d_ptr((size_t)S);
                d_off.upload(h_off.data(), (size_t)S);   // small pageable sources: staged by the driver before the call returns
                d_ptr.upload(h_ptr.data(), (size_t)S);
                DevBuf<char> t(n_ct * tb);
                dim3 grid((unsigned)n_ct, (unsigned)std::max<size_t>(1, std::min<size_t>(8, tb / 16 / 1024)));
                HB_LAUNCH(k_gather_slab_tiles, grid, 256, 0, idx.p, d_off.p, d_ptr.p, S, tb / 16, (uint4*)t.p);
                C.set_table(std::move(skeys), std::move(t), n_ct);
                C.drop_tasks();
            }
        } else if (C.L > 0) {   // no product ran: C is the zero leaf resize() gives a single-leaf C, and the caller gets it
            if (host_ok && cap_tiles >= C.L) {
                HB_CUDA(cudaEventRecord(done[0], e.stream));   // behind resize()'s zero fill
                HB_CUDA(cudaStreamWaitEvent(ss.d2h, done[0], 0));
                HB_CUDA(cudaMemcpyAsync(host_c_tiles, C.tiles.p, C.L * tb, cudaMemcpyDeviceToHost, ss.d2h));
                hk = C.keys.to_host();
                hk.resize(C.L);
            } else {
                host_ok = false;
            }
        }
        t_total.stop();
        mark("C merge queued");
        HB_CUDA(cudaStreamSynchronize(ss.d2h));
        mark("downloads complete");
        if (c_bi && c_bj && host_ok)
            for (size_t i = 0; i < hk.size(); ++i) { c_bi[i] = (int)morton_row(hk[i]); c_bj[i] = (int)morton_col(hk[i]); }
        if (trace) {
            sync_stream();
            auto at = [&](cudaEvent_t ev) { float t = -1.f; if (ev && cudaEventQuery(ev) == cudaSuccess) cudaEventElapsedTime(&t, t_total.a, ev); return t; };
            fprintf(stderr, "[hbsm pipe] S=%d runs A=%zu B=%zu device timeline %.2f ms\n", S, pa.n_runs, pb.n_runs, t_total.ms());
            for (auto& mk : marks) fprintf(stderr, "[hbsm pipe] host wall %8.2f ms  %s\n", mk.second, mk.first);
            for (int s2 = 0; s2 < S; ++s2)
                fprintf(stderr, "[hbsm pipe] slab %2d: uploaded %.2f  gemm start %.2f end %.2f  shipped %.2f  (%zu products, %zu C tiles)\n",
                        s2, at(up[s2]), timed[s2] ? at(tg[s2].a) : -1.f, timed[s2] ? at(tg[s2].b) : -1.f,
                        host_ok && timed[s2] ? at(shipped[s2]) : -1.f, outs[s2].tl.n_products, outs[s2].tl.n_ctiles);
        }
    } catch (...) {
        cudaStreamSynchronize(ss.h2d); cudaStreamSynchronize(e.stream); cudaStreamSynchronize(ss.d2h);
        destroy_events();
        throw;
    }
    destroy_events();
    if (n_ct > 0) {   // C's table may still be merging on this thread's stream: later calls on C order themselves behind it
        if (!C.pending_ev) HB_CUDA(cudaEventCreateWithFlags(&C.pending_ev, cudaEventDisableTiming));
        HB_CUDA(cudaEventRecord(C.pending_ev, e.stream));
    }
    C.n_mults = P_total;
    if (n_mults) *n_mults = P_total;
    if (n_blocks) *n_blocks = C.L;
    hbsm_stage_times st{};
    for (int s2 = 0; s2 < S; ++s2) if (timed[s2]) st.gemm_ms += tg[s2].ms();
    mark("return");
    st.total_ms = marks.back().second;   // host wall clock of the call: the device table of C may still be merging
    st.n_candidates = cand;
    st.n_products = P_total;
    st.n_ctiles = n_ct;
    st.gpu_launches = e.launches - launches0;
    st.gemm_kernel = (uint64_t)e.last_gemm_kernel;
    e.last = st;
    if (host_c_tiles && !host_ok) throw Error(HBSM_E_ARG, "hbsm_b200: host buffer too small for the tiles of C");
}

void op_product(const Matrix& A, bool tA, const Matrix& B, bool tB, Matrix& C, const ProductOpts& o, size_t* n_mults,
                size_t* n_blocks) {
    op_product_begin(A, tA, B, tB, C, o, false, true, false);
    op_product_finish(C, nullptr, n_mults, n_blocks);
}

}  // namespace hbsm_b200

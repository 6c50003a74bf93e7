// matrix.cu -- the flat block table: sizing, assembly (COO / whole tiles), readback, norms, line indices and the
// HBM-bound structure operations (add, transpose, upper triangle, rescale, copy, symmetric expansion).
// Reference behaviour reproduced here is cited as H:<line> of source/HierarchicalBlockSparseMatrix.h.
#include "matrix.cuh"
#include <chrono>
#include <cmath>

namespace hbsm_b200 {

// ---------------------------------------------------------------------------------------------------
// engine
// ---------------------------------------------------------------------------------------------------
Shared& shared() {
    static Shared s;
    return s;
}

Engine& engine() {
    thread_local Engine e;
    return e;
}


Engine::~Engine() {   // thread exit: errors are ignored (at process exit the runtime may already be gone)
    if (!ready) return;
    if (stream) cudaStreamSynchronize(stream);
    cache.drop_all();
    if (stream) cudaStreamDestroy(stream);
    if (stream2) { cudaStreamSynchronize(stream2); cudaStreamDestroy(stream2); }
    if (mailbox) cudaFreeHost(mailbox);
    ready = false; stream = nullptr; stream2 = nullptr; mailbox = nullptr;   // late frees fall back to the default stream
}

void ensure_engine() {
    Engine& e = engine();
    if (e.ready) {
        cudaSetDevice(e.device);
        return;
    }
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0)
        throw Error(HBSM_E_CUDA, "hbsm_b200: no CUDA device available (this engine has no CPU fallback)");
    int dev = shared().device.load();
    if (dev < 0) {   // first use without hbsm_init: device 0 for the whole process
        int expect = -1;
        shared().device.compare_exchange_strong(expect, 0);
        dev = shared().device.load();
    }
    if (dev >= count) throw Error(HBSM_E_CUDA, "hbsm_b200: device index out of range");
    HB_CUDA(cudaSetDevice(dev));
    cudaDeviceProp p;
    HB_CUDA(cudaGetDeviceProperties(&p, dev));
    if (p.major != 10)
        throw Error(HBSM_E_CUDA, std::string("hbsm_b200: kernels are built for sm_100a only; device is ") + p.name);
    e.device = dev;
    e.sm_count = p.multiProcessorCount;
    e.cc_major = p.major;
    e.cc_minor = p.minor;
    e.name = p.name;
    HB_CUDA(cudaStreamCreateWithFlags(&e.stream, cudaStreamNonBlocking));
    HB_CUDA(cudaStreamCreateWithFlags(&e.stream2, cudaStreamNonBlocking));
    cudaMemPool_t pool;
    HB_CUDA(cudaDeviceGetDefaultMemPool(&pool, dev));
    uint64_t thr = UINT64_MAX;
    HB_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    HB_CUDA(cudaHostAlloc((void**)&e.mailbox, 256 * sizeof(uint64_t), cudaHostAllocMapped));   // slots: 0-1 read_scalars, 2 root norm, 4 find, 8..8+64 halo edges
    e.ready = true;
}

// ---------------------------------------------------------------------------------------------------
// Matrix basics
// ---------------------------------------------------------------------------------------------------
void Matrix::clear() {  // H:614
    keys.release(); tiles.release(); norms.release();
    invalidate_indices();
    drop_tasks();
    L = 0; M = 0; N = 0; sized = false;
    halo_cap = 0; n_halo = 0;
    root_norm_cached = 0.0;
    pub.reset();
}

void Matrix::resize(int m, int n) {  // H:544
    if (b <= 0) throw Error(HBSM_E_ARG, "hbsm_b200: blocksize must be set before resize");
    if (m < 0 || n < 0) throw Error(HBSM_E_ARG, "hbsm_b200: negative dimension");
    clear();
    M = m; N = n; sized = true;
    if (m <= b && n <= b) {  // lowest level: a single zero-filled leaf, H:553-558
        DevBuf<uint64_t> k(1);
        k.zero();
        DevBuf<char> t(tile_bytes());
        t.zero();
        set_table(std::move(k), std::move(t), 1);
    }
}

void Matrix::set_table(DevBuf<uint64_t>&& k, DevBuf<char>&& t, size_t count) {
    keys = std::move(k);
    tiles = std::move(t);
    L = count;
    halo_cap = 0; n_halo = 0;
    pub.reset();
    norms.alloc(std::max<size_t>(count, 1) * esize());
    norms.zero();
    invalidate_indices();
}

// ---------------------------------------------------------------------------------------------------
// halo tail (multi-GPU op(B) operand): grow the three arrays once, hand out pointers to the tail
// ---------------------------------------------------------------------------------------------------
void reserve_halo(Matrix& A, size_t cap, uint64_t** d_keys, void** d_norms, void** d_tiles) {
    if (!A.sized) throw Error(HBSM_E_ARG, "hbsm_b200: halo reserve on an unsized matrix");
    ensure_engine();
    if (A.vdepth() == 0 && cap > 0) throw Error(HBSM_E_ARG, "hbsm_b200: a single-leaf matrix has no halo");
    if (cap > A.halo_cap) {
        const size_t tot = A.L + cap;
        DevBuf<uint64_t> k(tot);
        DevBuf<char> t(tot * A.tile_bytes()), nr(tot * A.esize());
        if (A.L) {
            HB_CUDA(cudaMemcpyAsync(k.p, A.keys.p, A.L * sizeof(uint64_t), cudaMemcpyDeviceToDevice, engine().stream));
            HB_CUDA(cudaMemcpyAsync(t.p, A.tiles.p, A.L * A.tile_bytes(), cudaMemcpyDeviceToDevice, engine().stream));
            HB_CUDA(cudaMemcpyAsync(nr.p, A.norms.p, A.L * A.esize(), cudaMemcpyDeviceToDevice, engine().stream));
        }
        A.keys = std::move(k); A.tiles = std::move(t); A.norms = std::move(nr);
        A.halo_cap = cap;
        sync_stream();
    }
    A.n_halo = 0;
    A.ext_by_row.reset(); A.ext_by_col.reset();
    if (d_keys) *d_keys = A.keys.p + A.L;
    if (d_norms) *d_norms = A.norms.p + A.L * A.esize();
    if (d_tiles) *d_tiles = A.tiles.p + A.L * A.tile_bytes();
}

void commit_halo(Matrix& A, size_t n_halo) {
    if (n_halo > A.halo_cap) throw Error(HBSM_E_ARG, "hbsm_b200: halo commit beyond the reserved capacity");
    A.n_halo = n_halo;
    A.ext_by_row.reset(); A.ext_by_col.reset();
}

namespace {

template <typename T> struct DT;
template <> struct DT<double> {
    static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
    static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
};
template <> struct DT<float> {
    static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
    static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
};

inline unsigned blocks_for(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// lower_bound over sorted keys; returns index or -1 if absent
__device__ __forceinline__ long long find_key(const uint64_t* __restrict__ keys, size_t n, uint64_t key) {
    size_t lo = 0, hi = n;
    while (lo < hi) {
        size_t mid = (lo + hi) >> 1;
        if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    return (lo < n && keys[lo] == key) ? (long long)lo : -1;
}

// ---- assembly kernels ----
// element key = tile Morton key * b^2 + column-major offset inside the tile; flag bit 0: out of [0,M)x[0,N)
__global__ void k_coo_keys(const int* __restrict__ rows, const int* __restrict__ cols, size_t n, int b, int M, int N,
                           long long vsize, uint64_t* __restrict__ keys, uint32_t* __restrict__ idx,
                           unsigned* __restrict__ flags) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int r = rows[i], c = cols[i];
    idx[i] = (uint32_t)i;
    bool inside = r >= 0 && r < M && c >= 0 && c < N;
    bool invirt = r >= 0 && r < vsize && c >= 0 && c < vsize;
    if (!inside) atomicOr(flags, invirt ? 1u : 3u);
    if (!invirt) { keys[i] = ~0ull; return; }   // dropped by the 4-way split of H:755-789
    uint64_t tk = morton_encode((uint32_t)(r / b), (uint32_t)(c / b));
    keys[i] = tk * (uint64_t)b * (uint64_t)b + (uint64_t)(c % b) * b + (uint64_t)(r % b);
}

__global__ void k_flag_tile_heads(const uint64_t* __restrict__ ekeys, size_t n, uint64_t bb, uint32_t* __restrict__ head) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t k = ekeys[i];
    if (k == ~0ull) { head[i] = 0; return; }
    head[i] = (i == 0 || ekeys[i - 1] / bb != k / bb) ? 1u : 0u;
}

__global__ void k_emit_tile_keys(const uint64_t* __restrict__ ekeys, size_t n, uint64_t bb,
                                 const uint32_t* __restrict__ head, const uint64_t* __restrict__ pos,
                                 uint64_t* __restrict__ tkeys) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (head[i]) tkeys[pos[i]] = ekeys[i] / bb;
}

// one thread per sorted element; run heads fold their run sequentially in input order (stable sort), so duplicates
// are summed exactly as the reference's leaf loop does (H:703-721): x = ((x + v1) + v2) ... / x = max(x, v)
template <typename T>
__global__ void k_scatter_runs(const uint64_t* __restrict__ ekeys, const uint32_t* __restrict__ eidx, size_t n,
                               uint64_t bb, int b, int M, int N, const int* __restrict__ rows, const int* __restrict__ cols,
                               const T* __restrict__ vals, const uint64_t* __restrict__ tkeys, size_t L,
                               T* __restrict__ tiles, int use_max) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t k = ekeys[i];
    if (k == ~0ull) return;
    if (i > 0 && ekeys[i - 1] == k) return;
    long long t = find_key(tkeys, L, k / bb);
    if (t < 0) return;
    T* dst = tiles + (size_t)t * bb + (k % bb);
    T x = *dst;
    for (size_t j = i; j < n && ekeys[j] == k; ++j) {
        uint32_t e = eidx[j];
        if (rows[e] >= M || cols[e] >= N) continue;   // padding of a boundary leaf, H:708
        T v = vals[e];
        if (use_max) x = (v > x) ? v : x;
        else x = DT<T>::add(x, v);
    }
    *dst = x;
}

// ---- readback kernels ----
template <typename T>
__global__ void k_get_values(const uint64_t* __restrict__ tkeys, size_t L, const T* __restrict__ tiles, int b,
                             const int* __restrict__ rows, const int* __restrict__ cols, size_t n, T* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int r = rows[i], c = cols[i];
    long long t = find_key(tkeys, L, morton_encode((uint32_t)(r / b), (uint32_t)(c / b)));
    out[i] = t < 0 ? (T)0 : tiles[(size_t)t * b * b + (size_t)(c % b) * b + (r % b)];   // absent child => 0, H:878
}

template <typename T>
__global__ void __launch_bounds__(256) k_tile_nnz(const T* __restrict__ tiles, size_t bb, uint32_t* __restrict__ cnt) {
    __shared__ uint32_t s[8];
    const T* t = tiles + (size_t)blockIdx.x * bb;
    uint32_t c = 0;
    for (size_t i = threadIdx.x; i < bb; i += blockDim.x) c += (fabs((double)t[i]) > 0.0) ? 1u : 0u;
    for (int d = 16; d > 0; d >>= 1) c += __shfl_down_sync(0xffffffffu, c, d);
    if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (unsigned w = 0; w < blockDim.x / 32; ++w) tot += s[w];
        cnt[blockIdx.x] = tot;
    }
}

// ordered compaction of one tile: storage (column-major) order, only fabs(v) > 0 (H:1051-1063)
template <typename T>
__global__ void __launch_bounds__(256) k_tile_gather(const uint64_t* __restrict__ tkeys, const T* __restrict__ tiles,
                                                      int b, const uint64_t* __restrict__ offs, int* __restrict__ rows,
                                                      int* __restrict__ cols, T* __restrict__ vals) {
    __shared__ uint32_t wsum[8];
    __shared__ uint32_t carry;
    const size_t bb = (size_t)b * b;
    const T* t = tiles + (size_t)blockIdx.x * bb;
    uint64_t key = tkeys[blockIdx.x];
    int r0 = (int)morton_row(key) * b, c0 = (int)morton_col(key) * b;
    uint64_t base = offs[blockIdx.x];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (size_t s = 0; s < bb; s += blockDim.x) {
        size_t i = s + threadIdx.x;
        T v = i < bb ? t[i] : (T)0;
        bool nz = i < bb && fabs((double)v) > 0.0;
        unsigned bal = __ballot_sync(0xffffffffu, nz);
        if (lane == 0) wsum[warp] = __popc(bal);
        __syncthreads();
        uint32_t before = carry;
        for (unsigned w = 0; w < warp; ++w) before += wsum[w];
        if (nz) {
            uint64_t p = base + before + __popc(bal & ((1u << lane) - 1u));
            rows[p] = r0 + (int)(i % b);
            cols[p] = c0 + (int)(i / b);
            vals[p] = v;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tot = 0;
            for (unsigned w = 0; w < blockDim.x / 32; ++w) tot += wsum[w];
            carry += tot;
        }
        __syncthreads();
    }
}

// ---- norms ----
// One lane per leaf does the reference's strictly sequential sum_i fl(s + fl(x_i*x_i)) (H:646-652) -- a tree or
// shuffle reduction would change the last ulp and could flip a borderline SpAMM test.  A warp owns 32 leaves and
// streams them in 256-byte coalesced segments through shared memory so HBM sees full-line requests.
template <typename T, int SEG /* elements per leaf per stage */>
__global__ void __launch_bounds__(128) k_leaf_norms(const T* __restrict__ tiles, size_t L, size_t bb, T* __restrict__ out) {
    constexpr int WARPS = 4;
    __shared__ T buf[WARPS][32][SEG + 1];
    const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    size_t leaf0 = ((size_t)blockIdx.x * WARPS + warp) * 32;
    if (leaf0 >= L) return;
    unsigned nleaf = (unsigned)min((size_t)32, L - leaf0);
    const size_t nseg = (bb + SEG - 1) / SEG;
    T acc = 0;
    T reg[SEG];   // staged next segment: reg[j] = element (j*32+lane) of the 32xSEG stage in leaf-major order
    auto load = [&](size_t sidx) {
#pragma unroll
        for (int j = 0; j < SEG; ++j) {
            unsigned flat = j * 32 + lane;
            unsigned lf = flat / SEG, e = flat % SEG;
            size_t pos = sidx * SEG + e;
            reg[j] = (lf < nleaf && pos < bb) ? tiles[(leaf0 + lf) * bb + pos] : (T)0;
        }
    };
    auto stash = [&]() {
#pragma unroll
        for (int j = 0; j < SEG; ++j) {
            unsigned flat = j * 32 + lane;
            buf[warp][flat / SEG][flat % SEG] = reg[j];
        }
    };
    load(0);
    for (size_t s = 0; s < nseg; ++s) {
        stash();
        __syncwarp();
        if (s + 1 < nseg) load(s + 1);
        size_t rem = bb - s * SEG;
        int cnt = rem < (size_t)SEG ? (int)rem : SEG;
        if (cnt == SEG) {
#pragma unroll
            for (int e = 0; e < SEG; ++e) { T x = buf[warp][lane][e]; acc = DT<T>::add(acc, DT<T>::mul(x, x)); }
        } else {
            for (int e = 0; e < cnt; ++e) { T x = buf[warp][lane][e]; acc = DT<T>::add(acc, DT<T>::mul(x, x)); }
        }
        __syncwarp();
    }
    if (lane < nleaf) out[leaf0 + lane] = acc;
}

// Bottom-up refresh of H:3918-3923 / H:656-662: every node = sum of its existing children in child order 0..3, starting
// from 0, in Treal.  Adding an absent child as +0.0 is exact (norms are non-negative), so a level can be folded DENSELY:
// parent p = ((c[4p] + c[4p+1]) + c[4p+2]) + c[4p+3].  The leaves below one level-m ancestor are one contiguous key range
// (Morton order), so a block finds the range of its ancestor by binary search, scatters the leaf norms into a dense
// 4^m-slot shared-memory table (m <= 6) and folds m levels there; the last block to finish folds the remaining <= 6 top
// levels the same way and posts the root to the engine's host mailbox as a double.  One launch, every SM busy, no
// scratch proportional to L.  Only the root is kept (inner-node norms are never consulted: the prune rule is flat).
template <typename T>
__device__ __forceinline__ void fold_dense_smem(T* s, uint32_t cnt) {
    // in place: after each round the first cnt/4 slots hold the parents
    for (; cnt > 1; cnt >>= 2) {
        const uint32_t np = cnt >> 2;
        T v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t p = threadIdx.x + j * blockDim.x;
            if (p < np) v[j] = DT<T>::add(DT<T>::add(DT<T>::add(s[4 * p], s[4 * p + 1]), s[4 * p + 2]), s[4 * p + 3]);
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t p = threadIdx.x + j * blockDim.x;
            if (p < np) s[p] = v[j];
        }
        __syncthreads();
    }
}
__device__ __forceinline__ size_t lower_bound_key(const uint64_t* __restrict__ keys, size_t n, uint64_t key) {
    size_t lo = 0, hi = n;
    while (lo < hi) {
        const size_t mid = (lo + hi) >> 1;
        if (keys[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}
template <typename T>
__global__ void __launch_bounds__(256) k_fold_dense(const uint64_t* __restrict__ keys, const T* __restrict__ vals, size_t n,
                                                    int depth, int m, T* top, unsigned* done_counter,
                                                    volatile uint64_t* mailbox_slot) {
    __shared__ T s[4096];
    __shared__ size_t range_s[2];
    __shared__ unsigned last_s;
    const uint32_t n_top = 1u << (2 * (depth - m));   // <= 4096
    const uint32_t slots = 1u << (2 * m);             // <= 4096
    for (uint32_t a = blockIdx.x; a < n_top; a += gridDim.x) {
        if (threadIdx.x < 2) range_s[threadIdx.x] = lower_bound_key(keys, n, (uint64_t)(a + threadIdx.x) << (2 * m));
        __syncthreads();
        const size_t lo = range_s[0], hi = range_s[1];
        if (lo < hi) {
            for (uint32_t i = threadIdx.x; i < slots; i += blockDim.x) s[i] = (T)0;
            __syncthreads();
            for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) s[keys[i] & (uint64_t)(slots - 1)] = vals[i];
            __syncthreads();
            fold_dense_smem<T>(s, slots);
            if (threadIdx.x == 0) top[a] = s[0];
        } else if (threadIdx.x == 0) {
            top[a] = (T)0;
        }
        __syncthreads();
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last_s = (atomicAdd(done_counter, 1u) == gridDim.x - 1) ? 1u : 0u;
    __syncthreads();
    if (!last_s) return;
    __threadfence();
    const volatile T* vt = top;
    for (uint32_t i = threadIdx.x; i < n_top; i += blockDim.x) s[i] = vt[i];
    __syncthreads();
    fold_dense_smem<T>(s, n_top);
    if (threadIdx.x == 0) {
        *mailbox_slot = (uint64_t)__double_as_longlong((double)s[0]);
        __threadfence_system();
    }
}

// Fallback for block grids deeper than 12 levels (side > 4096): the same refresh in ONE block over sparse (key, value)
// tables, level by level (head-flag compaction; heads add up their <= 4 followers), ping-ponging between two scratch
// tables of L entries each -- a level is only bounded by the level below it, there is no halving guarantee.
template <typename T>
__global__ void __launch_bounds__(1024) k_fold_root(const uint64_t* __restrict__ keys0, const T* __restrict__ vals0, size_t n0,
                                                    int depth, uint64_t* ka, T* va, uint64_t* kb, T* vb,
                                                    volatile uint64_t* mailbox_slot) {
    constexpr int ITEMS = 4;                 // consecutive entries per thread and round: 4096 per round, 3 barriers
    __shared__ uint32_t warp_cnt[33];
    __shared__ size_t carry_s;
    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint64_t* kin = keys0;
    const T* vin = vals0;
    size_t n = n0;
    uint64_t* kout = ka;
    T* vout = va;
    for (int l = 0; l < depth; ++l) {
        if (tid == 0) carry_s = 0;
        __syncthreads();
        for (size_t base = 0; base < n; base += 1024 * ITEMS) {
            const size_t i0 = base + (size_t)tid * ITEMS;
            uint64_t pk[ITEMS];
            bool head[ITEMS];
            uint64_t prev = (i0 > 0 && i0 - 1 < n) ? (kin[i0 - 1] >> 2) : ~0ull;
            uint32_t cnt = 0;
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                const size_t i = i0 + j;
                pk[j] = i < n ? (kin[i] >> 2) : ~0ull;
                head[j] = i < n && (i == 0 || pk[j] != prev);
                prev = pk[j];
                cnt += head[j] ? 1u : 0u;
            }
            uint32_t incl = cnt;              // block-wide exclusive scan of the per-thread head counts
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
                if ((int)lane >= d) incl += o;
            }
            if (lane == 31) warp_cnt[warp] = incl;
            __syncthreads();
            if (warp == 0) {
                const uint32_t v = warp_cnt[lane];
                uint32_t wi = v;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t o = __shfl_up_sync(0xffffffffu, wi, d);
                    if ((int)lane >= d) wi += o;
                }
                warp_cnt[lane] = wi - v;
                if (lane == 31) warp_cnt[32] = wi;
            }
            __syncthreads();
            size_t pos = carry_s + warp_cnt[warp] + (incl - cnt);
#pragma unroll
            for (int j = 0; j < ITEMS; ++j) {
                if (head[j]) {
                    T sum = 0;
                    for (size_t q = i0 + j; q < n && (kin[q] >> 2) == pk[j]; ++q) sum = DT<T>::add(sum, vin[q]);
                    kout[pos] = pk[j];
                    vout[pos] = sum;
                    ++pos;
                }
            }
            __syncthreads();
            if (tid == 0) carry_s += warp_cnt[32];
        }
        __syncthreads();
        n = carry_s;
        kin = kout;
        vin = vout;
        kout = (kout == ka) ? kb : ka;
        vout = (vout == va) ? vb : va;
        __syncthreads();
    }
    if (tid == 0) {
        *mailbox_slot = (uint64_t)__double_as_longlong((double)vin[0]);
        __threadfence_system();
    }
}

// ---- line index ----
__global__ void k_line_keys(const uint64_t* __restrict__ keys, size_t n, int by_col, int dbits, uint64_t* __restrict__ skey,
                            uint32_t* __restrict__ idx) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t r = morton_row(keys[i]), c = morton_col(keys[i]);
    uint32_t line = by_col ? c : r, other = by_col ? r : c;
    skey[i] = ((uint64_t)line << dbits) | other;
    idx[i] = (uint32_t)i;
}
__global__ void k_line_ptr(const uint64_t* __restrict__ skey, size_t n, int dbits, uint32_t n_lines,
                           uint32_t* __restrict__ ptr, uint32_t* __restrict__ other) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t line = (uint32_t)(skey[i] >> dbits);
    other[i] = (uint32_t)(skey[i] & ((1ull << dbits) - 1ull));
    uint32_t prev = i == 0 ? 0u : (uint32_t)(skey[i - 1] >> dbits) + 1u;
    for (uint32_t l = prev; l <= line; ++l) ptr[l] = (uint32_t)i;   // lines (prev_line, line] start here
    if (i == n - 1)
        for (uint32_t l = line + 1; l <= n_lines; ++l) ptr[l] = (uint32_t)n;
}

// ---- structure ops ----
// merge-union of two sorted key lists: flags per output slot which inputs contribute
__global__ void k_union_mark(const uint64_t* __restrict__ ka, size_t na, const uint64_t* __restrict__ kb, size_t nb,
                             uint32_t* __restrict__ keep_b /* 1 if kb[i] not in ka */) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb) return;
    keep_b[i] = find_key(ka, na, kb[i]) < 0 ? 1u : 0u;
}
// position of every A tile and of every B-only tile in the union: rankA(i) = i + #(B-only keys < ka[i]) etc.
__global__ void k_union_pos_a(const uint64_t* __restrict__ ka, size_t na, const uint64_t* __restrict__ kb, size_t nb,
                              const uint64_t* __restrict__ bonly_prefix, uint64_t* __restrict__ ukeys,
                              uint32_t* __restrict__ src_a, uint32_t* __restrict__ src_b) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= na) return;
    uint64_t key = ka[i];
    size_t lo = 0, hi = nb;
    while (lo < hi) { size_t mid = (lo + hi) >> 1; if (kb[mid] < key) lo = mid + 1; else hi = mid; }
    size_t p = i + bonly_prefix[lo];
    ukeys[p] = key;
    src_a[p] = (uint32_t)i;
    src_b[p] = (lo < nb && kb[lo] == key) ? (uint32_t)lo : 0xffffffffu;
}
__global__ void k_union_pos_b(const uint64_t* __restrict__ ka, size_t na, const uint64_t* __restrict__ kb, size_t nb,
                              const uint32_t* __restrict__ keep_b, const uint64_t* __restrict__ bonly_prefix,
                              uint64_t* __restrict__ ukeys, uint32_t* __restrict__ src_a, uint32_t* __restrict__ src_b) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb || !keep_b[i]) return;
    uint64_t key = kb[i];
    size_t lo = 0, hi = na;
    while (lo < hi) { size_t mid = (lo + hi) >> 1; if (ka[mid] < key) lo = mid + 1; else hi = mid; }
    size_t p = lo + bonly_prefix[i];
    ukeys[p] = key;
    src_a[p] = 0xffffffffu;
    src_b[p] = (uint32_t)i;
}

// C tile = A tile + B tile (fl(a+b), H:1674-1677), or a copy when only one exists (the reference aliases, H:1699).
// 16-byte vectorised when the tile is a multiple of 16 bytes; one CTA streams a slice of one tile.
template <typename T>
__global__ void __launch_bounds__(256) k_add_tiles(const T* __restrict__ ta, const T* __restrict__ tb,
                                                    const uint32_t* __restrict__ src_a, const uint32_t* __restrict__ src_b,
                                                    size_t bb, T* __restrict__ tc) {
    const size_t t = blockIdx.x;
    const uint32_t ia = src_a[t], ib = src_b[t];
    T* c = tc + t * bb;
    const T* a = ia != 0xffffffffu ? ta + (size_t)ia * bb : nullptr;
    const T* b = ib != 0xffffffffu ? tb + (size_t)ib * bb : nullptr;
    constexpr int V = 16 / sizeof(T);
    if ((bb % V) == 0) {
        const size_t nv = bb / V;
        const int4* a4 = reinterpret_cast<const int4*>(a);
        const int4* b4 = reinterpret_cast<const int4*>(b);
        int4* c4 = reinterpret_cast<int4*>(c);
        for (size_t i = (size_t)blockIdx.y * blockDim.x + threadIdx.x; i < nv; i += (size_t)gridDim.y * blockDim.x) {
            if (a && b) {
                int4 x = __ldg(a4 + i), y = __ldg(b4 + i);
                T* xp = reinterpret_cast<T*>(&x);
                const T* yp = reinterpret_cast<const T*>(&y);
#pragma unroll
                for (int j = 0; j < V; ++j) xp[j] = DT<T>::add(xp[j], yp[j]);
                c4[i] = x;
            } else {
                c4[i] = __ldg((a ? a4 : b4) + i);
            }
        }
    } else {
        for (size_t i = (size_t)blockIdx.y * blockDim.x + threadIdx.x; i < bb; i += (size_t)gridDim.y * blockDim.x)
            c[i] = (a && b) ? DT<T>::add(a[i], b[i]) : (a ? a[i] : b[i]);
    }
}

// out tile t = transpose of in tile src[t] (through shared memory so both sides are coalesced), H:3748-3752
template <typename T>
__global__ void __launch_bounds__(256) k_transpose_tiles(const T* __restrict__ tin, const uint32_t* __restrict__ src,
                                                          int b, T* __restrict__ tout) {
    __shared__ T s[32][33];
    const size_t bb = (size_t)b * b;
    const T* in = tin + (size_t)src[blockIdx.x] * bb;
    T* out = tout + (size_t)blockIdx.x * bb;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    for (int c0 = 0; c0 < b; c0 += 32)
        for (int r0 = 0; r0 < b; r0 += 32) {
            for (int j = ty; j < 32; j += 8) {
                int r = r0 + tx, c = c0 + j;
                s[j][tx] = (r < b && c < b) ? in[(size_t)c * b + r] : (T)0;
            }
            __syncthreads();
            for (int j = ty; j < 32; j += 8) {
                int r = c0 + tx, c = r0 + j;    // out(r,c) = in(c,r)
                if (r < b && c < b) out[(size_t)c * b + r] = s[tx][j];
            }
            __syncthreads();
        }
}

// same for leaves that are a multiple of 32: NSUB 32x32 sub-blocks per phase, so every thread has 4*NSUB independent loads
// in flight before the first barrier (the one-sub-block-per-phase loop above is latency-bound: 0.43 of the HBM copy rate
// for fp32 tiles, profiles/r01_hbm_stages.md)
template <typename T, int NSUB>
__global__ void __launch_bounds__(256) k_transpose_tiles_wide(const T* __restrict__ tin, const uint32_t* __restrict__ src,
                                                               int b, T* __restrict__ tout) {
    __shared__ T s[NSUB][32][33];
    const size_t bb = (size_t)b * b;
    const T* in = tin + (size_t)src[blockIdx.x] * bb;
    T* out = tout + (size_t)blockIdx.x * bb;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    const int nb = b >> 5, total = nb * nb;
    for (int q0 = 0; q0 < total; q0 += NSUB) {
#pragma unroll
        for (int u = 0; u < NSUB; ++u) {
            const int q = q0 + u;
            if (q < total) {
                const int r0 = (q % nb) * 32, c0 = (q / nb) * 32;
#pragma unroll
                for (int j = ty; j < 32; j += 8) s[u][j][tx] = in[(size_t)(c0 + j) * b + r0 + tx];
            }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < NSUB; ++u) {
            const int q = q0 + u;
            if (q < total) {
                const int r0 = (q % nb) * 32, c0 = (q / nb) * 32;
#pragma unroll
                for (int j = ty; j < 32; j += 8) out[(size_t)(r0 + j) * b + c0 + tx] = s[u][tx][j];   // out(r,c) = in(c,r)
            }
        }
        __syncthreads();
    }
}

__global__ void k_transpose_keys(const uint64_t* __restrict__ keys, size_t n, uint64_t* __restrict__ okeys,
                                 uint32_t* __restrict__ idx) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    okeys[i] = morton_transpose(keys[i]);
    idx[i] = (uint32_t)i;
}

// keep tiles with bi <= bj (H:3515-3559)
__global__ void k_upper_flags(const uint64_t* __restrict__ keys, size_t n, uint32_t* __restrict__ keep) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    keep[i] = morton_row(keys[i]) <= morton_col(keys[i]) ? 1u : 0u;
}
__global__ void k_compact_keys(const uint64_t* __restrict__ keys, size_t n, const uint32_t* __restrict__ keep,
                               const uint64_t* __restrict__ pos, uint64_t* __restrict__ okeys, uint32_t* __restrict__ src) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !keep[i]) return;
    okeys[pos[i]] = keys[i];
    src[pos[i]] = (uint32_t)i;
}
// copy tile src[t] -> t; mode 0 plain copy * alpha (alpha_on), mode 1: diagonal tiles keep only row <= col
template <typename T>
__global__ void __launch_bounds__(256) k_copy_tiles(const T* __restrict__ tin, const uint32_t* __restrict__ src,
                                                     const uint64_t* __restrict__ okeys, int b, int mask_diag,
                                                     int scale, T alpha, T* __restrict__ tout) {
    const size_t bb = (size_t)b * b;
    const size_t si = src ? (size_t)src[blockIdx.x] : (size_t)blockIdx.x;
    const T* in = tin + si * bb;
    T* out = tout + (size_t)blockIdx.x * bb;
    bool diag = false;
    if (mask_diag) { uint64_t k = okeys[blockIdx.x]; diag = morton_row(k) == morton_col(k); }
    for (size_t i = (size_t)blockIdx.y * blockDim.x + threadIdx.x; i < bb; i += (size_t)gridDim.y * blockDim.x) {
        T v = in[i];
        if (diag && (int)(i % b) > (int)(i / b)) v = (T)0;
        if (scale) v = DT<T>::mul(v, alpha);
        out[i] = v;
    }
}

// symmetric expansion of upper storage: S(i,j) = A(min,max).  Output tile t has source tile src[t]; flag bit0 =
// take it transposed (strict-lower tile), bit1 = diagonal tile (mirror the upper part onto the lower part).
template <typename T>
__global__ void __launch_bounds__(256) k_sym_tiles(const T* __restrict__ tin, const uint32_t* __restrict__ src,
                                                    const uint32_t* __restrict__ flag, int b, T* __restrict__ tout) {
    const size_t bb = (size_t)b * b;
    const T* in = tin + (size_t)src[blockIdx.x] * bb;
    T* out = tout + (size_t)blockIdx.x * bb;
    const uint32_t f = flag[blockIdx.x];
    for (size_t i = threadIdx.x; i < bb; i += blockDim.x) {
        int r = (int)(i % b), c = (int)(i / b);
        T v;
        if (f & 2u) { int rr = r < c ? r : c, cc = r < c ? c : r; v = in[(size_t)cc * b + rr]; }
        else if (f & 1u) v = in[(size_t)r * b + c];
        else v = in[i];
        out[i] = v;
    }
}
__global__ void k_sym_keys(const uint64_t* __restrict__ keys, size_t n, uint64_t* __restrict__ okeys,
                           uint32_t* __restrict__ osrc, uint32_t* __restrict__ valid) {
    // input tile i with bi<bj yields (bi,bj) and (bj,bi); bi==bj yields itself; bi>bj (never stored) is ignored
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t r = morton_row(keys[i]), c = morton_col(keys[i]);
    okeys[2 * i] = keys[i];               osrc[2 * i] = (uint32_t)i;     valid[2 * i] = r <= c ? 1u : 0u;
    okeys[2 * i + 1] = morton_transpose(keys[i]); osrc[2 * i + 1] = (uint32_t)i; valid[2 * i + 1] = r < c ? 1u : 0u;
}
__global__ void k_sym_compact(const uint64_t* __restrict__ keys2, const uint32_t* __restrict__ src2,
                              const uint32_t* __restrict__ valid, const uint64_t* __restrict__ pos, size_t n2,
                              uint64_t* __restrict__ okeys, uint32_t* __restrict__ osrc_packed) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n2 || !valid[i]) return;
    okeys[pos[i]] = keys2[i];
    osrc_packed[pos[i]] = (src2[i] << 1) | (uint32_t)(i & 1);   // low bit: mirrored copy
}
__global__ void k_sym_unpack(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ packed, size_t n,
                             uint32_t* __restrict__ src, uint32_t* __restrict__ flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    src[i] = packed[i] >> 1;
    uint32_t f = packed[i] & 1u;
    if (morton_row(keys[i]) == morton_col(keys[i])) f |= 2u;
    flag[i] = f;
}

template <typename T>
__global__ void __launch_bounds__(256) k_mask_diag(const uint64_t* __restrict__ keys, int b, T* __restrict__ tiles) {
    uint64_t k = keys[blockIdx.x];
    if (morton_row(k) != morton_col(k)) return;
    const size_t bb = (size_t)b * b;
    T* t = tiles + (size_t)blockIdx.x * bb;
    for (size_t i = threadIdx.x; i < bb; i += blockDim.x)
        if ((int)(i % b) > (int)(i / b)) t[i] = (T)0;
}

// ---- banded exponential-decay generator (SURVEY 8d): a_ij = (0.5 + 0.5 u(seed,i,j)) exp(-lambda |i-j|), |i-j| <= W ----
__host__ __device__ inline double hash_u01(uint64_t seed, uint64_t i, uint64_t j) {
    uint64_t h = splitmix64(seed ^ splitmix64(i * 0x100000001B3ull + splitmix64(j)));
    return (double)(h >> 11) * (1.0 / 9007199254740992.0);
}
__global__ void k_decay_keys(uint32_t lo, uint32_t hi, uint32_t g, uint32_t wb, uint64_t* __restrict__ keys) {
    // tile rows [lo,hi), per row columns [bi-wb, bi+wb] clipped; enumerated densely, invalid = ~0
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t span = 2 * (size_t)wb + 1;
    if (i >= (size_t)(hi - lo) * span) return;
    uint32_t bi = lo + (uint32_t)(i / span);
    long long bj = (long long)bi - wb + (long long)(i % span);
    keys[i] = (bj < 0 || bj >= g) ? ~0ull : morton_encode(bi, (uint32_t)bj);
}
template <typename T>
__global__ void __launch_bounds__(256) k_decay_fill(const uint64_t* __restrict__ keys, int b, int n, int W,
                                                     const double* __restrict__ table, uint64_t seed, int symmetric,
                                                     T* __restrict__ tiles) {
    const size_t bb = (size_t)b * b;
    uint64_t k = keys[blockIdx.x];
    long long r0 = (long long)morton_row(k) * b, c0 = (long long)morton_col(k) * b;
    T* t = tiles + (size_t)blockIdx.x * bb;
    for (size_t i = threadIdx.x; i < bb; i += blockDim.x) {
        long long r = r0 + (long long)(i % b), c = c0 + (long long)(i / b);
        long long d = r > c ? r - c : c - r;
        double v = 0.0;
        if (r < n && c < n && d <= W) {
            uint64_t hi_ = symmetric ? (uint64_t)(r < c ? r : c) : (uint64_t)r;
            uint64_t hj_ = symmetric ? (uint64_t)(r < c ? c : r) : (uint64_t)c;
            v = (0.5 + 0.5 * hash_u01(seed, hi_, hj_)) * table[d];
        }
        t[i] = (T)v;
    }
}

// frob_block_trunc (H:4904-4943): a subtree is dropped iff its (recomputed) norm^2 < trunc^2.  A node's norm^2 is a sum of
// non-negative child norm^2 with monotone rounding, so a leaf survives iff its OWN norm^2 >= trunc^2 -- the flat rule.
__global__ void k_trunc_flags(const void* __restrict__ norms, size_t n, int is_f64, double t2d, float t2f, uint32_t* __restrict__ keep) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool drop = is_f64 ? (reinterpret_cast<const double*>(norms)[i] < t2d) : (reinterpret_cast<const float*>(norms)[i] < t2f);
    keep[i] = drop ? 0u : 1u;
}

// quadrant extraction / assembly (used by the recursive inv_chol driver, H:3110): child q of the root <-> leaves whose
// leading key digit is q, re-keyed one level down / up.  Tiles are copied (the reference aliases subtrees by shared_ptr).
__global__ void k_rekey(const uint64_t* __restrict__ in, size_t n, uint64_t mask, uint64_t add, uint64_t* __restrict__ out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (in[i] & mask) | add;
}


// Leaf step of inv_chol (H:3118-3147): Z = inverse Cholesky factor of one dense SPD leaf (upper triangular, Z^T A Z = I) by
// the reference's column recurrence -- column i starts as e_i, is made A-orthogonal to the finished columns j < i one after
// the other (the order matters: each projection sees the previous update) and is normalised in the A-norm.  One block; thread
// k owns row k of the column in flight; the A-inner products are block reductions (not the reference's sequential sum: the
// result agrees to rounding, the reference's own tests ask for 1e-10).
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* red) {
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    const int w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();                      // red[] of the previous reduction has been read by everyone
    if ((threadIdx.x & 31) == 0) red[w] = v;
    __syncthreads();
    T s = 0;
    for (int i = 0; i < nw; ++i) s += red[i];
    return s;
}
template <typename T>
__global__ void __launch_bounds__(256) k_leaf_inv_chol(const T* __restrict__ a, int b, int n, T* __restrict__ z) {
    __shared__ T red[8];
    const int k = threadIdx.x;
    const bool live = k < n;
    for (int i = 0; i < n; ++i) {
        T zi = (live && k == i) ? (T)1 : (T)0;
        for (int j = 0; j < i; ++j) {
            // R = sum_k A(j,k) * zi[k], times Z(j,j); column i loses its component along column j
            T R = block_sum<T>(live ? a[(size_t)k * b + j] * zi : (T)0, red);
            R *= z[(size_t)j * b + j];
            if (live) zi -= z[(size_t)j * b + k] * R;
        }
        T R = block_sum<T>(live ? a[(size_t)k * b + i] * zi : (T)0, red);
        R = sqrt((T)1 / R);
        if (live) z[(size_t)i * b + k] = zi * R;
        __syncthreads();                  // column i is read (diagonal and entries) by the following columns
        __threadfence_block();
    }
}

template <typename F>
void dispatch(int dtype, F&& f) {
    if (dtype == HBSM_F64) f((double)0);
    else f((float)0);
}

int key_bits_for(const Matrix& A) { return std::max(1, 2 * A.vdepth()); }

}  // namespace

// compact helper: exclusive scan of flags -> positions, returns total (synchronises)
size_t scan_flags(const DevBuf<uint32_t>& flags, size_t n, DevBuf<uint64_t>& pos) {
    pos.alloc(n + 1);
    exclusive_scan_u32(flags.p, pos.p, n);
    uint64_t total = 0;
    HB_CUDA(cudaMemcpyAsync(&total, pos.p + n, sizeof(uint64_t), cudaMemcpyDeviceToHost, engine().stream));
    sync_stream();
    return (size_t)total;
}

// ---------------------------------------------------------------------------------------------------
// assembly
// ---------------------------------------------------------------------------------------------------
void assign_coo(Matrix& A, size_t n, const int* rows, const int* cols, const void* vals, bool use_max, bool checked) {
    if (!A.sized) throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: index outside matrix boundaries.");
    if (n == 0) return;   // H:679
    if (n >= 0xffffffffull) throw Error(HBSM_E_ARG, "hbsm_b200: more than 2^32-1 triplets in one assign call");
    ensure_engine();
    const int depth = A.vdepth();
    const long long vsize = (long long)A.b << depth;
    const uint64_t bb = A.tile_elems();
    DevBuf<int> d_rows(n), d_cols(n);
    DevBuf<char> d_vals(n * A.esize());
    d_rows.upload(rows, n);
    d_cols.upload(cols, n);
    HB_CUDA(cudaMemcpyAsync(d_vals.p, vals, n * A.esize(), cudaMemcpyHostToDevice, engine().stream));
    DevBuf<uint64_t> ekeys(n);
    DevBuf<uint32_t> eidx(n);
    DevBuf<unsigned> flags(1);
    flags.zero();
    HB_LAUNCH(k_coo_keys, blocks_for(n, 256), 256, 0, d_rows.p, d_cols.p, n, A.b, A.M, A.N, vsize, ekeys.p, eidx.p, flags.p);
    unsigned hflags = 0;
    HB_CUDA(cudaMemcpyAsync(&hflags, flags.p, sizeof(unsigned), cudaMemcpyDeviceToHost, engine().stream));
    sync_stream();
    if (hflags && !checked)   // H:682-688
        throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: index outside matrix boundaries.");
    // element keys < vsize^2; dropped elements (~0) sort to the end because the sort covers all 64 bits in that case
    int bits = 1;
    while (bits < 64 && (1ull << bits) < (uint64_t)vsize * (uint64_t)vsize) ++bits;
    if (hflags & 2u) bits = 64;
    radix_sort_pairs(ekeys.p, eidx.p, n, bits);
    DevBuf<uint32_t> head(n);
    HB_LAUNCH(k_flag_tile_heads, blocks_for(n, 256), 256, 0, ekeys.p, n, bb, head.p);
    DevBuf<uint64_t> pos;
    size_t Lnew = scan_flags(head, n, pos);
    if (Lnew == 0) return;
    DevBuf<uint64_t> tkeys(Lnew);
    HB_LAUNCH(k_emit_tile_keys, blocks_for(n, 256), 256, 0, ekeys.p, n, bb, head.p, pos.p, tkeys.p);

    Matrix fresh;   // where the new elements are folded
    Matrix* target = &A;
    if (depth == 0) {
        // single leaf: += / max onto the existing content (H:703-721), nothing to create
    } else if (A.L == 0) {
        DevBuf<char> t(Lnew * A.tile_bytes());
        t.zero();
        A.set_table(std::move(tkeys), std::move(t), Lnew);
    } else {
        // second assign on a populated tree: the reference throws when a root quadrant is touched twice (H:793)
        std::vector<uint64_t> ka = A.keys.to_host(), kn = tkeys.to_host();
        const int sh = 2 * (depth - 1);
        bool have[4] = {false, false, false, false};
        for (size_t i = 0; i < A.L; ++i) have[(ka[i] >> sh) & 3] = true;   // (a halo tail, if any, is not part of A)
        for (uint64_t k : kn)
            if (have[(k >> sh) & 3]) {
                char msg[160];
                snprintf(msg, sizeof msg,
                         "Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: non-null child%d matrix occured.",
                         (int)((k >> sh) & 3));
                throw_ref(msg);
            }
        fresh.dtype = A.dtype; fresh.b = A.b; fresh.M = A.M; fresh.N = A.N; fresh.sized = true;
        DevBuf<char> t(Lnew * A.tile_bytes());
        t.zero();
        fresh.set_table(std::move(tkeys), std::move(t), Lnew);
        target = &fresh;
    }
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        HB_LAUNCH(k_scatter_runs<T>, blocks_for(n, 256), 256, 0, ekeys.p, eidx.p, n, bb, A.b, A.M, A.N, d_rows.p, d_cols.p,
                  (const T*)d_vals.p, target->keys.p, target->L, (T*)target->tiles.p, use_max ? 1 : 0);
    });
    if (target == &fresh) {
        Matrix merged;
        size_t keep_mults = A.n_mults;
        op_add(A, fresh, merged);   // disjoint tile sets: pure union
        A.keys = std::move(merged.keys); A.tiles = std::move(merged.tiles); A.norms = std::move(merged.norms);
        A.L = merged.L; A.n_mults = keep_mults;
    }
    A.invalidate_indices();
    sync_stream();   // host staging buffers die here
}

void assign_tiles_device(Matrix& A, size_t n_tiles, const uint64_t* d_keys, const void* d_tiles, const void* d_norms) {
    if (!A.sized) throw Error(HBSM_E_ARG, "hbsm_b200: assign_tiles on an unsized matrix");
    ensure_engine();
    if (n_tiles == 0) return;
    if (A.vdepth() == 0) {
        if (n_tiles != 1) throw Error(HBSM_E_ARG, "hbsm_b200: a single-leaf matrix takes exactly one tile");
        HB_CUDA(cudaMemcpyAsync(A.tiles.p, d_tiles, A.tile_bytes(), cudaMemcpyDeviceToDevice, engine().stream));
        if (d_norms) HB_CUDA(cudaMemcpyAsync(A.norms.p, d_norms, A.esize(), cudaMemcpyDeviceToDevice, engine().stream));
        return;
    }
    if (A.L != 0) throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: non-null child0 matrix occured.");
    DevBuf<uint64_t> skeys(n_tiles);
    DevBuf<uint32_t> idx(n_tiles);
    HB_CUDA(cudaMemcpyAsync(skeys.p, d_keys, n_tiles * sizeof(uint64_t), cudaMemcpyDeviceToDevice, engine().stream));
    {
        // reuse k_transpose_keys-style iota: idx[i] = i
        DevBuf<uint64_t> dummy(n_tiles);
        HB_LAUNCH(k_transpose_keys, blocks_for(n_tiles, 256), 256, 0, skeys.p, n_tiles, dummy.p, idx.p);
    }
    radix_sort_pairs(skeys.p, idx.p, n_tiles, key_bits_for(A));
    DevBuf<char> t(n_tiles * A.tile_bytes());
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        dim3 grid((unsigned)n_tiles, (unsigned)std::max<size_t>(1, std::min<size_t>(8, A.tile_elems() / 1024)));
        HB_LAUNCH(k_copy_tiles<T>, grid, 256, 0, (const T*)d_tiles, idx.p, skeys.p, A.b, 0, 0, (T)1, (T*)t.p);
    });
    A.set_table(std::move(skeys), std::move(t), n_tiles);
    if (d_norms) {
        // gather norms in sorted order with the same permutation (1-element "tiles")
        dispatch(A.dtype, [&](auto z) {
            using T = decltype(z);
            HB_LAUNCH(k_copy_tiles<T>, dim3((unsigned)n_tiles, 1), 32, 0, (const T*)d_norms, idx.p, A.keys.p, 1, 0, 0, (T)1,
                      (T*)A.norms.p);
        });
    }
    sync_stream();
}

void assign_tiles_host(Matrix& A, size_t n_tiles, const int* bi, const int* bj, const void* tiles) {
    if (!A.sized) throw Error(HBSM_E_ARG, "hbsm_b200: assign_tiles on an unsized matrix");
    if (n_tiles == 0) return;
    ensure_engine();
    const uint32_t g = A.grid_side();
    std::vector<uint64_t> hk(n_tiles);
    for (size_t i = 0; i < n_tiles; ++i) {
        if (bi[i] < 0 || bj[i] < 0 || (uint32_t)bi[i] >= g || (uint32_t)bj[i] >= g ||
            (long long)bi[i] * A.b >= std::max(A.M, 1) || (long long)bj[i] * A.b >= std::max(A.N, 1))
            throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: index outside matrix boundaries.");
        hk[i] = morton_encode((uint32_t)bi[i], (uint32_t)bj[i]);
    }
    static const bool trace = getenv("HBSM_TRACE_ASSIGN") != nullptr;   // diagnosis: where an upload spends its time
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point b) {
        return std::chrono::duration<double, std::milli>(b - a).count();
    };
    if (trace) {
        cudaMemPool_t pool;
        uint64_t reserved = 0, used = 0, thr = 0;
        cudaDeviceGetMemPool(&pool, engine().device);
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved);
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used);
        cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        fprintf(stderr, "[pool before assign] reserved %.2f GB used %.2f GB release threshold %s\n", reserved / 1e9, used / 1e9,
                thr == UINT64_MAX ? "max" : "NOT max");
    }
    const auto t0 = now();
    DevBuf<uint64_t> dk(n_tiles);
    dk.upload(hk.data(), n_tiles);
    DevBuf<char> dt(n_tiles * A.tile_bytes());
    if (trace) sync_stream();
    const auto t1 = now();
    HB_CUDA(cudaMemcpyAsync(dt.p, tiles, n_tiles * A.tile_bytes(), cudaMemcpyHostToDevice, engine().stream));
    if (trace) sync_stream();
    const auto t2 = now();
    assign_tiles_device(A, n_tiles, dk.p, dt.p, nullptr);
    sync_stream();
    if (trace)
        fprintf(stderr, "[assign_tiles %zu tiles] alloc %.2f ms | H2D %.2f ms (%.1f GB/s) | sort + permute + table %.2f ms\n", n_tiles, ms(t0, t1),
                ms(t1, t2), n_tiles * A.tile_bytes() / ms(t1, t2) / 1e6, ms(t2, now()));
}

// ---------------------------------------------------------------------------------------------------
// readback
// ---------------------------------------------------------------------------------------------------
void get_values(const Matrix& A, size_t n, const int* rows, const int* cols, void* out) {
    if (A.empty()) throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::get_values: empty matrix occured.");
    if (n == 0) return;
    for (size_t i = 0; i < n; ++i)
        if (!(0 <= rows[i] && rows[i] < A.M && 0 <= cols[i] && cols[i] < A.N))
            throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::get_single_value: bad index at highest level.");
    ensure_engine();
    DevBuf<int> dr(n), dc(n);
    dr.upload(rows, n);
    dc.upload(cols, n);
    DevBuf<char> dv(n * A.esize());
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        HB_LAUNCH(k_get_values<T>, blocks_for(n, 256), 256, 0, A.keys.p, A.L, (const T*)A.tiles.p, A.b, dr.p, dc.p, n, (T*)dv.p);
    });
    HB_CUDA(cudaMemcpyAsync(out, dv.p, n * A.esize(), cudaMemcpyDeviceToHost, engine().stream));
    sync_stream();
}

// one tile by block coordinates (parity hook: sample C tiles at sizes where exporting everything is too much)
namespace {
__global__ void k_find_one(const uint64_t* __restrict__ keys, size_t n, uint64_t key, volatile uint64_t* mailbox) {
    mailbox[0] = (uint64_t)find_key(keys, n, key);
    __threadfence_system();
}
}  // namespace
bool export_tile(const Matrix& A, uint32_t bi, uint32_t bj, void* host_buf) {
    if (A.empty() || A.L == 0) return false;
    ensure_engine();
    Engine& e = engine();
    HB_LAUNCH(k_find_one, 1, 1, 0, A.keys.p, A.L, A.vdepth() == 0 ? 0ull : morton_encode(bi, bj), e.mailbox + 4);
    sync_stream();
    const long long at = (long long)e.mailbox[4];
    if (at < 0) return false;
    HB_CUDA(cudaMemcpyAsync(host_buf, A.tiles.p + (size_t)at * A.tile_bytes(), A.tile_bytes(), cudaMemcpyDeviceToHost, e.stream));
    sync_stream();
    return true;
}

// Order-independent checksum of the executed-product set recorded on C (parity hook): sum over products of
// splitmix64(ci << 42 | cj << 21 | k), modulo 2^64.  Equal sets give equal sums whatever the order or the sharding, so
// the per-rank checksums of a sharded product add up to the single-GPU one.
namespace {
__global__ void __launch_bounds__(256) k_task_checksum(const uint64_t* __restrict__ ckeys, const uint64_t* __restrict__ begin,
                                                        const uint32_t* __restrict__ task_k, size_t n_ctiles,
                                                        unsigned long long* __restrict__ acc) {
    const size_t w = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const unsigned lane = threadIdx.x & 31;
    unsigned long long sum = 0;
    if (w < n_ctiles) {
        const uint64_t key = ckeys[w];
        const uint64_t hi = ((uint64_t)morton_row(key) << 42) | ((uint64_t)morton_col(key) << 21);
        for (uint64_t p = begin[w] + lane; p < begin[w + 1]; p += 32) sum += splitmix64(hi | (uint64_t)task_k[p]);
    }
    for (int d = 16; d > 0; d >>= 1) sum += __shfl_down_sync(0xffffffffu, sum, d);
    if (lane == 0 && sum) atomicAdd(acc, sum);
}
}  // namespace
uint64_t task_checksum(const Matrix& C) {
    if (C.n_tasks == 0 || C.L == 0 || !C.task_begin.p) return 0;
    ensure_engine();
    DevBuf<unsigned long long> acc(1);
    acc.zero();
    HB_LAUNCH(k_task_checksum, blocks_for(C.L * 32, 256), 256, 0, C.keys.p, C.task_begin.p, C.task_k.p, C.L, acc.p);
    return (uint64_t)acc.to_host()[0];
}

// the k's of the products accumulated into C tile (bi, bj), ascending (parity hook); returns their number or -1 if absent
long long tile_tasks(const Matrix& C, uint32_t bi, uint32_t bj, size_t cap, int64_t* k_out) {
    if (C.empty() || C.L == 0 || C.n_tasks == 0 || !C.task_begin.p) return -1;
    ensure_engine();
    Engine& e = engine();
    HB_LAUNCH(k_find_one, 1, 1, 0, C.keys.p, C.L, C.vdepth() == 0 ? 0ull : morton_encode(bi, bj), e.mailbox + 4);
    sync_stream();
    const long long at = (long long)e.mailbox[4];
    if (at < 0) return -1;
    uint64_t be[2];
    HB_CUDA(cudaMemcpyAsync(be, C.task_begin.p + at, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, e.stream));
    sync_stream();
    const size_t n = (size_t)(be[1] - be[0]);
    if (n <= cap && n > 0) {
        std::vector<uint32_t> k(n);
        HB_CUDA(cudaMemcpyAsync(k.data(), C.task_k.p + be[0], n * sizeof(uint32_t), cudaMemcpyDeviceToHost, e.stream));
        sync_stream();
        for (size_t i = 0; i < n; ++i) k_out[i] = (int64_t)k[i];
    }
    return (long long)n;
}

static void tile_nnz_counts(const Matrix& A, DevBuf<uint32_t>& cnt) {
    cnt.alloc(A.L);
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        HB_LAUNCH(k_tile_nnz<T>, (unsigned)A.L, 256, 0, (const T*)A.tiles.p, A.tile_elems(), cnt.p);
    });
}

size_t count_nnz(const Matrix& A) {
    if (A.empty()) throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::get_nnz: empty matrix occured.");
    if (A.L == 0) return 0;
    ensure_engine();
    DevBuf<uint32_t> cnt;
    tile_nnz_counts(A, cnt);
    DevBuf<uint64_t> pos;
    return scan_flags(cnt, A.L, pos);
}

size_t get_all_values(const Matrix& A, size_t cap, int* rows, int* cols, void* vals) {
    if (A.empty() || A.L == 0) return 0;   // H:1047
    ensure_engine();
    DevBuf<uint32_t> cnt;
    tile_nnz_counts(A, cnt);
    DevBuf<uint64_t> pos;
    size_t total = scan_flags(cnt, A.L, pos);
    if (cap < total || total == 0) return total;
    DevBuf<int> dr(total), dc(total);
    DevBuf<char> dv(total * A.esize());
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        HB_LAUNCH(k_tile_gather<T>, (unsigned)A.L, 256, 0, A.keys.p, (const T*)A.tiles.p, A.b, pos.p, dr.p, dc.p, (T*)dv.p);
    });
    dr.download(rows, total);
    dc.download(cols, total);
    HB_CUDA(cudaMemcpyAsync(vals, dv.p, total * A.esize(), cudaMemcpyDeviceToHost, engine().stream));
    sync_stream();
    return total;
}

// ---------------------------------------------------------------------------------------------------
// norms
// ---------------------------------------------------------------------------------------------------
void compute_leaf_norms(const Matrix& A, void* d_out) { compute_leaf_norms_range(A, 0, A.L, d_out); }

// leaves [t0, t0 + cnt) only; d_out is the base of the norm array (entry t0 + i is written)
void compute_leaf_norms_range(const Matrix& A, size_t t0, size_t cnt, void* d_out) {
    if (cnt == 0) return;
    ensure_engine();
    const unsigned grid = (unsigned)((cnt + 127) / 128);
    const char* src = A.tiles.p + t0 * A.tile_bytes();
    if (A.dtype == HBSM_F64) {
        auto kfn = k_leaf_norms<double, 32>;
        HB_LAUNCH(kfn, grid, 128, 0, (const double*)src, cnt, A.tile_elems(), (double*)d_out + t0);
    } else {
        auto kfn = k_leaf_norms<float, 64>;
        HB_LAUNCH(kfn, grid, 128, 0, (const float*)src, cnt, A.tile_elems(), (float*)d_out + t0);
    }
}

// Root value of the bottom-up refresh (H:3918-3923 / H:656-662): k_fold_dense, one launch, result through the mailbox.
double hierarchical_norm(const Matrix& A, const void* d_leaf_norms) {
    if (A.L == 0) return 0.0;
    ensure_engine();
    Engine& e = engine();
    const int depth = A.vdepth();
    if (depth <= 12) {
        const int m = std::min(depth, 6);
        const uint32_t n_top = 1u << (2 * (depth - m));
        DevBuf<char> top((size_t)n_top * A.esize());
        DevBuf<unsigned> done(1);
        done.zero();
        const unsigned grid = std::min<unsigned>(n_top, 8u * (unsigned)e.sm_count);
        dispatch(A.dtype, [&](auto z) {
            using T = decltype(z);
            HB_LAUNCH(k_fold_dense<T>, grid, 256, 0, A.keys.p, (const T*)d_leaf_norms, A.L, depth, m, (T*)top.p, done.p, e.mailbox + 2);
        });
        sync_stream();
    } else {
        DevBuf<uint64_t> ka(A.L), kb(A.L);
        DevBuf<char> va(A.L * A.esize()), vb(A.L * A.esize());
        dispatch(A.dtype, [&](auto z) {
            using T = decltype(z);
            HB_LAUNCH(k_fold_root<T>, 1, 1024, 0, A.keys.p, (const T*)d_leaf_norms, A.L, depth, ka.p, (T*)va.p, kb.p, (T*)vb.p,
                      e.mailbox + 2);
        });
        sync_stream();
    }
    double root;
    const uint64_t bits = e.mailbox[2];
    memcpy(&root, &bits, sizeof root);
    return root;
}

void update_norms(Matrix& A) {   // H:3905
    A.pub.reset();   // a published (key, norm) table describes the previous norms
    if (A.L == 0) { A.root_norm_cached = 0.0; return; }
    compute_leaf_norms(A, A.norms.p);
    A.root_norm_cached = hierarchical_norm(A, A.norms.p);
}

double frob_squared(const Matrix& A) {   // H:641
    if (A.empty()) throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::get_frob_squared: empty matrix occured.");
    if (A.L == 0) return 0.0;
    DevBuf<char> tmp(A.L * A.esize());
    compute_leaf_norms(A, tmp.p);
    return hierarchical_norm(A, tmp.p);
}

// ---------------------------------------------------------------------------------------------------
// line indices
// ---------------------------------------------------------------------------------------------------
const LineIndex& line_index(const Matrix& A, bool by_col, bool with_halo) {
    const bool ext = with_halo && A.n_halo > 0;
    LineIndex& ix = const_cast<LineIndex&>(ext ? (by_col ? A.ext_by_col : A.ext_by_row) : (by_col ? A.by_col : A.by_row));
    ensure_engine();
    // an operand may be shared (read-only) by products running on different host threads: the lazy build is serialised,
    // and a thread that finds an index built on another thread's stream orders its own stream behind the build
    std::lock_guard<std::mutex> lock(shared().index_mutex);
    if (ix.valid) {
        if (ix.built_on != engine().stream && ix.ready_ev) HB_CUDA(cudaStreamWaitEvent(engine().stream, ix.ready_ev, 0));
        return ix;
    }
    const int depth = A.vdepth();
    const int dbits = std::max(depth, 1);
    const size_t n = ext ? A.n_ext() : A.L;   // halo keys sit behind the owned ones, in any order
    ix.n_lines = A.grid_side();
    ix.ptr.alloc((size_t)ix.n_lines + 1);
    ix.other.alloc(std::max<size_t>(n, 1));
    ix.tile.alloc(std::max<size_t>(n, 1));
    if (n == 0) {
        ix.ptr.zero();
    } else {
        DevBuf<uint64_t> skey(n);
        HB_LAUNCH(k_line_keys, blocks_for(n, 256), 256, 0, A.keys.p, n, by_col ? 1 : 0, dbits, skey.p, ix.tile.p);
        radix_sort_pairs(skey.p, ix.tile.p, n, 2 * dbits);
        HB_LAUNCH(k_line_ptr, blocks_for(n, 256), 256, 0, skey.p, n, dbits, ix.n_lines, ix.ptr.p, ix.other.p);
    }
    if (!ix.ready_ev) HB_CUDA(cudaEventCreateWithFlags(&ix.ready_ev, cudaEventDisableTiming));
    HB_CUDA(cudaEventRecord(ix.ready_ev, engine().stream));
    ix.built_on = engine().stream;
    ix.valid = true;
    return ix;
}

// ---------------------------------------------------------------------------------------------------
// structure operations
// ---------------------------------------------------------------------------------------------------
static unsigned slices_for(const Matrix& A) {
    return (unsigned)std::max<size_t>(1, std::min<size_t>(8, A.tile_elems() * A.esize() / 8192));
}

void op_add(const Matrix& A, const Matrix& B, Matrix& C) {   // H:1644
    C.clear();
    if (A.empty() && B.empty()) return;
    if (A.M != B.M || A.N != B.N)
        throw_ref("Error in HierarchicalBlockSparseMatrix::add(): matrices to add have different sizes!");
    if (A.dtype != B.dtype || A.b != B.b) throw Error(HBSM_E_ARG, "hbsm_b200: add: operands differ in dtype or blocksize");
    ensure_engine();
    C.dtype = A.dtype;
    C.b = A.b;
    C.resize(A.M, A.N);
    C.n_mults = A.n_mults + B.n_mults;   // H:1719
    const size_t na = A.L, nb = B.L;
    if (na + nb == 0) return;
    DevBuf<uint32_t> keep_b(std::max<size_t>(nb, 1));
    DevBuf<uint64_t> bpre;
    size_t n_bonly = 0;
    if (nb) {
        HB_LAUNCH(k_union_mark, blocks_for(nb, 256), 256, 0, A.keys.p, na, B.keys.p, nb, keep_b.p);
        n_bonly = scan_flags(keep_b, nb, bpre);
    } else {
        bpre.alloc(1);
        bpre.zero();
    }
    const size_t nu = na + n_bonly;
    DevBuf<uint64_t> ukeys(nu);
    DevBuf<uint32_t> src_a(nu), src_b(nu);
    if (na) HB_LAUNCH(k_union_pos_a, blocks_for(na, 256), 256, 0, A.keys.p, na, B.keys.p, nb, bpre.p, ukeys.p, src_a.p, src_b.p);
    if (nb) HB_LAUNCH(k_union_pos_b, blocks_for(nb, 256), 256, 0, A.keys.p, na, B.keys.p, nb, keep_b.p, bpre.p, ukeys.p, src_a.p, src_b.p);
    DevBuf<char> t(nu * C.tile_bytes());
    dispatch(C.dtype, [&](auto z) {
        using T = decltype(z);
        dim3 grid((unsigned)nu, slices_for(C));
        HB_LAUNCH(k_add_tiles<T>, grid, 256, 0, (const T*)A.tiles.p, (const T*)B.tiles.p, src_a.p, src_b.p, C.tile_elems(), (T*)t.p);
    });
    C.set_table(std::move(ukeys), std::move(t), nu);
    sync_stream();
}

void op_transpose(const Matrix& A, Matrix& C) {   // H:3733
    if (!C.empty()) throw_ref("Error in HierarchicalBlockSparseMatrix::transpose(): non-empty matrix to write result!");
    ensure_engine();
    if (A.empty()) return;
    C.dtype = A.dtype;
    C.b = A.b;
    C.resize(A.N, A.M);
    if (A.L == 0) return;
    DevBuf<uint64_t> okeys(A.L);
    DevBuf<uint32_t> idx(A.L);
    HB_LAUNCH(k_transpose_keys, blocks_for(A.L, 256), 256, 0, A.keys.p, A.L, okeys.p, idx.p);
    radix_sort_pairs(okeys.p, idx.p, A.L, key_bits_for(A));
    DevBuf<char> t(A.L * A.tile_bytes());
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        if (A.b % 32 == 0 && A.b >= 64) HB_LAUNCH((k_transpose_tiles_wide<T, 4>), (unsigned)A.L, 256, 0, (const T*)A.tiles.p, idx.p, A.b, (T*)t.p);
        else if (A.b == 32) HB_LAUNCH((k_transpose_tiles_wide<T, 1>), (unsigned)A.L, 256, 0, (const T*)A.tiles.p, idx.p, A.b, (T*)t.p);
        else HB_LAUNCH(k_transpose_tiles<T>, (unsigned)A.L, 256, 0, (const T*)A.tiles.p, idx.p, A.b, (T*)t.p);
    });
    C.set_table(std::move(okeys), std::move(t), A.L);
    sync_stream();
}

void op_upper(const Matrix& A, Matrix& C) {   // H:3515
    if (A.M != A.N) throw_ref("Error in HierarchicalBlockSparseMatrix::get_upper_triangle(): call for non-square matrix!");
    ensure_engine();
    C.clear();
    if (A.empty()) return;
    C.dtype = A.dtype;
    C.b = A.b;
    C.resize(A.M, A.N);
    if (A.L == 0) return;
    DevBuf<uint32_t> keep(A.L);
    HB_LAUNCH(k_upper_flags, blocks_for(A.L, 256), 256, 0, A.keys.p, A.L, keep.p);
    DevBuf<uint64_t> pos;
    size_t nk = scan_flags(keep, A.L, pos);
    if (nk == 0) { if (A.vdepth() > 0) { C.keys.release(); C.tiles.release(); C.L = 0; } return; }
    DevBuf<uint64_t> okeys(nk);
    DevBuf<uint32_t> src(nk);
    HB_LAUNCH(k_compact_keys, blocks_for(A.L, 256), 256, 0, A.keys.p, A.L, keep.p, pos.p, okeys.p, src.p);
    DevBuf<char> t(nk * A.tile_bytes());
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        dim3 grid((unsigned)nk, slices_for(A));
        HB_LAUNCH(k_copy_tiles<T>, grid, 256, 0, (const T*)A.tiles.p, src.p, okeys.p, A.b, 1, 0, (T)1, (T*)t.p);
    });
    C.set_table(std::move(okeys), std::move(t), nk);
    sync_stream();
}

void op_rescale(Matrix& C, const Matrix& A, double alpha) {   // H:3078
    if (!C.empty()) throw_ref("Error in HierarchicalBlockSparseMatrix::rescale(): non-empty matrix called this method!");
    ensure_engine();
    if (A.empty()) return;
    C.dtype = A.dtype;
    C.b = A.b;
    C.resize(A.M, A.N);
    if (A.L == 0) return;
    DevBuf<uint64_t> okeys(A.L);
    HB_CUDA(cudaMemcpyAsync(okeys.p, A.keys.p, A.L * sizeof(uint64_t), cudaMemcpyDeviceToDevice, engine().stream));
    DevBuf<char> t(A.L * A.tile_bytes());
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        dim3 grid((unsigned)A.L, slices_for(A));
        HB_LAUNCH(k_copy_tiles<T>, grid, 256, 0, (const T*)A.tiles.p, (const uint32_t*)nullptr, okeys.p, A.b, 0, 1, (T)alpha, (T*)t.p);
    });
    C.set_table(std::move(okeys), std::move(t), A.L);
    sync_stream();
}

void op_copy(Matrix& C, const Matrix& A) {   // H:1490
    if (&C == &A) return;
    ensure_engine();
    C.clear();
    if (A.empty()) return;
    C.dtype = A.dtype;
    C.b = A.b;
    C.resize(A.M, A.N);
    C.n_mults = A.n_mults;
    C.root_norm_cached = A.vdepth() > 0 ? A.root_norm_cached : 0.0;   // H:1507-1513: inner nodes only
    if (A.L == 0) return;
    DevBuf<uint64_t> okeys(A.L);
    HB_CUDA(cudaMemcpyAsync(okeys.p, A.keys.p, A.L * sizeof(uint64_t), cudaMemcpyDeviceToDevice, engine().stream));
    DevBuf<char> t(A.L * A.tile_bytes());
    HB_CUDA(cudaMemcpyAsync(t.p, A.tiles.p, A.L * A.tile_bytes(), cudaMemcpyDeviceToDevice, engine().stream));
    C.set_table(std::move(okeys), std::move(t), A.L);
    sync_stream();
}

bool trunc_begin(const Matrix& A, Matrix& C) {
    ensure_engine();
    C.clear();
    if (A.empty()) return false;    // copy of an empty matrix
    C.dtype = A.dtype;
    C.b = A.b;
    C.resize(A.M, A.N);
    C.n_mults = A.n_mults;
    C.root_norm_cached = A.vdepth() > 0 ? A.root_norm_cached : 0.0;   // copy() keeps the (now stale) root norm, H:1507-1513
    if (A.L == 0) return false;
    if (A.vdepth() == 0) {   // a single leaf has no children to drop
        HB_CUDA(cudaMemcpyAsync(C.tiles.p, A.tiles.p, A.tile_bytes(), cudaMemcpyDeviceToDevice, engine().stream));
        sync_stream();
        return false;
    }
    return true;
}

void trunc_keep_flags(const Matrix& A, const void* d_nsq, double trunc_value, uint32_t* keep) {
    const float tf = (float)trunc_value;
    HB_LAUNCH(k_trunc_flags, blocks_for(A.L, 256), 256, 0, d_nsq, A.L, A.dtype == HBSM_F64 ? 1 : 0, trunc_value * trunc_value,
              tf * tf, keep);
}

size_t trunc_compact(const Matrix& A, const DevBuf<uint32_t>& keep, Matrix& C) {
    DevBuf<uint64_t> pos;
    size_t nk = scan_flags(keep, A.L, pos);
    if (nk == 0) return 0;
    DevBuf<uint64_t> okeys(nk);
    DevBuf<uint32_t> src(nk);
    HB_LAUNCH(k_compact_keys, blocks_for(A.L, 256), 256, 0, A.keys.p, A.L, keep.p, pos.p, okeys.p, src.p);
    DevBuf<char> t(nk * A.tile_bytes());
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        dim3 grid((unsigned)nk, slices_for(A));
        HB_LAUNCH(k_copy_tiles<T>, grid, 256, 0, (const T*)A.tiles.p, src.p, okeys.p, A.b, 0, 0, (T)1, (T*)t.p);
    });
    C.set_table(std::move(okeys), std::move(t), nk);
    sync_stream();
    return nk;
}

bool op_trunc(const Matrix& A, Matrix& C, double trunc_value) {   // H:4935: C = copy of A without the small subtrees
    if (&C == &A) throw Error(HBSM_E_ARG, "hbsm_b200: frob_block_trunc: target must not alias the source");
    if (!trunc_begin(A, C)) return false;
    DevBuf<char> fresh(A.L * A.esize());
    compute_leaf_norms(A, fresh.p);
    DevBuf<uint32_t> keep(A.L);
    trunc_keep_flags(A, fresh.p, trunc_value, keep.p);
    return trunc_compact(A, keep, C) < A.L;
}

bool op_extract_quadrant(const Matrix& A, int q, Matrix& C) {
    if (&C == &A) throw Error(HBSM_E_ARG, "hbsm_b200: extract_quadrant: target must not alias the source");
    if (q < 0 || q > 3) throw Error(HBSM_E_ARG, "hbsm_b200: quadrant index must be 0..3");
    if (A.empty() || A.vdepth() == 0) throw Error(HBSM_E_ARG, "hbsm_b200: extract_quadrant needs a matrix with children");
    ensure_engine();
    C.clear();
    C.dtype = A.dtype;
    C.b = A.b;
    const int P = A.vdepth();
    const int half = A.b << (P - 1);
    C.resize(half, half);   // children carry their virtual size (H:791-833)
    if (A.L == 0) return false;
    std::vector<uint64_t> keys = A.keys.to_host();
    const int sh = 2 * (P - 1);
    size_t lo = 0, hi = 0;   // leaves of a quadrant are one contiguous key range
    for (size_t i = 0; i < A.L; ++i) {
        const int d = (int)((keys[i] >> sh) & 3u);
        if (d < q) lo = i + 1;
        if (d <= q) hi = i + 1;
    }
    if (hi <= lo) return false;   // absent child (for a leaf child C keeps its zero tile)
    const size_t n = hi - lo;
    if (P - 1 == 0) {   // the child is a single leaf: C already owns one zero tile
        HB_CUDA(cudaMemcpyAsync(C.tiles.p, A.tiles.p + lo * A.tile_bytes(), A.tile_bytes(), cudaMemcpyDeviceToDevice, engine().stream));
        HB_CUDA(cudaMemcpyAsync(C.norms.p, A.norms.p + lo * A.esize(), A.esize(), cudaMemcpyDeviceToDevice, engine().stream));
        sync_stream();
        return true;
    }
    DevBuf<uint64_t> ck(n);
    HB_LAUNCH(k_rekey, blocks_for(n, 256), 256, 0, A.keys.p + lo, n, (1ull << sh) - 1ull, 0ull, ck.p);
    DevBuf<char> ct(n * A.tile_bytes());
    HB_CUDA(cudaMemcpyAsync(ct.p, A.tiles.p + lo * A.tile_bytes(), n * A.tile_bytes(), cudaMemcpyDeviceToDevice, engine().stream));
    C.set_table(std::move(ck), std::move(ct), n);
    HB_CUDA(cudaMemcpyAsync(C.norms.p, A.norms.p + lo * A.esize(), n * A.esize(), cudaMemcpyDeviceToDevice, engine().stream));
    sync_stream();
    return true;
}

void op_assemble_quadrants(Matrix& C, int M, int N, const Matrix* quads[4]) {
    ensure_engine();
    const Matrix* first = nullptr;
    for (int q = 0; q < 4; ++q) if (quads[q] && !quads[q]->empty()) { if (!first) first = quads[q]; }
    if (!first) throw Error(HBSM_E_ARG, "hbsm_b200: assemble_quadrants needs at least one quadrant");
    for (int q = 0; q < 4; ++q) if (quads[q] == &C) throw Error(HBSM_E_ARG, "hbsm_b200: assemble_quadrants: target aliases a quadrant");
    C.clear();
    C.dtype = first->dtype;
    C.b = first->b;
    C.resize(M, N);
    const int P = C.vdepth();
    if (P == 0) throw Error(HBSM_E_ARG, "hbsm_b200: assemble_quadrants: the target is a single leaf");
    size_t total = 0;
    for (int q = 0; q < 4; ++q) {
        if (!quads[q] || quads[q]->empty()) continue;
        if (quads[q]->vdepth() != P - 1 || quads[q]->b != C.b || quads[q]->dtype != C.dtype)
            throw Error(HBSM_E_ARG, "hbsm_b200: assemble_quadrants: quadrant shape does not fit the target");
        total += quads[q]->L;
    }
    if (total == 0) return;
    DevBuf<uint64_t> keys(total);
    DevBuf<char> tiles(total * C.tile_bytes());
    size_t at = 0;
    const int sh = 2 * (P - 1);
    for (int q = 0; q < 4; ++q) {   // quadrant order = ascending leading digit = ascending Morton order
        const Matrix* Q = quads[q];
        if (!Q || Q->empty() || Q->L == 0) continue;
        HB_LAUNCH(k_rekey, blocks_for(Q->L, 256), 256, 0, Q->keys.p, Q->L, ~0ull, (uint64_t)q << sh, keys.p + at);
        HB_CUDA(cudaMemcpyAsync(tiles.p + at * C.tile_bytes(), Q->tiles.p, Q->L * C.tile_bytes(), cudaMemcpyDeviceToDevice, engine().stream));
        at += Q->L;
    }
    C.set_table(std::move(keys), std::move(tiles), total);
    sync_stream();
}

// inv_chol leaf (H:3118-3147): A is a single-leaf matrix, Z becomes the zdim x zdim single-leaf inverse factor of its leading
// `valid` x `valid` block (identity pattern elsewhere is NOT written: rows/columns >= valid stay zero, as upstream)
void op_leaf_inv_chol(const Matrix& A, Matrix& Z, int zdim, int valid) {
    ensure_engine();
    if (A.empty() || A.vdepth() != 0 || A.L != 1) throw Error(HBSM_E_ARG, "hbsm_b200: leaf_inv_chol wants a single-leaf matrix");
    if (zdim <= 0 || zdim > A.b) throw Error(HBSM_E_ARG, "hbsm_b200: leaf_inv_chol: bad result dimension");
    if (A.b > 256) throw Error(HBSM_E_ARG, "hbsm_b200: leaf_inv_chol supports leaves up to 256");
    Z.dtype = A.dtype;
    Z.b = A.b;
    Z.resize(zdim, zdim);                 // one zero-filled leaf
    const int n = std::min(valid, A.b);
    if (n <= 0) return;
    dispatch(A.dtype, [&](auto zt) {
        using T = decltype(zt);
        HB_LAUNCH(k_leaf_inv_chol<T>, 1, 256, 0, (const T*)A.tiles.p, A.b, n, (T*)Z.tiles.p);
    });
    sync_stream();
}

void sym_expand(const Matrix& A, Matrix& S) {
    ensure_engine();
    S.clear();
    S.dtype = A.dtype;
    S.b = A.b;
    S.resize(A.M, A.N);
    if (A.L == 0) return;
    const size_t n2 = 2 * A.L;
    DevBuf<uint64_t> k2(n2);
    DevBuf<uint32_t> s2(n2), valid(n2);
    HB_LAUNCH(k_sym_keys, blocks_for(A.L, 256), 256, 0, A.keys.p, A.L, k2.p, s2.p, valid.p);
    DevBuf<uint64_t> pos;
    size_t ns = scan_flags(valid, n2, pos);
    if (ns == 0) return;
    DevBuf<uint64_t> okeys(ns);
    DevBuf<uint32_t> packed(ns);
    HB_LAUNCH(k_sym_compact, blocks_for(n2, 256), 256, 0, k2.p, s2.p, valid.p, pos.p, n2, okeys.p, packed.p);
    radix_sort_pairs(okeys.p, packed.p, ns, key_bits_for(A));
    DevBuf<uint32_t> src(ns), flag(ns);
    HB_LAUNCH(k_sym_unpack, blocks_for(ns, 256), 256, 0, okeys.p, packed.p, ns, src.p, flag.p);
    DevBuf<char> t(ns * A.tile_bytes());
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        HB_LAUNCH(k_sym_tiles<T>, (unsigned)ns, 256, 0, (const T*)A.tiles.p, src.p, flag.p, A.b, (T*)t.p);
    });
    S.set_table(std::move(okeys), std::move(t), ns);
    sync_stream();
}

void mask_diag_upper(Matrix& C) {
    if (C.L == 0) return;
    ensure_engine();
    dispatch(C.dtype, [&](auto z) {
        using T = decltype(z);
        HB_LAUNCH(k_mask_diag<T>, (unsigned)C.L, 256, 0, C.keys.p, C.b, (T*)C.tiles.p);
    });
}

void generate_decay(Matrix& A, int n, const double* table, int W, uint64_t seed, bool symmetric, int lo, int hi) {
    ensure_engine();
    A.resize(n, n);
    const uint32_t g = (uint32_t)((n + A.b - 1) / A.b);
    if (hi < 0 || hi > (int)g) hi = (int)g;
    if (lo < 0) lo = 0;
    if (lo >= hi) return;
    const uint32_t wb = (uint32_t)std::min<long long>(g, ((long long)W + A.b - 1) / A.b);
    if (A.vdepth() == 0) {
        DevBuf<double> dtab((size_t)W + 1);
        dtab.upload(table, (size_t)W + 1);
        dispatch(A.dtype, [&](auto z) {
            using T = decltype(z);
            HB_LAUNCH(k_decay_fill<T>, 1, 256, 0, A.keys.p, A.b, n, W, dtab.p, seed, symmetric ? 1 : 0, (T*)A.tiles.p);
        });
        sync_stream();
        return;
    }
    const size_t span = 2 * (size_t)wb + 1, cand = (size_t)(hi - lo) * span;
    DevBuf<uint64_t> ck(cand);
    DevBuf<uint32_t> ci(cand);
    HB_LAUNCH(k_decay_keys, blocks_for(cand, 256), 256, 0, (uint32_t)lo, (uint32_t)hi, g, wb, ck.p);
    // sort (invalid ~0 keys go last), count valid
    HB_CUDA(cudaMemsetAsync(ci.p, 0, cand * sizeof(uint32_t), engine().stream));
    radix_sort_pairs(ck.p, ci.p, cand, 64);
    std::vector<uint64_t> hk = ck.to_host();
    size_t L = 0;
    while (L < cand && hk[L] != ~0ull) ++L;
    if (L == 0) return;
    DevBuf<uint64_t> keys(L);
    HB_CUDA(cudaMemcpyAsync(keys.p, ck.p, L * sizeof(uint64_t), cudaMemcpyDeviceToDevice, engine().stream));
    DevBuf<char> t(L * A.tile_bytes());
    DevBuf<double> dtab((size_t)W + 1);
    dtab.upload(table, (size_t)W + 1);
    dispatch(A.dtype, [&](auto z) {
        using T = decltype(z);
        HB_LAUNCH(k_decay_fill<T>, (unsigned)L, 256, 0, keys.p, A.b, n, W, dtab.p, seed, symmetric ? 1 : 0, (T*)t.p);
    });
    A.set_table(std::move(keys), std::move(t), L);
    sync_stream();
}

}  // namespace hbsm_b200

// sharded.cu -- the multi-GPU product behind the C ABI (SURVEY 8e): one process per GPU, C sharded by block rows, NCCL over
// NVLink 5 / NVSwitch for the one exchange step a product has.  The reference has no distributed layer at all; its stated
// caller (a task runtime) ships whole sub-matrices.  Here rank r owns the block rows [bounds[r], bounds[r+1]) of C, the tiles of
// op(A) with ci in that range and the tiles of op(B) with k in that range.  One product is
//
//   engine stream : thr[k] = max nsq of my op(A) tiles (., k) | all-gather thr (world x g reals, a few KB) | flags + scan
//                   -> [one host read: 2 x world counts] -> halo keys+norms from the published table | task list | own-only C
//                   tiles' leaf GEMMs | ---- wait(tiles) ---- | C tiles that read halo tiles
//   comm stream   :                                             pack my requested tiles | grouped ncclSend/ncclRecv straight
//                                                               into op(B)'s halo tail ----^
//
// Every rank holds the (key, norm^2) table of the whole op(B) (hbsm_publish, the distributed half of update_internal_info) and,
// after the all-gather, every rank's request thresholds.  Requester and owner therefore evaluate the SAME predicate on the SAME
// numbers -- fl(thr_q[k] * nsq(B_kj)) > fl(tau*tau), monotone rounding => exactly the tiles at least one executed product of
// rank q touches -- so no request masks and no counts travel: the only NCCL traffic of a product is the thresholds and the
// tiles.  There is no reduction (a rank owns whole block rows of C) and the executed-product set is the disjoint union of
// the per-rank sets, bit-identical to the single-GPU one because the prune rule is per leaf pair (H:6649-6651, SURVEY 0.3).
//
// NCCL is resolved at run time (dlopen): the library loads, and every single-GPU entry point works, on hosts without NCCL.
#include "matrix.cuh"
#include <dlfcn.h>
#include <nccl.h>
#include <numeric>

namespace hbsm_b200 {

namespace {

struct NcclApi {
    void* handle = nullptr;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclAllReduce) AllReduce = nullptr;
    decltype(&ncclSend) Send = nullptr;
    decltype(&ncclRecv) Recv = nullptr;
    decltype(&ncclGroupStart) GroupStart = nullptr;
    decltype(&ncclGroupEnd) GroupEnd = nullptr;
    decltype(&ncclGetVersion) GetVersion = nullptr;
    std::string path;
};

struct Comm {
    std::mutex mu;            // collectives are issued by one host thread at a time, in the same order on every rank
    NcclApi api;
    std::string lib_override;
    bool ready = false;
    int rank = 0, world = 1;
    ncclComm_t comm = nullptr;
    cudaStream_t stream = nullptr;     // pack + tile exchange
    cudaEvent_t ev_plan = nullptr, ev_tiles = nullptr, ev_x0 = nullptr, ev_x1 = nullptr;
    hbsm_shard_stats last{};
};
Comm& comm() {
    static Comm c;
    return c;
}

template <typename F>
F sym(void* h, const char* name) {
    void* p = dlsym(h, name);
    if (!p) throw Error(HBSM_E_RUNTIME, std::string("hbsm_b200: NCCL library lacks ") + name);
    return reinterpret_cast<F>(p);
}

void load_nccl(Comm& c) {
    if (c.api.handle) return;
    std::vector<std::string> tries;
    if (!c.lib_override.empty()) tries.push_back(c.lib_override);
    if (const char* e = getenv("HBSM_NCCL_LIB")) tries.push_back(e);
    void* h = nullptr;
    std::string got;
    for (const auto& t : tries) {
        h = dlopen(t.c_str(), RTLD_NOW | RTLD_GLOBAL);
        if (h) { got = t; break; }
    }
    if (!h) {   // a copy already mapped into the process (e.g. the one torch ships) wins over the system one
        h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
        if (h) got = "libnccl.so.2 (already loaded)";
    }
    if (!h) {
        h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (h) got = "libnccl.so.2";
    }
    if (!h) throw Error(HBSM_E_RUNTIME, std::string("hbsm_b200: cannot load NCCL (libnccl.so.2): ") + (dlerror() ? dlerror() : "?"));
    NcclApi& a = c.api;
    a.GetUniqueId = sym<decltype(a.GetUniqueId)>(h, "ncclGetUniqueId");
    a.CommInitRank = sym<decltype(a.CommInitRank)>(h, "ncclCommInitRank");
    a.CommDestroy = sym<decltype(a.CommDestroy)>(h, "ncclCommDestroy");
    a.GetErrorString = sym<decltype(a.GetErrorString)>(h, "ncclGetErrorString");
    a.AllGather = sym<decltype(a.AllGather)>(h, "ncclAllGather");
    a.AllReduce = sym<decltype(a.AllReduce)>(h, "ncclAllReduce");
    a.Send = sym<decltype(a.Send)>(h, "ncclSend");
    a.Recv = sym<decltype(a.Recv)>(h, "ncclRecv");
    a.GroupStart = sym<decltype(a.GroupStart)>(h, "ncclGroupStart");
    a.GroupEnd = sym<decltype(a.GroupEnd)>(h, "ncclGroupEnd");
    a.GetVersion = sym<decltype(a.GetVersion)>(h, "ncclGetVersion");
    a.path = got;
    a.handle = h;
}

#define HB_NCCL(call)                                                                                     \
    do {                                                                                                  \
        ncclResult_t r_ = (call);                                                                         \
        if (r_ != ncclSuccess)                                                                            \
            throw Error(HBSM_E_RUNTIME, std::string("hbsm_b200: NCCL: ") + comm().api.GetErrorString(r_) + " in " #call); \
    } while (0)

#define HB_LAUNCH_ON(stream_, kernel, grid, block, smem, ...)                                  \
    do {                                                                                       \
        kernel<<<(grid), (block), (smem), (stream_)>>>(__VA_ARGS__);                           \
        ::hbsm_b200::engine().launches++;                                                      \
        ::hbsm_b200::shared().launches.fetch_add(1, std::memory_order_relaxed);                \
        HB_CUDA(cudaGetLastError());                                                           \
    } while (0)

inline unsigned blocks_of(size_t n, unsigned bs) { return (unsigned)std::max<size_t>(1, (n + bs - 1) / bs); }

Comm& ready_comm() {
    Comm& c = comm();
    if (!c.ready) throw Error(HBSM_E_ARG, "hbsm_b200: no communicator (call hbsm_comm_init on every rank first)");
    return c;
}

ncclDataType_t nccl_real(int dtype) { return dtype == HBSM_F64 ? ncclFloat64 : ncclFloat32; }

template <typename F>
void dispatch_real(int dtype, F&& f) {
    if (dtype == HBSM_F64) f(double(0));
    else f(float(0));
}

// ---- kernels ----
template <typename T> struct IntOf;
template <> struct IntOf<double> { typedef long long I; };
template <> struct IntOf<float> { typedef int I; };

template <typename T>
__global__ void k_fill_minus_one(T* __restrict__ p, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = (T)-1;
}
// thr[k] = max leaf norm^2 over my op(A) tiles (., k).  Non-negative IEEE values order like signed integers and -1.0 is a
// negative integer, so a signed atomicMax on the bit pattern does it.
template <typename T>
__global__ void k_request(const uint64_t* __restrict__ keys, const T* __restrict__ norms, size_t L, int k_is_row, T* __restrict__ thr) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= L) return;
    const uint32_t k = k_is_row ? morton_row(keys[i]) : morton_col(keys[i]);
    typedef typename IntOf<T>::I I;
    T v = norms[i];
    atomicMax(reinterpret_cast<I*>(thr) + k, *reinterpret_cast<I*>(&v));
}
// entry e < n_all: "do I need published tile e?" (remote, requested by MY thresholds); entry n_all + q*L_own + i: "does
// peer q need my tile i?" (the same test against q's thresholds).  Both read the published norms, so the two sides of every
// transfer agree bit for bit.
template <typename T>
__global__ void k_shard_flags(const uint64_t* __restrict__ keys_all, const T* __restrict__ norms_all, size_t n_all, size_t own_lo,
                              size_t L_own, const T* __restrict__ thr_all, uint32_t g, int world, int rank, int k_is_col, int spamm,
                              T tau2, uint32_t* __restrict__ flags) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t total = n_all + (size_t)world * L_own;
    if (e >= total) return;
    size_t t;
    int q;
    bool keep;
    if (e < n_all) {
        t = e; q = rank;
        keep = (t < own_lo || t >= own_lo + L_own);
    } else {
        const size_t x = e - n_all;
        q = (int)(x / L_own);
        t = own_lo + x % L_own;
        keep = (q != rank);
    }
    if (keep) {
        const uint64_t key = keys_all[t];
        const uint32_t k = k_is_col ? morton_col(key) : morton_row(key);
        const T th = thr_all[(size_t)q * g + k];
        keep = th >= (T)0;
        if (keep && spamm) keep = DT<T>::mul(th, norms_all[t]) > tau2;
    }
    flags[e] = keep ? 1u : 0u;
}
struct Edges { uint64_t at[132]; int n; };
__global__ void k_post_edges(const uint64_t* __restrict__ pos, Edges edges, volatile uint64_t* mailbox) {
    for (int i = threadIdx.x; i < edges.n; i += blockDim.x) mailbox[i] = pos[edges.at[i]];
    __threadfence_system();
}
// needed remote tiles: key and norm into op(B)'s halo tail (the tile follows over NCCL); requested own tiles: send list
template <typename T>
__global__ void k_shard_fill(const uint32_t* __restrict__ flags, const uint64_t* __restrict__ pos, size_t n_all, size_t total,
                             size_t own_lo, size_t L_own, const uint64_t* __restrict__ keys_all, const T* __restrict__ norms_all,
                             uint64_t* __restrict__ tail_keys, T* __restrict__ tail_norms, uint32_t* __restrict__ send_idx) {
    const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total || !flags[e]) return;
    if (e < n_all) {
        tail_keys[pos[e]] = keys_all[e];
        tail_norms[pos[e]] = norms_all[e];
    } else {
        send_idx[pos[e] - pos[n_all]] = (uint32_t)((e - n_all) % L_own);
    }
}
// one warp-sized stride of 16-byte words per tile: pack[j] = tiles[idx[j]]
__global__ void __launch_bounds__(256) k_pack_tiles(const uint4* __restrict__ tiles, const uint32_t* __restrict__ idx, size_t n,
                                                    uint32_t words_per_tile, uint4* __restrict__ pack) {
    const size_t total = n * words_per_tile;
    for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (size_t)gridDim.x * blockDim.x) {
        const size_t j = w / words_per_tile;
        const uint32_t o = (uint32_t)(w % words_per_tile);
        pack[w] = __ldg(tiles + (size_t)idx[j] * words_per_tile + o);
    }
}

}  // namespace

// ---------------------------------------------------------------------------------------------------
// communicator
// ---------------------------------------------------------------------------------------------------
void comm_set_library(const char* path) {
    Comm& c = comm();
    std::lock_guard<std::mutex> lock(c.mu);
    c.lib_override = path ? path : "";
}

void comm_unique_id(void* out128) {
    Comm& c = comm();
    std::lock_guard<std::mutex> lock(c.mu);
    load_nccl(c);
    ncclUniqueId id;
    HB_NCCL(c.api.GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == HBSM_COMM_ID_BYTES, "NCCL unique id size");
    memcpy(out128, &id, sizeof id);
}

void comm_init(const void* id128, int rank, int world) {
    if (world < 1 || world > 64 || rank < 0 || rank >= world) throw Error(HBSM_E_ARG, "hbsm_b200: comm_init: bad rank / world (world <= 64)");
    ensure_engine();
    Comm& c = comm();
    std::lock_guard<std::mutex> lock(c.mu);
    if (c.ready) throw Error(HBSM_E_ARG, "hbsm_b200: communicator already initialised");
    load_nccl(c);
    ncclUniqueId id;
    memcpy(&id, id128, sizeof id);
    HB_NCCL(c.api.CommInitRank(&c.comm, world, id, rank));
    HB_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    HB_CUDA(cudaEventCreateWithFlags(&c.ev_plan, cudaEventDisableTiming));
    HB_CUDA(cudaEventCreateWithFlags(&c.ev_tiles, cudaEventDisableTiming));
    HB_CUDA(cudaEventCreate(&c.ev_x0));
    HB_CUDA(cudaEventCreate(&c.ev_x1));
    c.rank = rank; c.world = world;
    c.ready = true;
}

void comm_finalize() {
    Comm& c = comm();
    std::lock_guard<std::mutex> lock(c.mu);
    if (!c.ready) return;
    cudaStreamSynchronize(c.stream);
    c.api.CommDestroy(c.comm);
    cudaStreamDestroy(c.stream);
    cudaEventDestroy(c.ev_plan); cudaEventDestroy(c.ev_tiles); cudaEventDestroy(c.ev_x0); cudaEventDestroy(c.ev_x1);
    c.comm = nullptr; c.stream = nullptr; c.ready = false; c.rank = 0; c.world = 1;
}

void comm_info(int* rank, int* world, int* nccl_version) {
    Comm& c = comm();
    if (rank) *rank = c.ready ? c.rank : 0;
    if (world) *world = c.ready ? c.world : 1;
    if (nccl_version) {
        *nccl_version = 0;
        if (c.api.handle) c.api.GetVersion(nccl_version);
    }
}

// sum / max of a few host scalars over the ranks (counters of a sharded call, timings)
void comm_allreduce_f64(double* vals, int n, bool take_max) {
    Comm& c = ready_comm();
    std::lock_guard<std::mutex> lock(c.mu);
    if (n <= 0) return;
    DevBuf<double> d((size_t)n);
    d.upload(vals, (size_t)n);
    HB_NCCL(c.api.AllReduce(d.p, d.p, (size_t)n, ncclFloat64, take_max ? ncclMax : ncclSum, c.comm, engine().stream));
    d.download(vals, (size_t)n);
    sync_stream();
}

void comm_allgather_u64(const uint64_t* mine, size_t n, uint64_t* all) {
    Comm& c = ready_comm();
    std::lock_guard<std::mutex> lock(c.mu);
    if (n == 0) return;
    DevBuf<uint64_t> d(n * (size_t)c.world);
    HB_CUDA(cudaMemcpyAsync(d.p + n * (size_t)c.rank, mine, n * sizeof(uint64_t), cudaMemcpyHostToDevice, engine().stream));
    HB_NCCL(c.api.AllGather(d.p + n * (size_t)c.rank, d.p, n, ncclUint64, c.comm, engine().stream));
    d.download(all, n * (size_t)c.world);
    sync_stream();
}

void comm_barrier() {
    double x = 0;
    comm_allreduce_f64(&x, 1, false);
}

// ---------------------------------------------------------------------------------------------------
// publish: the (Morton key, leaf norm^2) table of a row-sharded matrix, gathered on every rank -- the distributed half of
// update_internal_info() (H:3905).  Like the cached norms it is valid until the matrix changes.
// ---------------------------------------------------------------------------------------------------
void publish(Matrix& B) {
    Comm& c = ready_comm();
    std::lock_guard<std::mutex> lock(c.mu);
    if (B.empty()) throw Error(HBSM_E_ARG, "hbsm_b200: publish of an unsized matrix");
    Engine& e = engine();
    EventTimer tm;
    tm.start();
    const int W = c.world;
    auto pub = std::make_unique<Published>();
    pub->world = W; pub->rank = c.rank;
    // round 1: the tile counts
    DevBuf<uint64_t> cnt((size_t)W);
    const uint64_t mine = B.L;
    HB_CUDA(cudaMemcpyAsync(cnt.p + c.rank, &mine, sizeof mine, cudaMemcpyHostToDevice, e.stream));
    HB_NCCL(c.api.AllGather(cnt.p + c.rank, cnt.p, 1, ncclUint64, c.comm, e.stream));
    std::vector<uint64_t> counts = cnt.to_host();
    pub->offsets.assign((size_t)W + 1, 0);
    size_t lmax = 0;
    for (int q = 0; q < W; ++q) {
        pub->offsets[q + 1] = pub->offsets[q] + (size_t)counts[q];
        lmax = std::max(lmax, (size_t)counts[q]);
    }
    pub->n_all = pub->offsets[W];
    if (pub->n_all >= 0xffffffffull) throw Error(HBSM_E_ARG, "hbsm_b200: publish: more than 2^32-1 tiles");
    const size_t es = B.esize();
    pub->keys_all.alloc(std::max<size_t>(pub->n_all, 1));
    pub->norms_all.alloc(std::max<size_t>(pub->n_all, 1) * es);
    if (lmax > 0) {
        // round 2: keys and norms, padded to the longest part (all-gather wants equal counts), then squeezed rank-major
        DevBuf<uint64_t> kpad(lmax * (size_t)W);
        DevBuf<char> npad(lmax * (size_t)W * es);
        if (B.L) {
            HB_CUDA(cudaMemcpyAsync(kpad.p + lmax * (size_t)c.rank, B.keys.p, B.L * sizeof(uint64_t), cudaMemcpyDeviceToDevice, e.stream));
            HB_CUDA(cudaMemcpyAsync(npad.p + lmax * (size_t)c.rank * es, B.norms.p, B.L * es, cudaMemcpyDeviceToDevice, e.stream));
        }
        HB_NCCL(c.api.GroupStart());
        HB_NCCL(c.api.AllGather(kpad.p + lmax * (size_t)c.rank, kpad.p, lmax, ncclUint64, c.comm, e.stream));
        HB_NCCL(c.api.AllGather(npad.p + lmax * (size_t)c.rank * es, npad.p, lmax, nccl_real(B.dtype), c.comm, e.stream));
        HB_NCCL(c.api.GroupEnd());
        for (int q = 0; q < W; ++q) {
            if (!counts[q]) continue;
            HB_CUDA(cudaMemcpyAsync(pub->keys_all.p + pub->offsets[q], kpad.p + lmax * (size_t)q, counts[q] * sizeof(uint64_t),
                                    cudaMemcpyDeviceToDevice, e.stream));
            HB_CUDA(cudaMemcpyAsync(pub->norms_all.p + pub->offsets[q] * es, npad.p + lmax * (size_t)q * es, counts[q] * es,
                                    cudaMemcpyDeviceToDevice, e.stream));
        }
    }
    tm.stop();
    sync_stream();
    c.last.publish_ms = tm.ms();
    B.pub = std::move(pub);
}

// ---------------------------------------------------------------------------------------------------
// the sharded product
// ---------------------------------------------------------------------------------------------------
void sharded_product(const Matrix& A, bool tA, Matrix& B, bool tB, Matrix& C, const ProductOpts& o, size_t* n_mults, size_t* n_blocks) {
    Comm& c = ready_comm();
    std::lock_guard<std::mutex> lock(c.mu);
    Engine& e = engine();
    if (A.empty() || B.empty()) throw Error(HBSM_E_ARG, "hbsm_b200: product of an empty (unsized) matrix");
    if (A.dtype != B.dtype || A.b != B.b) throw Error(HBSM_E_ARG, "hbsm_b200: operands differ in dtype or blocksize");
    if (!B.pub || B.pub->world != c.world || B.pub->rank != c.rank)
        throw Error(HBSM_E_ARG, "hbsm_b200: sharded product: op(B) has no published table (call hbsm_publish after update_internal_info)");
    if (o.spamm && !o.updated) throw Error(HBSM_E_ARG, "hbsm_b200: sharded spamm needs refreshed norms (updated = true): the published table carries them");
    const Published& pb = *B.pub;
    const int W = c.world, me = c.rank;
    const size_t own_lo = pb.offsets[me], L_own = pb.offsets[me + 1] - pb.offsets[me];
    if (L_own != B.L) throw Error(HBSM_E_ARG, "hbsm_b200: sharded product: the published table of op(B) is stale");
    const size_t n_all = pb.n_all;
    const uint32_t g = std::max(A.grid_side(), B.grid_side());
    const size_t es = A.esize();
    hbsm_shard_stats st{};
    EventTimer t_plan;
    t_plan.start();

    // 1. request thresholds, all-gathered in place
    DevBuf<char> thr_all((size_t)W * g * es);
    dispatch_real(A.dtype, [&](auto z) {
        using T = decltype(z);
        T* mine = (T*)thr_all.p + (size_t)me * g;
        HB_LAUNCH(k_fill_minus_one<T>, blocks_of(g, 256), 256, 0, mine, g);
        if (A.L) HB_LAUNCH(k_request<T>, blocks_of(A.L, 256), 256, 0, A.keys.p, (const T*)A.norms.p, A.L, tA ? 1 : 0, mine);
    });
    if (W > 1) HB_NCCL(c.api.AllGather(thr_all.p + (size_t)me * g * es, thr_all.p, g, nccl_real(A.dtype), c.comm, e.stream));

    // 2. what I need / what every peer needs from me: flags, scan, 2 x world counts through the mailbox
    const size_t total = n_all + (size_t)W * L_own;
    std::vector<size_t> recv_counts((size_t)W, 0), send_counts((size_t)W, 0);
    size_t n_in = 0, n_out = 0;
    DevBuf<uint32_t> flags;
    DevBuf<uint64_t> pos;
    if (total > 0 && W > 1) {
        flags.alloc(total);
        pos.alloc(total + 1);
        dispatch_real(A.dtype, [&](auto z) {
            using T = decltype(z);
            const T tt = (T)o.tau;
            HB_LAUNCH(k_shard_flags<T>, blocks_of(total, 256), 256, 0, pb.keys_all.p, (const T*)pb.norms_all.p, n_all, own_lo, L_own,
                      (const T*)thr_all.p, g, W, me, tB ? 1 : 0, o.spamm ? 1 : 0, (T)(tt * tt), flags.p);
        });
        exclusive_scan_u32(flags.p, pos.p, total);
        Edges ed;
        ed.n = 2 * (W + 1);
        for (int q = 0; q <= W; ++q) {
            ed.at[q] = pb.offsets[q];
            ed.at[W + 1 + q] = n_all + (size_t)q * L_own;
        }
        HB_LAUNCH(k_post_edges, 1, 64, 0, pos.p, ed, e.mailbox + 8);
        sync_stream();
        for (int q = 0; q < W; ++q) {
            recv_counts[q] = (size_t)(e.mailbox[8 + q + 1] - e.mailbox[8 + q]);
            send_counts[q] = (size_t)(e.mailbox[8 + W + 1 + q + 1] - e.mailbox[8 + W + 1 + q]);
            n_in += recv_counts[q];
            n_out += send_counts[q];
        }
    }

    // 3. halo tail: keys + norms now (enough for the task list), tiles over NCCL
    uint64_t* tail_k = nullptr;
    void* tail_n = nullptr;
    void* tail_t = nullptr;
    DevBuf<uint32_t> send_idx(std::max<size_t>(n_out, 1));
    DevBuf<char> pack;
    if (n_in > 0) reserve_halo(B, std::max(B.halo_cap, n_in > B.halo_cap ? std::max<size_t>(n_in + n_in / 4, 64) : n_in), &tail_k, &tail_n, &tail_t);
    if (n_in > 0 || n_out > 0) {
        dispatch_real(A.dtype, [&](auto z) {
            using T = decltype(z);
            HB_LAUNCH(k_shard_fill<T>, blocks_of(total, 256), 256, 0, flags.p, pos.p, n_all, total, own_lo, L_own, pb.keys_all.p,
                      (const T*)pb.norms_all.p, tail_k, (T*)tail_n, send_idx.p);
        });
    }
    commit_halo(B, n_in);
    const size_t tb = B.tile_bytes();
    if (n_out > 0) pack.alloc(n_out * tb);
    t_plan.stop();
    const bool exchange = n_in > 0 || n_out > 0;
    if (exchange) {
        HB_CUDA(cudaEventRecord(c.ev_plan, e.stream));
        HB_CUDA(cudaStreamWaitEvent(c.stream, c.ev_plan, 0));
        HB_CUDA(cudaEventRecord(c.ev_x0, c.stream));
        if (n_out > 0) {
            const uint32_t words = (uint32_t)(tb / 16);
            if (tb % 16 != 0) throw Error(HBSM_E_ARG, "hbsm_b200: sharded product needs leaf tiles that are a multiple of 16 bytes");
            const unsigned grid = (unsigned)std::min<size_t>(blocks_of(n_out * words, 256), (size_t)e.sm_count * 8);
            HB_LAUNCH_ON(c.stream, k_pack_tiles, grid, 256, 0, (const uint4*)B.tiles.p, send_idx.p, n_out, words, (uint4*)pack.p);
        }
        const size_t te = B.tile_elems();
        HB_NCCL(c.api.GroupStart());
        size_t so = 0, ro = 0;
        for (int q = 0; q < W; ++q) {
            if (send_counts[q]) HB_NCCL(c.api.Send(pack.p + so * tb, send_counts[q] * te, nccl_real(B.dtype), q, c.comm, c.stream));
            if (recv_counts[q]) HB_NCCL(c.api.Recv((char*)tail_t + ro * tb, recv_counts[q] * te, nccl_real(B.dtype), q, c.comm, c.stream));
            so += send_counts[q];
            ro += recv_counts[q];
        }
        HB_NCCL(c.api.GroupEnd());
        HB_CUDA(cudaEventRecord(c.ev_x1, c.stream));
        HB_CUDA(cudaEventRecord(c.ev_tiles, c.stream));
    }

    // 4. the engine product: own-only C tiles first, the halo readers behind the transfer
    try {
        op_product_begin(A, tA, B, tB, C, o, /*defer_halo_tiles=*/true, /*launch=*/true, /*launch_in_finish=*/false);
        op_product_finish(C, exchange ? c.ev_tiles : nullptr, n_mults, n_blocks);
    } catch (...) {
        if (exchange) cudaStreamSynchronize(c.stream);
        op_product_abort();
        commit_halo(B, 0);
        throw;
    }
    commit_halo(B, 0);   // (finish synchronised the engine stream behind the transfer: pack and send_idx may go)
    st.plan_ms = t_plan.ms();
    if (exchange) {
        float x = 0;
        cudaEventElapsedTime(&x, c.ev_x0, c.ev_x1);
        st.exchange_ms = x;
    }
    st.sent_tiles = n_out;
    st.recv_tiles = n_in;
    st.publish_ms = c.last.publish_ms;
    c.last = st;
}

// leaf products per C block row over all ranks: every rank counts its own rows against the published table of op(B) (a
// structure-only stand-in for the whole operand), the per-row counts are summed over the ranks (rows are disjoint)
void sharded_row_weights(const Matrix& A, bool tA, const Matrix& B, bool tB, const ProductOpts& o, int grid_side, uint64_t* host_out) {
    Comm& c = ready_comm();
    std::lock_guard<std::mutex> lock(c.mu);
    if (!B.pub || B.pub->world != c.world) throw Error(HBSM_E_ARG, "hbsm_b200: row weights: op(B) has no published table");
    if (A.empty() || B.empty() || A.dtype != B.dtype || A.b != B.b) throw Error(HBSM_E_ARG, "hbsm_b200: row weights: bad operands");
    const Published& pb = *B.pub;
    const uint32_t g = std::max(A.grid_side(), B.grid_side());
    if (grid_side != (int)g) throw Error(HBSM_E_ARG, "hbsm_b200: row weights: grid_side must be the block-grid side of the product");
    Matrix S;   // keys + norms of the WHOLE op(B); no tiles (the count pass never touches them)
    S.dtype = B.dtype; S.b = B.b; S.M = B.M; S.N = B.N; S.sized = true;
    S.L = pb.n_all;
    S.keys.alloc(std::max<size_t>(pb.n_all, 1));
    S.norms.alloc(std::max<size_t>(pb.n_all, 1) * B.esize());
    if (pb.n_all) {
        HB_CUDA(cudaMemcpyAsync(S.keys.p, pb.keys_all.p, pb.n_all * sizeof(uint64_t), cudaMemcpyDeviceToDevice, engine().stream));
        HB_CUDA(cudaMemcpyAsync(S.norms.p, pb.norms_all.p, pb.n_all * B.esize(), cudaMemcpyDeviceToDevice, engine().stream));
    }
    DevBuf<uint64_t> cnt((size_t)g);
    cnt.zero();
    {
        DevBuf<uint64_t> mine((size_t)A.grid_side());
        product_row_counts(A, tA, S, tB, o, mine.p);
        HB_CUDA(cudaMemcpyAsync(cnt.p, mine.p, (size_t)A.grid_side() * sizeof(uint64_t), cudaMemcpyDeviceToDevice, engine().stream));
    }
    if (c.world > 1) HB_NCCL(c.api.AllReduce(cnt.p, cnt.p, (size_t)g, ncclUint64, ncclSum, c.comm, engine().stream));
    cnt.download(host_out, (size_t)g);
    sync_stream();
}

hbsm_shard_stats shard_stats_last() { return comm().last; }

}  // namespace hbsm_b200

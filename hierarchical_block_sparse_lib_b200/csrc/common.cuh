// common.cuh -- engine-wide helpers: error handling, the engine singleton (device, stream, memory pool),
// stream-ordered device buffers, Morton keys.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>
#include <algorithm>
#include <utility>
#include <atomic>
#include <mutex>
#include "../../include/hbsm_b200.h"

namespace hbsm_b200 {

struct Error : public std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define HB_CUDA(expr)                                                                          \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess)                                                                 \
            throw ::hbsm_b200::Error(HBSM_E_CUDA, std::string("CUDA error: ") +                \
                                     cudaGetErrorString(_e) + " at " __FILE__ ":" +            \
                                     std::to_string(__LINE__));                                \
    } while (0)

// the reference's own exception text is preserved: "Error in HierarchicalBlockSparseMatrix<Treal>::..."
[[noreturn]] inline void throw_ref(const char* msg) { throw Error(HBSM_E_RUNTIME, msg); }

// Process-wide state.  The reference's multiply/spamm/add are re-entrant statics (H:255-305) and its stated caller is a
// worker pool, so everything that carries per-call state lives in the per-THREAD Engine below; only the device choice, the
// launch counter and the debug switch are shared.
struct Shared {
    std::atomic<int> device{-1};
    std::atomic<uint64_t> launches{0};     // kernels launched by this library, all threads
    std::atomic<int> gemm_variant{0};      // 0 tensor-core kernels, 1 generic FMA kernel, 3 fp32 single-C-tile kernels (hbsm_set_gemm_variant)
    std::mutex index_mutex;                // lazily built line indices of matrices shared between threads
};
Shared& shared();

// Exact-size cache of LARGE blocks in front of the stream-ordered pool, one per host thread (its blocks are only ever reused on
// that thread's engine stream, so stream order is kept).  The pool itself never gives memory back (unbounded release
// threshold), but handing out a GB-sized block from fragmented free space makes it re-map physical chunks into a new
// contiguous range: 30-600 ms per allocation, measured in the per-rank host-to-host loop (assign A, B; product; free
// everything; repeat) where the uploads themselves take 26 ms.  Loops like that ask for the same sizes again and again.
struct BlockCache {
    static constexpr size_t MIN_BYTES = (size_t)64 << 20;
    static constexpr size_t MAX_BLOCKS = 12;
    static constexpr size_t MAX_TOTAL = (size_t)32 << 30;   // never hold more than this back from the pool (180 GB devices)
    std::vector<std::pair<size_t, void*>> blocks;   // oldest first
    size_t total = 0;
    void* take(size_t bytes) {
        for (size_t i = blocks.size(); i-- > 0;)
            if (blocks[i].first == bytes) {
                void* p = blocks[i].second;
                blocks.erase(blocks.begin() + (long)i);
                total -= bytes;
                return p;
            }
        return nullptr;
    }
    // keeps the block unless it is too large to keep; fills `evicted` with the blocks the caller must hand to the pool
    void give(size_t bytes, void* p, std::vector<void*>& evicted) {
        if (bytes > MAX_TOTAL) { evicted.push_back(p); return; }
        blocks.emplace_back(bytes, p);
        total += bytes;
        while (blocks.size() > MAX_BLOCKS || total > MAX_TOTAL) {
            total -= blocks.front().first;
            evicted.push_back(blocks.front().second);
            blocks.erase(blocks.begin());
        }
    }
    void drop_all() { for (auto& b : blocks) cudaFree(b.second); blocks.clear(); total = 0; }   // (errors ignored: at process exit the runtime may be gone)
};

// Per host thread: its own stream, mailbox, pending product and stage times.  Two threads can run products concurrently on
// their own streams; a handle may be used by one thread at a time (like the reference's objects), any thread after another.
struct Engine {
    int device = -1;
    int sm_count = 0;
    int cc_major = 0, cc_minor = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;   // second compute stream: the halo-reading leaf GEMM of a sharded product
    uint64_t launches = 0;  // kernels launched by this thread
    bool ready = false;
    std::string name;
    int last_gemm_kernel = 0;  // which leaf kernel the last product ran: 0 generic FMA, 1 fp64 TMA-tiled DMMA, 3 fp32 tcgen05
    hbsm_stage_times last{};
    // pinned, device-mapped host words: kernels post the few scalars the host needs between launches (sizes of the next
    // allocations) straight into host memory, so those read-backs never queue on a PCIe copy engine behind bulk transfers
    uint64_t* mailbox = nullptr;
    BlockCache cache;   // large blocks this thread freed, for exact-size reuse
    ~Engine();
};
Engine& engine();
void ensure_engine();

// every kernel launch goes through this so gpu_launches can be reported honestly
#define HB_LAUNCH(kernel, grid, block, smem, ...)                                              \
    do {                                                                                       \
        kernel<<<(grid), (block), (smem), ::hbsm_b200::engine().stream>>>(__VA_ARGS__);        \
        ::hbsm_b200::engine().launches++;                                                      \
        ::hbsm_b200::shared().launches.fetch_add(1, std::memory_order_relaxed);                \
        HB_CUDA(cudaGetLastError());                                                           \
    } while (0)

// stream-ordered device buffer (cudaMallocAsync pool with an unbounded release threshold = caching allocator)
template <typename T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    DevBuf() {}
    explicit DevBuf(size_t count) { alloc(count); }
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), n(o.n) { o.p = nullptr; o.n = 0; }
    DevBuf& operator=(DevBuf&& o) noexcept {
        if (this != &o) { release(); p = o.p; n = o.n; o.p = nullptr; o.n = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    void alloc(size_t count) {
        release();
        n = count;
        if (count == 0) return;
        ensure_engine();
        const size_t bytes = std::max<size_t>(count * sizeof(T), 256);
        if (bytes >= BlockCache::MIN_BYTES && (p = (T*)engine().cache.take(bytes)) != nullptr) return;
        cudaError_t err = cudaMallocAsync((void**)&p, bytes, engine().stream);
        if (err == cudaErrorMemoryAllocation && !engine().cache.blocks.empty()) {   // the cache must never be the reason for an OOM
            cudaGetLastError();
            cudaStreamSynchronize(engine().stream);
            engine().cache.drop_all();
            err = cudaMallocAsync((void**)&p, bytes, engine().stream);
        }
        if (err != cudaSuccess) { p = nullptr; n = 0; }
        HB_CUDA(err);
    }
    void release() {
        if (p) {
            const size_t bytes = std::max<size_t>(n * sizeof(T), 256);
            if (bytes >= BlockCache::MIN_BYTES && engine().ready) {
                std::vector<void*> evicted;
                engine().cache.give(bytes, p, evicted);
                for (void* q : evicted) cudaFreeAsync(q, engine().stream);
            } else {
                cudaFreeAsync(p, engine().stream);
            }
            p = nullptr;
        }
        n = 0;
    }
    void zero() { if (p && n) HB_CUDA(cudaMemsetAsync(p, 0, n * sizeof(T), engine().stream)); }
    void upload(const T* host, size_t count) {
        if (count) HB_CUDA(cudaMemcpyAsync(p, host, count * sizeof(T), cudaMemcpyHostToDevice, engine().stream));
    }
    void download(T* host, size_t count) const {
        if (count) HB_CUDA(cudaMemcpyAsync(host, p, count * sizeof(T), cudaMemcpyDeviceToHost, engine().stream));
    }
    std::vector<T> to_host() const {
        std::vector<T> v(n);
        download(v.data(), n);
        HB_CUDA(cudaStreamSynchronize(engine().stream));
        return v;
    }
};

inline void sync_stream() { HB_CUDA(cudaStreamSynchronize(engine().stream)); }

// splitmix64: the hash of the seeded generators (generate_decay, generators.py), the task checksum and the Lanczos start vector
__host__ __device__ inline uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// ---- Morton keys: digit = 2*colbit + rowbit (H:52-56), most significant level first ----
__host__ __device__ inline uint64_t spread_bits(uint32_t x) {
    uint64_t v = x;
    v = (v | (v << 16)) & 0x0000FFFF0000FFFFull;
    v = (v | (v << 8)) & 0x00FF00FF00FF00FFull;
    v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v << 2)) & 0x3333333333333333ull;
    v = (v | (v << 1)) & 0x5555555555555555ull;
    return v;
}
__host__ __device__ inline uint32_t compact_bits(uint64_t v) {
    v &= 0x5555555555555555ull;
    v = (v | (v >> 1)) & 0x3333333333333333ull;
    v = (v | (v >> 2)) & 0x0F0F0F0F0F0F0F0Full;
    v = (v | (v >> 4)) & 0x00FF00FF00FF00FFull;
    v = (v | (v >> 8)) & 0x0000FFFF0000FFFFull;
    v = (v | (v >> 16)) & 0x00000000FFFFFFFFull;
    return (uint32_t)v;
}
__host__ __device__ inline uint64_t morton_encode(uint32_t bi, uint32_t bj) {
    return spread_bits(bi) | (spread_bits(bj) << 1);
}
__host__ __device__ inline uint32_t morton_row(uint64_t key) { return compact_bits(key); }
__host__ __device__ inline uint32_t morton_col(uint64_t key) { return compact_bits(key >> 1); }
__host__ __device__ inline uint64_t morton_transpose(uint64_t key) {
    return ((key & 0x5555555555555555ull) << 1) | ((key >> 1) & 0x5555555555555555ull);
}

struct EventTimer {
    cudaEvent_t a = nullptr, b = nullptr;
    EventTimer() { cudaEventCreate(&a); cudaEventCreate(&b); }
    ~EventTimer() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
    void start() { cudaEventRecord(a, engine().stream); }
    void stop() { cudaEventRecord(b, engine().stream); }
    double ms() { float t = 0; cudaEventSynchronize(b); cudaEventElapsedTime(&t, a, b); return t; }
};

// ---- primitives.cu ----
// post up to two device scalars (either may be null) into the engine's host mailbox and wait: returns {*a, *b}
std::pair<uint64_t, uint64_t> read_scalars(const uint64_t* d_a, const uint64_t* d_b);
// exclusive prefix sum of n uint32 counts into uint64 offsets; out[n] = total (out has n+1 entries)
void exclusive_scan_u32(const uint32_t* d_in, uint64_t* d_out, size_t n);
// stable LSD radix sort of (key,value) pairs on the low `key_bits` bits; result left in d_keys/d_vals
void radix_sort_pairs(uint64_t* d_keys, uint32_t* d_vals, size_t n, int key_bits);
// same, on bits [lo_bit, key_bits) only (stable: ties keep their input order)
void radix_sort_pairs_bits(uint64_t* d_keys, uint32_t* d_vals, size_t n, int lo_bit, int key_bits);

}  // namespace hbsm_b200

// matrix.cuh -- the flat (Morton block table) replacement for the reference's pointer quadtree (H:37-60).
//
// HBM layout of one matrix:
//   keys  [L]            uint64  ascending Morton keys of the existing leaf tiles (digit = 2*colbit + rowbit, H:52-56)
//   tiles [L][b*b]       Treal   dense column-major tiles (H:715) in key order; for b in {32,64,128,256} every tile
//                                starts on a 128-byte boundary (b*b*sizeof(Treal) is a multiple of 128)
//   norms [L]            Treal   cached leaf ||.||_F^2 (frob_norm_squared_internal of the leaves, H:48); zero until
//                                update_internal_info (H:3905) -- products/add/transpose leave it stale, as upstream
// plus lazily built line indices (tiles grouped by block row or by block column) used by the task-list builder.
#pragma once
#include "common.cuh"
#include <memory>

namespace hbsm_b200 {

// tiles grouped by line (block row or block column), inside a line ascending in the other coordinate
struct LineIndex {
    bool valid = false;
    uint32_t n_lines = 0;
    DevBuf<uint32_t> ptr;    // [n_lines + 1]
    DevBuf<uint32_t> other;  // [L] the other block coordinate
    DevBuf<uint32_t> tile;   // [L] index into keys/tiles/norms
    cudaEvent_t ready_ev = nullptr;    // recorded behind the build, on ...
    cudaStream_t built_on = nullptr;   // ... this stream (the building thread's)
    void reset() { valid = false; n_lines = 0; ptr.release(); other.release(); tile.release(); }
    LineIndex() {}
    LineIndex(const LineIndex&) = delete;
    LineIndex& operator=(const LineIndex&) = delete;
    ~LineIndex() { if (ready_ev) cudaEventDestroy(ready_ev); }
};

// (Morton key, leaf norm^2) table of a row-sharded matrix gathered on every rank (sharded.cu, hbsm_publish): rank-major, each
// rank's part in its own (ascending Morton) tile order
struct Published {
    int world = 0, rank = 0;
    std::vector<size_t> offsets;   // [world + 1]
    size_t n_all = 0;
    DevBuf<uint64_t> keys_all;     // [n_all]
    DevBuf<char> norms_all;        // [n_all] Treal
};

struct Matrix {
    int dtype = HBSM_F64;
    int b = -1;
    int M = 0, N = 0;
    bool sized = false;
    size_t L = 0;
    DevBuf<uint64_t> keys;
    DevBuf<char> tiles;
    DevBuf<char> norms;
    double root_norm_cached = 0.0;  // frob_norm_squared_internal of the root, stored exactly (float values fit)
    size_t n_mults = 0;
    LineIndex by_row, by_col;
    // halo tail (multi-GPU): keys/norms/tiles have room for `halo_cap` more tiles after the L owned ones; the first
    // `n_halo` of them hold tiles received from peer ranks for the next product in which this matrix is op(B).
    // Halo keys are NOT merged into the sorted table: the product only needs (line, other, tile index) triples.
    size_t halo_cap = 0, n_halo = 0;
    LineIndex ext_by_row, ext_by_col;   // line indices over the L + n_halo tiles
    // executed products of the call that produced this matrix (parity hook, hbsm_export_tasks)
    DevBuf<uint64_t> task_begin;    // [L + 1]
    DevBuf<uint32_t> task_k;        // [P]
    size_t n_tasks = 0;
    // set by the one call that returns before its device work on this matrix is complete (hbsm_product_from_host: C's table
    // is still merging when the host results are done); the next C-ABI call on the handle orders itself behind it
    cudaEvent_t pending_ev = nullptr;
    std::unique_ptr<Published> pub;   // valid until the matrix (or its cached norms) changes
    Matrix() {}
    Matrix(const Matrix&) = delete;
    Matrix& operator=(const Matrix&) = delete;
    ~Matrix() { if (pending_ev) cudaEventDestroy(pending_ev); }

    size_t esize() const { return dtype == HBSM_F64 ? 8 : 4; }
    size_t tile_elems() const { return (size_t)b * (size_t)b; }
    size_t tile_bytes() const { return tile_elems() * esize(); }
    bool empty() const { return !sized; }
    // virtual depth P (H:521-541): 0 when the matrix is a single leaf
    int vdepth() const { return depth_for(M, N, b); }
    static int depth_for(int m, int n, int bs) {
        if (m <= bs && n <= bs) return 0;
        int maxdim = m > n ? m : n;
        int covers = maxdim / bs + (maxdim % bs != 0);
        int P = 1, two = 2;
        while (covers > two) { two *= 2; ++P; }
        return P;
    }
    uint32_t grid_side() const { return 1u << vdepth(); }
    void invalidate_indices() { by_row.reset(); by_col.reset(); ext_by_row.reset(); ext_by_col.reset(); }
    size_t n_ext() const { return L + n_halo; }
    void drop_tasks() { task_begin.release(); task_k.release(); n_tasks = 0; }
    void clear();                     // H:614
    void resize(int m, int n);        // H:544
    void set_table(DevBuf<uint64_t>&& k, DevBuf<char>&& t, size_t count);  // adopt a sorted table, zero norms
};

// ---- matrix.cu ----
void assign_coo(Matrix& A, size_t n, const int* rows, const int* cols, const void* vals, bool use_max, bool checked);
void assign_tiles_host(Matrix& A, size_t n_tiles, const int* bi, const int* bj, const void* tiles);
void assign_tiles_device(Matrix& A, size_t n_tiles, const uint64_t* d_keys, const void* d_tiles, const void* d_norms);
void get_values(const Matrix& A, size_t n, const int* rows, const int* cols, void* out);
size_t get_all_values(const Matrix& A, size_t cap, int* rows, int* cols, void* vals);
size_t count_nnz(const Matrix& A);
bool export_tile(const Matrix& A, uint32_t bi, uint32_t bj, void* host_buf);   // false = no such tile
uint64_t task_checksum(const Matrix& C);   // order-independent checksum of C's recorded executed-product set
long long tile_tasks(const Matrix& C, uint32_t bi, uint32_t bj, size_t cap, int64_t* k_out);   // -1 = no such tile
void compute_leaf_norms(const Matrix& A, void* d_out);   // bit-exact sequential sum per leaf (H:646-652)
void compute_leaf_norms_range(const Matrix& A, size_t t0, size_t cnt, void* d_out_base);
double hierarchical_norm(const Matrix& A, const void* d_leaf_norms);   // root value of H:3918-3923 / H:656-662
void update_norms(Matrix& A);
double frob_squared(const Matrix& A);
const LineIndex& line_index(const Matrix& A, bool by_col, bool with_halo = false);
void reserve_halo(Matrix& A, size_t cap, uint64_t** d_keys, void** d_norms, void** d_tiles);   // tail pointers
void commit_halo(Matrix& A, size_t n_halo);
void op_add(const Matrix& A, const Matrix& B, Matrix& C);
void op_transpose(const Matrix& A, Matrix& C);
void op_upper(const Matrix& A, Matrix& C);
void op_rescale(Matrix& C, const Matrix& A, double alpha);
void op_copy(Matrix& C, const Matrix& A);
bool op_trunc(const Matrix& A, Matrix& C, double trunc_value);   // frob_block_trunc, H:4935; true if something was removed
// the pieces every truncation shares.  trunc_begin: C = A's shape, n_mults and stale root norm, without tiles; false when
// nothing can be dropped (unsized, no tiles, or a single leaf, which is copied whole).  trunc_keep_flags: keep[t] = 0 iff
// leaf t's ||.||_F^2 (d_nsq, Treal) < trunc_value^2 in Treal.  trunc_compact: C's tiles = A's tiles with keep[t] != 0, in
// A's order, with zero (stale) cached norms; returns how many.  scan_flags: exclusive scan of n flags into pos[n + 1],
// returns the total (synchronises).
bool trunc_begin(const Matrix& A, Matrix& C);
void trunc_keep_flags(const Matrix& A, const void* d_nsq, double trunc_value, uint32_t* keep);
size_t trunc_compact(const Matrix& A, const DevBuf<uint32_t>& keep, Matrix& C);
size_t scan_flags(const DevBuf<uint32_t>& flags, size_t n, DevBuf<uint64_t>& pos);
// merge-union of two ascending key lists (op_add's): ukeys ascending, src_a[u] / src_b[u] = the index of ukeys[u] in ka / kb, or
// 0xffffffff where absent; returns the union's size (synchronises)
size_t key_union(const uint64_t* ka, size_t na, const uint64_t* kb, size_t nb, DevBuf<uint64_t>& ukeys, DevBuf<uint32_t>& src_a,
                 DevBuf<uint32_t>& src_b);
// for t < n: tile o = dst[t] of tout = fl(alpha * tile src[o] of X), alpha rounded to X's dtype first (op_rescale's arithmetic)
void scale_tiles_into(const Matrix& X, const uint32_t* src, const uint32_t* dst, size_t n, double alpha, void* tout);
bool op_extract_quadrant(const Matrix& A, int q, Matrix& C);        // false = absent; child q (0=TL 1=BL 2=TR 3=BR, H:52-56) as its own matrix
void op_assemble_quadrants(Matrix& C, int M, int N, const Matrix* quads[4]);   // inverse; null / empty = absent child
void op_leaf_inv_chol(const Matrix& A, Matrix& Z, int zdim, int valid);   // dense leaf step of inv_chol, H:3118-3147
void sym_expand(const Matrix& A, Matrix& S);             // S = triu(A) + striu(A)^T as a full matrix
void mask_diag_upper(Matrix& C);                         // zero the strict lower part of diagonal tiles in place
void generate_decay(Matrix& A, int n, const double* table, int W, uint64_t seed, bool symmetric, int lo, int hi);

// ---- serialize.cu: the reference's wire format (H:1124-1487) ----
size_t serialized_size(const Matrix& A);
void serialize(const Matrix& A, char* buf, size_t cap);
void deserialize(Matrix& A, const char* buf, size_t size);

// ---- estimators.cu: a-priori skip counts / error bounds from cached norms (H:4945, H:5236) ----
void count_skips(const Matrix& A, bool tA, const Matrix& B, bool tB, size_t n, const double* taus, bool apply_truncation, bool apply_spamm,
                 unsigned long* out);
size_t spamm_errors(const Matrix& A, bool tA, const Matrix& B, bool tB, size_t n, const double* taus, double* out);   // returns 0 or n

// ---- product.cu ----
struct ProductOpts {
    bool spamm = false;
    double tau = 0.0;
    bool updated = true;
    bool upper_only = false;   // keep only C tiles with ci <= cj (symm_square / symm_rk)
    // accumulating product (hbsm_multiply_accumulate): C <- alpha*P + beta*C_old, where C_old is c_old's table when the product
    // begins (c_old is C itself; it may also be A or B).  nullptr: the plain product, C overwritten.
    const Matrix* c_old = nullptr;
    double alpha = 1.0, beta = 0.0;
};
void op_product(const Matrix& A, bool tA, const Matrix& B, bool tB, Matrix& C, const ProductOpts& o,
                size_t* n_mults, size_t* n_blocks);
// split form for the multi-GPU overlap: begin builds the task list and starts the leaf GEMMs of the C tiles that only read
// B's own tiles (when defer_halo_tiles and B has a committed halo whose TILES are still in flight); finish waits for
// `wait_for` (may be null), computes the remaining C tiles and completes C.  One product in flight at a time.
void op_product_begin(const Matrix& A, bool tA, const Matrix& B, bool tB, Matrix& C, const ProductOpts& o, bool defer_halo_tiles,
                      bool launch = true, bool launch_in_finish = false);
void op_product_to_host(const Matrix& A, bool tA, const Matrix& B, bool tB, Matrix& C, const ProductOpts& o, void* host_tiles,
                        size_t cap_tiles, int n_chunks, size_t* n_mults, size_t* n_blocks);
void op_product_finish(Matrix& C, cudaEvent_t wait_for, size_t* n_mults, size_t* n_blocks);
// The whole host-to-host call in one pipeline: A and B (sized, without tiles) are assembled from HOST tiles, their norms
// refreshed, C = op(A)*op(B) computed and its tiles delivered to HOST memory, with the PCIe uploads, the leaf GEMMs and the
// downloads overlapped block-row slab by block-row slab.  Same end state as assign_tiles(A); assign_tiles(B);
// update_norms(A); update_norms(B); product(A,B,C).  host_c_tiles/c_bi/c_bj receive C's tiles and block coordinates in
// slab-major order (Morton order inside a slab).
struct HostTiles { size_t n; const int* bi; const int* bj; const void* tiles; };
void op_product_from_host(Matrix& A, const HostTiles& ha, bool tA, Matrix& B, const HostTiles& hb, bool tB, Matrix& C,
                          const ProductOpts& o, int n_slabs, void* host_c_tiles, size_t cap_tiles, int* c_bi, int* c_bj,
                          size_t* n_mults, size_t* n_blocks);
void op_product_abort();
void product_row_counts(const Matrix& A, bool tA, const Matrix& B, bool tB, const ProductOpts& o, uint64_t* d_out);
// op_product's operand checks of a SpAMM product (same codes and messages), without a target and before any device work
void check_spamm_operands(const Matrix& A, bool tA, const Matrix& B, bool tB, bool updated);
// The candidate leaf pairs of op(A)*op(B): every (ci, k, cj) with both tiles present (only C tiles with ci <= cj when
// upper_only), planned by the task-list builder without SpAMM.  begin[n_ctiles + 1] and ab[Q] = (A tile, B tile), grouped by
// C tile in the order the product runs them; returns Q (begin and ab stay unallocated when Q == 0).
size_t product_candidates(const Matrix& A, bool tA, const Matrix& B, bool tB, bool upper_only, DevBuf<uint64_t>& begin,
                          DevBuf<uint2>& ab, size_t* n_ctiles);
// ---- spamm_error.cu: SpAMM error control (DESIGN section 12) ----
struct SpammTol {
    double tau, bound, level;
    size_t n_candidates, n_skipped, n_levels;
};
void spamm_error_bounds(const Matrix& A, bool tA, const Matrix& B, bool tB, bool symm_square, bool updated, size_t n,
                        const double* taus, double* bounds, size_t* n_skipped);
SpammTol spamm_tau_for_error(const Matrix& A, bool tA, const Matrix& B, bool tB, bool symm_square, bool updated, double eps);
// ---- dense.cu: Y = alpha*op(A)*X + beta*Y with dense column-major X, Y in A's dtype (op: HBSM_OP_*), Lanczos on it ----
void validate_dense(const Matrix& A, int op, int m, long long ldx, long long ldy, const void* X, const void* Y);   // HBSM_E_ARG
void dense_product_device(const Matrix& A, int op, int m, const void* d_X, long long ldx, void* d_Y, long long ldy, double alpha,
                          double beta);   // engine stream
void dense_product_host(const Matrix& A, int op, int m, const void* X, long long ldx, void* Y, long long ldy, double alpha,
                        double beta);     // synchronous
struct SpectralResult { double norm, lambda_min, lambda_max; int n_iter; };
SpectralResult spectral_norm(const Matrix& A, bool symmetric_upper, int max_iter, double rel_tol);
// The operator the dense product walks: A's tiles through row and column line arrays (ptr[n_lines + 1], other, tile), each
// line contiguous and ascending in `other` -- A's own line indices, or any subset of them (spectral_trunc.cu's masked index)
struct LineView { const uint32_t *ptr = nullptr, *other = nullptr, *tile = nullptr; };
struct OpView { LineView row, col; };
OpView own_view(const Matrix& A);   // A's own row and column line indices (built if needed)
// Decision mode of the Lanczos driver: stop as soon as ||op||_2 <= eps or > eps is decided (dense.cu, decide())
struct LanczosDecision {
    double eps;        // in
    bool feasible;     // out: the operator's norm is <= eps (certified up to the Lanczos caveat), false when undecided
    double bound;      // out: the upper estimate of the norm at the last step (theta + residual bound, in norm units)
};
// Lanczos on the operator of `view` (A's shape, dtype and leaf size); dec == nullptr: the full-convergence run of
// spectral_norm (A validated and holding tiles); else decision mode, accepting only once the extreme pairs converged to rel_tol.
SpectralResult lanczos(const Matrix& A, const OpView& view, bool symmetric_upper, int max_iter, double rel_tol, LanczosDecision* dec);
// ---- spectral_trunc.cu: truncation with spectral-norm error control ----
struct TruncInfo {
    size_t n_dropped, n_frob;
    double drop_nsq, err_bound;
    bool certified_by_lanczos;
    int n_decisions;
    long long lanczos_steps;
};
TruncInfo spectral_block_trunc(const Matrix& A, bool symmetric_upper, double eps, int max_iter, Matrix& C);
void truncation_spectral_errors(const Matrix& A, bool symmetric_upper, size_t n, const double* taus, int max_iter, double rel_tol,
                                double* out_norms, int* out_iters);
// ---- sharded.cu: one process per GPU, NCCL resolved at run time ----
void comm_set_library(const char* path);
void comm_unique_id(void* out128);
void comm_init(const void* id128, int rank, int world);
void comm_finalize();
void comm_info(int* rank, int* world, int* nccl_version);
void comm_allreduce_f64(double* vals, int n, bool take_max);
void comm_allgather_u64(const uint64_t* mine, size_t n, uint64_t* all);
void comm_barrier();
void publish(Matrix& B);
void sharded_product(const Matrix& A, bool tA, Matrix& B, bool tB, Matrix& C, const ProductOpts& o, size_t* n_mults, size_t* n_blocks);
void sharded_row_weights(const Matrix& A, bool tA, const Matrix& B, bool tB, const ProductOpts& o, int grid_side, uint64_t* host_out);
hbsm_shard_stats shard_stats_last();
bool worth_product(const Matrix& A, bool tA, const Matrix& B, bool tB, bool spamm, double tau);

}  // namespace hbsm_b200

/* hbsm_b200.h -- C ABI of the B200-native engine for the quadtree multiply / SpAMM / add hot path of
 * toxaart/hierarchical_block_sparse_lib.
 *
 * The reference has no FFI layer: its boundary is the public section of the header-only class
 * hbsm::HierarchicalBlockSparseMatrix<Treal> (reference source/HierarchicalBlockSparseMatrix.h:166-428,
 * cited below as H:<line>).  Each entry point here is what a binding of that class would call; the
 * drop-in C++ class over this ABI is include/hbsm/HierarchicalBlockSparseMatrix.h.
 *
 * Conventions: every function returns 0 on success or an HBSM_E_* code; hbsm_last_error() returns the
 * thread-local message (the reference's own exception text where one exists).  All pointers are HOST
 * pointers unless the parameter name starts with d_.  `void*` value buffers hold double (HBSM_F64) or
 * float (HBSM_F32) according to the handle's dtype.  Calls are synchronous with respect to returned host
 * data.  There is NO CPU fallback: every call fails with HBSM_E_CUDA if no sm_100 device is usable.
 */
#ifndef HBSM_B200_H
#define HBSM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

typedef struct hbsm_matrix_s* hbsm_handle;

enum { HBSM_F64 = 0, HBSM_F32 = 1 };

enum {
    HBSM_OK = 0,
    HBSM_E_CUDA = 1,      /* CUDA runtime / no device */
    HBSM_E_ARG = 2,       /* invalid argument */
    HBSM_E_RUNTIME = 3    /* the reference would throw std::runtime_error; message in hbsm_last_error() */
};

/* Stage timings (milliseconds, CUDA events on the engine stream) of the most recent product call. */
typedef struct hbsm_stage_times_s {
    double norms_ms;      /* leaf norm refresh inside the call (0 when updated=true) */
    double index_ms;      /* row/column line indices of op(A), op(B) */
    double tasklist_ms;   /* count + fill + C table ordering */
    double gemm_ms;       /* leaf GEMM kernel(s) */
    double total_ms;      /* whole call, first kernel to last */
    uint64_t n_candidates;/* Q: leaf pairs tested */
    uint64_t n_products;  /* P: leaf products executed */
    uint64_t n_ctiles;    /* tiles of C */
    uint64_t gpu_launches;/* kernels launched by the call */
    uint64_t gemm_kernel; /* leaf kernel used: 0 generic FMA, 1 fp64 TMA-tiled DMMA, 3 fp32 tcgen05 (2 is retired) */
} hbsm_stage_times;

/* ---- library ---- */
int hbsm_init(int device);                 /* select device, create the engine stream; idempotent */
int hbsm_finalize(void);
const char* hbsm_last_error(void);
int hbsm_device_info(char* name, size_t cap, int* sm_count, int* cc_major, int* cc_minor);
uint64_t hbsm_kernel_launch_count(void);   /* kernels launched by this library since init */

/* ---- lifetime, sizing (ctor/dtor H:171-178, set_params H:186, resize H:194, clear H:196) ---- */
int hbsm_create(int dtype, hbsm_handle* out);
int hbsm_destroy(hbsm_handle h);
int hbsm_set_blocksize(hbsm_handle h, int blocksize);     /* H:450: throws unless empty */
int hbsm_get_blocksize(hbsm_handle h, int* blocksize);    /* H:457 */
int hbsm_resize(hbsm_handle h, int n_rows, int n_cols);   /* H:544 */
int hbsm_clear(hbsm_handle h);                            /* H:614 */
int hbsm_is_empty(hbsm_handle h, int* out);               /* H:470 */
int hbsm_children_exist(hbsm_handle h, int* out);         /* H:464 */
int hbsm_dims(hbsm_handle h, int* n_rows, int* n_cols);   /* H:588, H:601 */
int hbsm_depth(hbsm_handle h, int* out);                  /* H:496 */
int hbsm_expected_depth(hbsm_handle h, int* out);         /* H:521 */
int hbsm_is_consistent(hbsm_handle h, int* out);          /* H:1809 */
int hbsm_dtype(hbsm_handle h, int* out);

/* ---- assembly / readback (H:668-849, H:852-1121) ---- */
int hbsm_assign_coo(hbsm_handle h, size_t n, const int* rows, const int* cols, const void* vals,
                    int use_max, int boundaries_checked);
/* bulk path: whole dense column-major tiles, tile t at block coordinates (bi[t], bj[t]); coordinates unique */
int hbsm_assign_tiles(hbsm_handle h, size_t n_tiles, const int* bi, const int* bj, const void* tiles);
int hbsm_get_values(hbsm_handle h, size_t n, const int* rows, const int* cols, void* out);      /* H:1012 */
int hbsm_get_all_values(hbsm_handle h, size_t cap, int* rows, int* cols, void* vals, size_t* n); /* H:1034; cap=0 -> count */
/* parity hook: the dense column-major tile at block coordinates (bi, bj) -> host_tile (b*b elements); *found = 0 if absent */
int hbsm_export_tile(hbsm_handle h, int bi, int bj, void* host_tile, int* found);
int hbsm_nnz(hbsm_handle h, size_t* out);                 /* H:985 */
int hbsm_n_blocks(hbsm_handle h, size_t* out);            /* H:7311 */
int hbsm_get_n_block_multiplications(hbsm_handle h, size_t* out);   /* H:218 */
int hbsm_set_n_block_multiplications(hbsm_handle h, size_t n);      /* H:220 */

/* ---- norms (H:641 get_frob_squared, H:3905 update_internal_info, H:216 cached getter) ---- */
int hbsm_update_norms(hbsm_handle h);
int hbsm_frob_squared(hbsm_handle h, void* out);
int hbsm_frob_squared_cached(hbsm_handle h, void* out);

/* ---- products (multiply H:2142/H:260, spamm H:3931/H:305) ---- */
int hbsm_multiply(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C,
                  size_t* n_block_multiplies, size_t* n_resizes);
int hbsm_spamm(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, double tau, int updated,
               size_t* n_block_multiplies, size_t* n_resizes);
/* The same product in two calls, for callers that overlap a transfer with it (multi-GPU): begin builds the task list and
 * launches the leaf GEMMs of every C tile that reads only B's own tiles (defer_halo_tiles != 0 and a halo committed with
 * hbsm_halo_commit whose keys and norms are valid but whose TILES are still arriving); finish makes the engine stream wait
 * for `cuda_event_or_null` (a cudaEvent_t recorded after the transfer), computes the remaining C tiles and completes C
 * exactly as hbsm_multiply / hbsm_spamm would.  One product may be in flight at a time.
 * defer_halo_tiles = 2: begin only plans (task list + the split); finish launches the own-only C tiles, waits for the
 * event, launches the rest.  Use it when the transfer is queued between the two calls: kernels queued BEFORE the
 * persistent leaf GEMM (one CTA per SM) get their SMs first, kernels queued after it wait for it to drain (measured at 8
 * GPUs: the NCCL all-to-all of the halo tiles ran only after the first GEMM, 0.6 ms of a 5.6 ms step). */
int hbsm_product_begin(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, int spamm, double tau, int updated,
                       int defer_halo_tiles);
int hbsm_product_finish(hbsm_handle C, void* cuda_event_or_null, size_t* n_block_multiplies, size_t* n_resizes);
/* drops the calling thread's product in flight, if any (a caller whose transfer failed between begin and finish); a C
 * that was empty at begin is empty again.  A rejected begin leaves C as it was; a finish on another C is refused and
 * drops the product the same way. */
int hbsm_product_abort(void);
/* the same begin with the symmetric-family option: upper_only != 0 plans only the C tiles with ci <= cj and finish zeroes
 * the strict lower part of the diagonal tiles (symm_square H:3563 / symm_rk H:3711 on an expanded operand; sharded:
 * triu(op(A)*op(B)) of the rank's block rows) */
int hbsm_product_begin_ex(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, int spamm, double tau, int updated,
                          int defer_halo_tiles, int upper_only);
/* multiply (spamm = 0) or SpAMM whose result is ALSO delivered to host memory: the leaf GEMMs run in ranges of C's tile
 * list and every finished range is copied to `host_tiles` (pinned memory recommended; room for cap_tiles tiles, in the
 * order of hbsm_export_leaves) on a second stream while the next ranges compute.  If cap_tiles is smaller than the number
 * of C tiles nothing is copied and HBSM_E_ARG is returned after C is complete (read *n_resizes and call again / export). */
int hbsm_product_to_host(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, int spamm, double tau, int updated,
                         void* host_tiles, size_t cap_tiles, size_t* n_block_multiplies, size_t* n_resizes);
/* The whole host-to-host call as ONE pipeline (what a caller whose matrices live in host memory, like the reference's,
 * does per multiply): A and B are sized handles without tiles; their tiles come from HOST arrays (tile t of A at block
 * coordinates (a_bi[t], a_bj[t]), dense column-major, pinned memory recommended, Morton-ordered input streams best), are
 * uploaded block-row slab by block-row slab, their norms refreshed as they land, and every slab of C = op(A)*op(B) is
 * computed and shipped to host_c_tiles as soon as the tiles it reads have arrived: PCIe upload, leaf GEMMs and PCIe
 * download overlap.  End state = hbsm_assign_tiles(A), hbsm_assign_tiles(B), hbsm_update_norms(A), hbsm_update_norms(B),
 * hbsm_multiply / hbsm_spamm(A,B,C).  host_c_tiles (room for cap_tiles tiles), c_bi, c_bj (cap_tiles ints each, may be
 * null) receive C's tiles and their block coordinates in slab-major order (Morton order inside a slab).  n_slabs = 0
 * lets the engine choose.  HBSM_E_ARG after C is complete if cap_tiles was too small (read *n_resizes, export C). */
int hbsm_product_from_host(hbsm_handle A, size_t n_a, const int* a_bi, const int* a_bj, const void* a_tiles, int tA,
                           hbsm_handle B, size_t n_b, const int* b_bi, const int* b_bj, const void* b_tiles, int tB,
                           hbsm_handle C, int spamm, double tau, int n_slabs, void* host_c_tiles, size_t cap_tiles,
                           int* c_bi, int* c_bj, size_t* n_block_multiplies, size_t* n_resizes);
int hbsm_worth_to_multiply(hbsm_handle A, int tA, hbsm_handle B, int tB, int* out);             /* H:1873 */
int hbsm_worth_to_spamm(hbsm_handle A, int tA, hbsm_handle B, int tB, double tau, int* out);    /* H:2006 */

/* ---- structure ops (add H:1644, transpose H:3733, get_upper_triangle H:3515, rescale H:3078, copy H:1490) ---- */
int hbsm_add(hbsm_handle A, hbsm_handle B, hbsm_handle C);
int hbsm_transpose(hbsm_handle A, hbsm_handle C);
int hbsm_upper_triangle(hbsm_handle A, hbsm_handle C);
int hbsm_rescale(hbsm_handle C, hbsm_handle A, double alpha);
int hbsm_copy(hbsm_handle C, hbsm_handle A);

/* frob_block_trunc H:4935: C = A without the leaves whose ||.||_F^2 < trunc_value^2 (the hierarchical rule of H:4904
 * collapses to this flat one); *removed = 1 if any leaf was dropped.  hbsm_leaf_norms: freshly computed leaf ||.||_F^2 in
 * ascending Morton order (the order of hbsm_export_leaves), independent of the cache; cap = 0 -> count. */
int hbsm_frob_block_trunc(hbsm_handle A, hbsm_handle C, double trunc_value, int* removed);
int hbsm_leaf_norms(hbsm_handle h, size_t cap, void* out, size_t* n);

/* ---- quadrants (the recursion of inv_chol H:3110 runs on the host over these): child q of the root (0=TL 1=BL 2=TR 3=BR,
 * H:52-56) as its own matrix of the child's virtual size, and the inverse (NULL / empty handle = absent child) ---- */
int hbsm_extract_quadrant(hbsm_handle A, int q, hbsm_handle C, int* exists);   /* *exists = 0: the child is absent */
int hbsm_assemble_quadrants(hbsm_handle C, int n_rows, int n_cols, hbsm_handle q0, hbsm_handle q1, hbsm_handle q2, hbsm_handle q3);
/* the dense leaf step of inv_chol (H:3118-3147) on device: A = a single-leaf matrix, Z <- zdim x zdim single-leaf inverse
 * Cholesky factor (upper triangular, Z^T A Z = I) of its leading valid x valid block; valid <= zdim <= b <= 256 */
int hbsm_leaf_inv_chol(hbsm_handle A, hbsm_handle Z, int zdim, int valid);

/* ---- a-priori estimators from the CACHED norms (count_skips H:4945, get_spamm_errors H:5236); taus in double ---- */
int hbsm_count_skips(hbsm_handle A, int tA, hbsm_handle B, int tB, size_t n, const double* taus, int apply_truncation, int apply_spamm,
                     unsigned long* out);
/* *n_out = n, or 0 when the pair has no executable product (the reference returns an empty vector) */
int hbsm_spamm_errors(hbsm_handle A, int tA, hbsm_handle B, int tB, size_t n, const double* taus, double* out, size_t* n_out);

/* ---- wire format (get_size H:1124, write_to_buffer H:1159, assign_from_buffer H:1348): byte-compatible ---- */
int hbsm_serialized_size(hbsm_handle h, size_t* out);
int hbsm_serialize(hbsm_handle h, char* buffer, size_t capacity);
int hbsm_deserialize(hbsm_handle h, const char* buffer, size_t size);

/* ---- symmetric family, exact (symm_multiply H:3244, symm_square H:3563, symm_rk H:3711) ---- */
int hbsm_symm_multiply(hbsm_handle A, int sA, hbsm_handle B, int sB, hbsm_handle C);
int hbsm_symm_square(hbsm_handle A, hbsm_handle C);
int hbsm_symm_rk(hbsm_handle A, int transposed, hbsm_handle C);
/* SpAMM-pruned symmetric square: triu(spamm(sym(A), sym(A), tau)) -- BASELINE config 3's tau sweep */
int hbsm_symm_square_spamm(hbsm_handle A, hbsm_handle C, double tau, size_t* n_block_multiplies, size_t* n_resizes);

/* ---- block-sparse times dense multivector and spectral estimates (engine extras; the reference's spectral_norm,
 * get_row_sums, ... stubs are unchanged) ----
 * Y = alpha * op(A) * X + beta * Y.  X (K x m) and Y (M x m), K x M the shape of op(A), are dense column-major arrays in A's
 * dtype with leading dimensions ldx >= max(1, K), ldy >= max(1, M); rows of Y between M and ldy are never touched.
 * op: HBSM_OP_N (A), HBSM_OP_T (A^T), HBSM_OP_SYM_UPPER (triu(A) + striu(A)^T of a square A: tiles below the diagonal and
 * the strict lower part of diagonal tiles are ignored).  beta == 0 never reads Y.  Deterministic (bitwise repeatable).
 * Only A's own tiles are used (a committed halo plays no part).  m == 0 is a no-op.  Leaf sizes up to 256 (any size, not
 * only powers of two); a larger leaf size returns HBSM_E_ARG, from hbsm_spectral_norm too. */
enum { HBSM_OP_N = 0, HBSM_OP_T = 1, HBSM_OP_SYM_UPPER = 2 };
/* host arrays; staged with cudaMemcpyAsync, synchronous like the other host-pointer calls */
int hbsm_multiply_dense(hbsm_handle A, int op, int m, const void* X, int ldx, void* Y, int ldy, double alpha, double beta);
/* device arrays; ordered after the work already queued on cuda_stream (any stream, 0 included), and the work queued there
 * afterwards sees Y complete; no host synchronisation */
int hbsm_multiply_dense_device(hbsm_handle A, int op, int m, const void* d_X, int ldx, void* d_Y, int ldy,
                               double alpha, double beta, void* cuda_stream);
/* ||A||_2 by Lanczos: symmetric_upper = 0 -> on A^T A (one N and one T product per step), 1 -> on triu(A)+striu(A)^T
 * (lambda_min / lambda_max may be NULL; they receive the extreme Ritz values of the operator: the eigenvalue bounds of
 * triu(A)+striu(A)^T for 1, those of A^T A -- squared singular values -- for 0).  Stops when the residual bound of the extreme Ritz pair (for 1: of both extreme pairs) is <= rel_tol * the
 * largest |Ritz value|, on breakdown, or after max_iter steps; *n_iter = steps used (0 for a matrix without tiles). */
int hbsm_spectral_norm(hbsm_handle A, int symmetric_upper, int max_iter, double rel_tol,
                       double* norm, double* lambda_min, double* lambda_max, int* n_iter);

/* ---- truncation with spectral-norm error control (engine extras; the reference's get_spectral_squared_of_error_matrix
 * H:421 and spectral_norm H:427 stubs are unchanged) ----
 * A truncation at level v drops exactly the leaves whose fresh ||.||_F^2 (nsq, hbsm_leaf_norms) is <= v; E_v is the dropped
 * part.  The error operator is E_v, or triu(E_v) + striu(E_v)^T with symmetric_upper, where tiles below the diagonal play no
 * part: they are never dropped and never counted.  A single leaf (depth 0) is never truncated, as in hbsm_frob_block_trunc.
 *
 * hbsm_spectral_block_trunc: C = A without the leaves of the largest level v the search accepts with ||E_v||_2 <= eps.
 * C is exactly what hbsm_frob_block_trunc(A, C, tau) leaves for any tau with v < tau^2 <= the next distinct nsq (when A has
 * no tiles below the diagonal, with symmetric_upper): the same tiles, n_mults and stale cached norms.  The search runs over
 * the distinct levels between two rigorous brackets: the Frobenius bound (sum of nsq, of 2 nsq with symmetric_upper) <=
 * eps^2 accepts without Lanczos; a leaf off the diagonal with nsq > b eps^2 can never be dropped.  Each level in between is
 * decided by Lanczos on E_v, stopped as soon as it can decide: an extreme Ritz value above eps (eps^2 on E^T E) rejects,
 * Ritz value + residual bound <= eps, once the extreme Ritz pairs have converged to a relative residual bound of 1e-3,
 * accepts, breakdown decides with the exact Ritz values, and max_iter without a decision rejects.  Caveat: the accepting test
 * is an estimate, not a proof -- an extreme eigenvector (nearly) orthogonal to the hashed start vector can escape the Krylov
 * space, and then ||E_v||_2 may exceed eps.  Rejections are rigorous.
 * HBSM_E_ARG (before any device work): eps < 0 or NaN, max_iter < 1, C == A, symmetric_upper with a non-square A, leaf size
 * above 256.  Deterministic (bitwise repeatable). */
typedef struct {
    size_t n_dropped;          /* leaves dropped */
    double drop_nsq;           /* the level v: the largest dropped nsq; -1 when nothing is dropped */
    size_t n_frob;             /* leaves the Frobenius bound alone drops at eps */
    double err_bound;          /* the certificate of the chosen level, in norm units: sqrt(Frobenius bound), or the Lanczos
                                * upper estimate theta + residual bound */
    int certified_by_lanczos;  /* 1: the chosen level lies above the Frobenius bracket and was accepted by Lanczos */
    int n_decisions;           /* Lanczos decisions run */
    long long lanczos_steps;   /* Lanczos steps over all decisions */
} hbsm_trunc_info;
int hbsm_spectral_block_trunc(hbsm_handle A, int symmetric_upper, double eps, int max_iter, hbsm_handle C, hbsm_trunc_info* info);
/* out_norms[i] = ||E_i||_2 (triu + striu^T with symmetric_upper), E_i = the leaves hbsm_frob_block_trunc(A, C, taus[i])
 * would drop (nsq < taus[i]^2 in A's dtype), estimated exactly as hbsm_spectral_norm(max_iter, rel_tol) would for a matrix
 * holding only E_i's tiles (the same bits); out_iters[i] = its Lanczos steps (0 when E_i is empty).  HBSM_E_ARG (before any
 * device work): max_iter < 1, rel_tol <= 0, symmetric_upper with a non-square A, leaf size above 256, n > 0 with a null
 * taus / out_norms / out_iters. */
int hbsm_truncation_spectral_errors(hbsm_handle A, int symmetric_upper, size_t n, const double* taus, int max_iter, double rel_tol,
                                    double* out_norms, int* out_iters);

/* ---- SpAMM with error control (engine extras; hbsm_spamm_errors keeps the reference's a-priori estimate) ----
 * Candidates: the leaf pairs (ci, k, cj) of the exact product with A_ik of op(A) and B_kj of op(B) present (what
 * hbsm_multiply executes).  Candidate level p = fl(nsq(A_ik) * nsq(B_kj)) in the dtype, from the cached norms (updated = 1) or
 * from fresh norms in temporaries that leave the caches alone (updated = 0), exactly as hbsm_spamm forms it.  At tau a
 * candidate is skipped iff !(p > fl(tau * tau)) in the dtype (fp32: tau rounded to float first); a NaN p at every tau.
 * The bound of tau: sqrt(w * sum over C tiles t of S_t^2), S_t = the sum over t's skipped candidates of
 * s = sqrt(nsq_A) sqrt(nsq_B) / (1 - gamma), gamma = b^2 u / (1 - b^2 u) covering the rounding of the computed nsq (u the
 * dtype's unit roundoff), w = 1.  It bounds ||P_exact - P_tau||_F, hence ||.||_2, every operation rounded upward.  It bounds
 * the error of skipping in exact arithmetic: the rounding of the leaf GEMMs that do run is separate.
 * symm_square != 0: the product of hbsm_symm_square_spamm(A, C, tau) -- B must be A, tA = tB = 0, A square; the candidates
 * are those of sym_expand(A) (norms refreshed, so `updated` is ignored) with ci <= cj, the error operator sym(triu(E)), and
 * w = 2 (||sym(T)||_F^2 <= 2 ||T||_F^2 for every tile).  A committed halo of B takes part, as in hbsm_spamm.
 * A NaN level makes every bound +Inf.  No candidates: bounds 0, tau 0.  One device pass, deterministic (bitwise repeatable).
 * HBSM_E_ARG (before any device work): hbsm_spamm's operand errors (same codes and messages), n > 0 with a null taus or
 * bounds, eps < 0, NaN or infinite, symm_square with another B, a transpose or a non-square A, updated = 0 with a committed
 * halo on B. */
typedef struct {
    double tau;            /* pass to hbsm_spamm / hbsm_multiply_accumulate(spamm = 1) / hbsm_symm_square_spamm */
    double bound;          /* certified bound of that tau (<= eps), Frobenius and hence also spectral */
    double level;          /* v: largest skipped p (dtype value), -1 when nothing is skipped */
    size_t n_candidates;   /* Q */
    size_t n_skipped;      /* candidates skipped at tau: the product executes Q - n_skipped */
    size_t n_levels;       /* distinct p among the candidates */
} hbsm_spamm_tol_info;
/* bounds[i] = the bound of taus[i]; n_skipped[i] (may be NULL) = candidates skipped at taus[i] */
int hbsm_spamm_error_bounds(hbsm_handle A, int tA, hbsm_handle B, int tB, int symm_square, int updated, size_t n,
                            const double* taus, double* bounds, size_t* n_skipped);
/* The largest-skipping tau whose bound is <= eps: the highest level v with bound <= eps and a tau with v <= fl(tau * tau) <
 * the next level, so the product at tau executes exactly the candidates with p > v.  When no tau squares into that interval
 * the level below is taken; nothing skippable gives tau = 0.  HBSM_E_ARG after the pass: a NaN level, or pairs whose norm
 * product underflows to 0 (skipped at every tau) with a bound above eps. */
int hbsm_spamm_tau_for_error(hbsm_handle A, int tA, hbsm_handle B, int tB, int symm_square, int updated, double eps,
                             hbsm_spamm_tol_info* info);

/* ---- accumulating product (engine extra; BLAS form: the reference's multiply / spamm need an empty C) ----
 * C <- alpha * op(A) * op(B) + beta * C: multiply (spamm = 0) or SpAMM with tau (as hbsm_spamm, `updated` included), in one
 * call, without a stored product or temporaries the size of C.  P below is what hbsm_multiply / hbsm_spamm would compute.
 * - C may be the same handle as A, as B, or as both (X <- 2X - X*X is one call): only the old contents of every operand are
 *   read, and C's new table is installed after the leaf GEMMs.
 * - C may be unsized: it is then a zero matrix of the product's shape and gets sized.  A sized C must have op(A)'s row
 *   count, op(B)'s column count, A's dtype and leaf size.
 * - Values, bit for bit, are those of add(rescale(P, alpha), rescale(C, beta)): tiles of P and of C, fl(fl(alpha p) +
 *   fl(beta c)) where both have the tile, fl(alpha p) or fl(beta c) where one has it.  beta == 0 never reads C (NaN or Inf
 *   there does not propagate) and the result is rescale(P, alpha), P's tiles only.  In fp32 alpha and beta are rounded to
 *   float first, as hbsm_rescale does.  A single-leaf product whose one leaf product SpAMM skips is P's zero leaf, as
 *   hbsm_spamm leaves it: fl(fl(alpha 0) + fl(beta c)), signs of zeros and non-finite alpha included.
 * - *n_block_multiplies = the leaf products executed, *n_resizes = C's tile count after the call.  C's n_mults is the
 *   executed count, plus C's previous n_mults when beta != 0 (as hbsm_add adds them).  Cached leaf norms are stale and
 *   the cached root norm is 0, as after a product.  The task hooks (hbsm_export_tasks, hbsm_task_checksum, hbsm_export_tile_tasks) report this call's products (none for a tile that
 *   came only from the old C), hbsm_stage_times_last is filled in (gemm_ms includes the scaling of the old-only tiles).
 *   A committed halo of B takes part as in hbsm_multiply; a halo on C is dropped.
 * - Deterministic (bitwise repeatable).  HBSM_E_ARG before any device work: the operand errors of hbsm_multiply /
 *   hbsm_spamm (same codes and messages; only "C must be empty" is dropped), a sized C of the wrong shape, dtype or leaf
 *   size, and a product already in flight on this thread (hbsm_product_begin). */
int hbsm_multiply_accumulate(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, double alpha, double beta,
                             int spamm, double tau, int updated, size_t* n_block_multiplies, size_t* n_resizes);

/* ---- parity / bench hooks ---- */
/* executed products of the call that produced C, sorted by (Morton key of (ci,cj), k); cap=0 -> count */
int hbsm_export_tasks(hbsm_handle C, size_t cap, int64_t* ci, int64_t* cj, int64_t* k, size_t* n);
/* order-independent checksum of that executed-product set: sum over products of splitmix64(ci<<42 | cj<<21 | k) mod 2^64
 * (the per-rank checksums of a sharded product add up to the single-GPU value) */
int hbsm_task_checksum(hbsm_handle C, uint64_t* out);
/* the k's (ascending) of the products accumulated into C tile (bi, bj); *found = 0 if C has no such tile; cap too small ->
 * only *n is set */
int hbsm_export_tile_tasks(hbsm_handle C, int bi, int bj, size_t cap, int64_t* k, size_t* n, int* found);
/* leaves in ascending Morton order; norms/tiles may be NULL; cap=0 -> count */
int hbsm_export_leaves(hbsm_handle h, size_t cap, int64_t* bi, int64_t* bj, void* norms_cached, void* tiles, size_t* n);
int hbsm_stage_times_last(hbsm_stage_times* out);
int hbsm_set_gemm_variant(int variant);    /* 0 = auto (TMA-tiled DMMA / grouped tcgen05), 1 = generic FMA kernel (debug/parity),
                                            * 3 = fp32: single-C-tile tcgen05 kernels instead of the 2x2-group ones (parity);
                                            * any other value: HBSM_E_ARG */

/* ---- device-side interface (multi-GPU plumbing, device-resident benchmarks) ---- */
/* borrowed pointers into the matrix's device block table: valid until the matrix is modified */
int hbsm_device_table(hbsm_handle h, size_t* n_tiles, const uint64_t** d_morton_keys, const void** d_norms,
                      const void** d_tiles);
/* build a matrix from device arrays (keys need not be sorted; tiles column-major, b*b each); copies */
int hbsm_assign_device_tiles(hbsm_handle h, size_t n_tiles, const uint64_t* d_morton_keys, const void* d_tiles,
                             const void* d_norms_or_null);
/* Halo tail of an op(B) operand (multi-GPU, SURVEY 8e): make room for `capacity` more tiles behind the matrix's own
 * ones and return device pointers to the tail of its key / leaf-norm / tile arrays, so that tiles owned by peer ranks
 * can be received in place (NCCL writes straight into the tail).  hbsm_halo_commit(h, n) makes the first n tail tiles
 * part of the NEXT products in which h is the right operand (they never enter h's own block table: readback, add,
 * norms of h are unaffected); n = 0 drops them.  Any modification of h drops the halo.
 * (The library's own multi-GPU product, hbsm_sharded_product below, uses exactly this; the entry points stay public for
 * callers that bring their own transport.) */
int hbsm_halo_reserve(hbsm_handle h, size_t capacity, uint64_t** d_keys, void** d_norms, void** d_tiles);
int hbsm_halo_commit(hbsm_handle h, size_t n_halo);
/* banded decay generator a_ij = (0.5+0.5u(seed,i,j)) * table[|i-j|], |i-j| <= W (table has W+1 entries, e.g.
 * exp(-lambda d)), built on device; u = splitmix64 hash -> [0,1); symmetric != 0 uses u(seed,min,max).
 * Tile rows [row_tile_lo,row_tile_hi) only (shard); full matrix with 0,-1. */
int hbsm_generate_decay(hbsm_handle h, int n, const double* table, int W, uint64_t seed, int symmetric,
                        int row_tile_lo, int row_tile_hi);
uint64_t hbsm_morton_encode(uint32_t bi, uint32_t bj);
void hbsm_morton_decode(uint64_t key, uint32_t* bi, uint32_t* bj);
void* hbsm_stream(void);                  /* cudaStream_t of the engine */

/* ---- multi-GPU: one process per GPU, C sharded by block rows (SURVEY 8e) --------------------------------------------
 * The reference has no distributed layer; its static multiply/spamm (H:255-305) see one address space.  Here rank r holds, of
 * every operand, the tiles whose block ROW (C row for op(A), contraction index k for op(B), after the transposition flags)
 * lies in its slab, in matrices that carry the full logical dimensions, and gets the same slab of C.  NCCL is loaded at run
 * time (libnccl.so.2; hbsm_comm_set_library or $HBSM_NCCL_LIB override the search), so single-GPU hosts need none.
 * Every call below except set_library / unique_id / info is COLLECTIVE: all ranks call it, in the same order. */
#define HBSM_COMM_ID_BYTES 128
int hbsm_comm_set_library(const char* path);
/* rank 0 creates the id and hands its 128 bytes to the other ranks by any means (MPI, a file, torch's store ...) */
int hbsm_comm_unique_id(void* id_out);
int hbsm_comm_init(const void* id, int rank, int world);    /* after hbsm_init(device); world <= 64 */
int hbsm_comm_finalize(void);
int hbsm_comm_info(int* rank, int* world, int* nccl_version);
int hbsm_comm_barrier(void);
int hbsm_comm_allreduce_f64(double* vals, int n, int take_max);         /* host scalars: sum (or max) over the ranks */
int hbsm_comm_allgather_u64(const uint64_t* mine, size_t n, uint64_t* all);   /* all has n * world entries */
/* equal slabs of block rows: rank r owns [lo, hi); for world in {2,4,8} these are the top-level quadtree block rows */
int hbsm_shard_rows(int grid_side, int world, int rank, int* lo, int* hi);
/* balanced slabs: bounds[world + 1] chosen on the prefix sums of per-block-row weights (e.g. leaf products per C block row) so
 * that every slab carries about the same weight (the band of a decay matrix is clipped at the matrix edge: equal slabs leave
 * the edge ranks ~7 % lighter) */
int hbsm_shard_rows_balanced(const uint64_t* row_weights, int grid_side, int world, int* bounds);
/* the distributed half of update_internal_info() (H:3905): all-gathers this matrix' (Morton key, leaf norm^2) table.  Call it
 * after the norms are refreshed on a matrix that will be the RIGHT operand of sharded products; valid until h changes. */
int hbsm_publish(hbsm_handle h);
/* C_r = this rank's block rows of op(A)*op(B).  A, B: this rank's slabs with refreshed norms, B published.  Remote op(B)
 * tiles that at least one executed product of this rank touches are received straight behind B's own tiles (NCCL send/recv
 * over NVLink) while the leaf GEMMs of the C tiles that need none of them already run; there is no reduction.  upper_only:
 * plan only C tiles with ci <= cj and mask the diagonal tiles (sharded symm_square / symm_rk on a full-storage symmetric
 * operand, H:3563 / H:3711).  n_block_multiplies / n_resizes are this rank's (sum them with hbsm_comm_allreduce_f64). */
int hbsm_sharded_product(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, int spamm, double tau, int upper_only,
                         size_t* n_block_multiplies, size_t* n_resizes);
/* leaf products per C block row of op(A)*op(B) summed over the ranks (count pass only; B published): weights[grid_side], the
 * input of hbsm_shard_rows_balanced.  grid_side = block-grid side of the product (max of the operands'). */
int hbsm_sharded_row_weights(hbsm_handle A, int tA, hbsm_handle B, int tB, int spamm, double tau, int upper_only, int grid_side,
                             uint64_t* weights);
typedef struct hbsm_shard_stats {
    double plan_ms;       /* thresholds + all-gather + flags + scan + count read-back + halo keys/norms (engine stream) */
    double exchange_ms;   /* pack + grouped ncclSend/ncclRecv of the tiles (comm stream; overlaps the task list and first GEMM) */
    double publish_ms;    /* last hbsm_publish */
    uint64_t sent_tiles, recv_tiles;
} hbsm_shard_stats;
int hbsm_shard_stats_last(hbsm_shard_stats* out);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* HBSM_B200_H */

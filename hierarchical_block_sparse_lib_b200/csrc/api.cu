// api.cu -- the C ABI of include/hbsm_b200.h over the flat engine.  Every entry point catches engine exceptions and
// returns a status code; the message (the reference's own std::runtime_error text where one exists) is kept per thread.
#include "matrix.cuh"

using namespace hbsm_b200;

struct hbsm_matrix_s {
    Matrix m;
};

namespace {
thread_local std::string g_last_error;

template <typename F>
int guarded(F&& f) {
    try {
        f();
        return HBSM_OK;
    } catch (const Error& e) {
        g_last_error = e.what();
        return e.code;
    } catch (const std::exception& e) {
        g_last_error = e.what();
        return HBSM_E_RUNTIME;
    } catch (...) {
        g_last_error = "hbsm_b200: unknown exception";
        return HBSM_E_RUNTIME;
    }
}

Matrix& M(hbsm_handle h) {
    if (!h) throw Error(HBSM_E_ARG, "hbsm_b200: null matrix handle");
    Matrix& m = h->m;
    if (m.pending_ev) {   // device work queued by another call (possibly another thread's stream) has to land first
        if (engine().ready) cudaStreamWaitEvent(engine().stream, m.pending_ev, 0);
        else cudaEventSynchronize(m.pending_ev);
        cudaEventDestroy(m.pending_ev);
        m.pending_ev = nullptr;
    }
    return m;
}

void store_real(const Matrix& m, void* out, double v) {
    if (m.dtype == HBSM_F64) *(double*)out = v;
    else *(float*)out = (float)v;
}
}  // namespace

extern "C" {

int hbsm_init(int device) {
    return guarded([&] {
        int expect = -1;   // one device per process (one process per GPU); every thread's engine binds to it
        if (!shared().device.compare_exchange_strong(expect, device) && expect != device)
            throw Error(HBSM_E_ARG, "hbsm_b200: engine already bound to another device");
        ensure_engine();
    });
}

int hbsm_finalize(void) {
    return guarded([&] {
        Engine& e = engine();
        if (!e.ready) return;
        HB_CUDA(cudaStreamSynchronize(e.stream));
        e.cache.drop_all();   // large blocks kept for exact-size reuse go back to the driver
    });
}

const char* hbsm_last_error(void) { return g_last_error.c_str(); }

int hbsm_device_info(char* name, size_t cap, int* sm_count, int* cc_major, int* cc_minor) {
    return guarded([&] {
        ensure_engine();
        Engine& e = engine();
        if (name && cap) { strncpy(name, e.name.c_str(), cap - 1); name[cap - 1] = 0; }
        if (sm_count) *sm_count = e.sm_count;
        if (cc_major) *cc_major = e.cc_major;
        if (cc_minor) *cc_minor = e.cc_minor;
    });
}

uint64_t hbsm_kernel_launch_count(void) { return shared().launches.load(); }

int hbsm_create(int dtype, hbsm_handle* out) {
    return guarded([&] {
        if (!out || (dtype != HBSM_F64 && dtype != HBSM_F32)) throw Error(HBSM_E_ARG, "hbsm_b200: bad dtype");
        hbsm_matrix_s* h = new hbsm_matrix_s();
        h->m.dtype = dtype;
        *out = h;
    });
}

int hbsm_destroy(hbsm_handle h) {
    return guarded([&] { delete h; });
}

int hbsm_set_blocksize(hbsm_handle h, int blocksize) {
    return guarded([&] {
        if (!M(h).empty())   // H:450
            throw_ref("Error in HierarchicalBlockSparseMatrix<Treal>::set_params: Matrix must be empty when setting params.");
        M(h).b = blocksize;
    });
}
int hbsm_get_blocksize(hbsm_handle h, int* blocksize) {
    return guarded([&] { *blocksize = M(h).b; });
}
int hbsm_resize(hbsm_handle h, int n_rows, int n_cols) {
    return guarded([&] { ensure_engine(); M(h).resize(n_rows, n_cols); });
}
int hbsm_clear(hbsm_handle h) {
    return guarded([&] { M(h).clear(); });
}
int hbsm_is_empty(hbsm_handle h, int* out) {
    return guarded([&] { *out = M(h).empty() ? 1 : 0; });
}
int hbsm_children_exist(hbsm_handle h, int* out) {
    return guarded([&] { *out = (M(h).sized && M(h).vdepth() > 0 && M(h).L > 0) ? 1 : 0; });
}
int hbsm_dims(hbsm_handle h, int* n_rows, int* n_cols) {
    return guarded([&] { if (n_rows) *n_rows = M(h).M; if (n_cols) *n_cols = M(h).N; });
}
int hbsm_depth(hbsm_handle h, int* out) {   // H:496: deepest existing leaf
    return guarded([&] { *out = (M(h).sized && M(h).L > 0) ? M(h).vdepth() : 0; });
}
int hbsm_expected_depth(hbsm_handle h, int* out) {
    return guarded([&] { *out = M(h).vdepth(); });
}
int hbsm_is_consistent(hbsm_handle h, int* out) {   // H:1809: a sized, childless non-leaf is inconsistent
    return guarded([&] { *out = (M(h).sized && M(h).L > 0) ? 1 : 0; });
}
int hbsm_dtype(hbsm_handle h, int* out) {
    return guarded([&] { *out = M(h).dtype; });
}

int hbsm_assign_coo(hbsm_handle h, size_t n, const int* rows, const int* cols, const void* vals, int use_max,
                    int boundaries_checked) {
    return guarded([&] { assign_coo(M(h), n, rows, cols, vals, use_max != 0, boundaries_checked != 0); });
}
int hbsm_assign_tiles(hbsm_handle h, size_t n_tiles, const int* bi, const int* bj, const void* tiles) {
    return guarded([&] { assign_tiles_host(M(h), n_tiles, bi, bj, tiles); });
}
int hbsm_get_values(hbsm_handle h, size_t n, const int* rows, const int* cols, void* out) {
    return guarded([&] { get_values(M(h), n, rows, cols, out); });
}
int hbsm_get_all_values(hbsm_handle h, size_t cap, int* rows, int* cols, void* vals, size_t* n) {
    return guarded([&] { *n = get_all_values(M(h), cap, rows, cols, vals); });
}
int hbsm_export_tile(hbsm_handle h, int bi, int bj, void* host_tile, int* found) {
    return guarded([&] {
        if (bi < 0 || bj < 0) throw Error(HBSM_E_ARG, "hbsm_b200: export_tile: negative block coordinate");
        *found = export_tile(M(h), (uint32_t)bi, (uint32_t)bj, host_tile) ? 1 : 0;
    });
}
int hbsm_nnz(hbsm_handle h, size_t* out) {
    return guarded([&] { *out = count_nnz(M(h)); });
}
int hbsm_n_blocks(hbsm_handle h, size_t* out) {
    return guarded([&] { *out = M(h).L; });
}
int hbsm_get_n_block_multiplications(hbsm_handle h, size_t* out) {
    return guarded([&] { *out = M(h).n_mults; });
}
int hbsm_set_n_block_multiplications(hbsm_handle h, size_t n) {
    return guarded([&] { M(h).n_mults = n; });
}

int hbsm_update_norms(hbsm_handle h) {
    return guarded([&] { update_norms(M(h)); sync_stream(); });
}
int hbsm_frob_squared(hbsm_handle h, void* out) {
    return guarded([&] { store_real(M(h), out, frob_squared(M(h))); });
}
int hbsm_frob_squared_cached(hbsm_handle h, void* out) {
    return guarded([&] { store_real(M(h), out, M(h).root_norm_cached); });
}

int hbsm_multiply(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, size_t* n_block_multiplies,
                  size_t* n_resizes) {
    return guarded([&] {
        ProductOpts o;
        op_product(M(A), tA != 0, M(B), tB != 0, M(C), o, n_block_multiplies, n_resizes);
    });
}
int hbsm_spamm(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, double tau, int updated,
               size_t* n_block_multiplies, size_t* n_resizes) {
    return guarded([&] {
        ProductOpts o;
        o.spamm = true;
        o.tau = tau;
        o.updated = updated != 0;
        op_product(M(A), tA != 0, M(B), tB != 0, M(C), o, n_block_multiplies, n_resizes);
    });
}
int hbsm_multiply_accumulate(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, double alpha, double beta,
                             int spamm, double tau, int updated, size_t* n_block_multiplies, size_t* n_resizes) {
    return guarded([&] {
        ProductOpts o;
        o.spamm = spamm != 0;
        o.tau = tau;
        o.updated = updated != 0;
        o.c_old = &M(C);
        o.alpha = alpha;
        o.beta = beta;
        op_product(M(A), tA != 0, M(B), tB != 0, M(C), o, n_block_multiplies, n_resizes);
    });
}
int hbsm_product_begin_ex(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, int spamm, double tau, int updated,
                          int defer_halo_tiles, int upper_only) {
    return guarded([&] {
        ProductOpts o;
        o.spamm = spamm != 0;
        o.tau = tau;
        o.updated = updated != 0;
        o.upper_only = upper_only != 0;   // symm_square / symm_rk: only C tiles with ci <= cj; finish masks the diagonal tiles
        // defer_halo_tiles: 1 = launch the own-only C tiles now; 2 = plan only, hbsm_product_finish launches them too (so that a
        // transfer queued in between gets its SMs before the persistent leaf GEMM occupies all of them)
        op_product_begin(M(A), tA != 0, M(B), tB != 0, M(C), o, defer_halo_tiles != 0, defer_halo_tiles != 2, defer_halo_tiles == 2);
    });
}
int hbsm_product_begin(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, int spamm, double tau, int updated,
                       int defer_halo_tiles) {
    return hbsm_product_begin_ex(A, tA, B, tB, C, spamm, tau, updated, defer_halo_tiles, 0);
}
int hbsm_product_finish(hbsm_handle C, void* cuda_event_or_null, size_t* n_block_multiplies, size_t* n_resizes) {
    const int rc = guarded([&] { op_product_finish(M(C), (cudaEvent_t)cuda_event_or_null, n_block_multiplies, n_resizes); });
    if (rc != HBSM_OK) op_product_abort();
    return rc;
}
int hbsm_product_abort(void) {
    return guarded([&] { op_product_abort(); });
}
int hbsm_product_to_host(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, int spamm, double tau, int updated,
                         void* host_tiles, size_t cap_tiles, size_t* n_block_multiplies, size_t* n_resizes) {
    return guarded([&] {
        ProductOpts o;
        o.spamm = spamm != 0;
        o.tau = tau;
        o.updated = updated != 0;
        try {
            op_product_to_host(M(A), tA != 0, M(B), tB != 0, M(C), o, host_tiles, cap_tiles, 8, n_block_multiplies, n_resizes);
        } catch (...) {
            op_product_abort();
            throw;
        }
    });
}
int hbsm_product_from_host(hbsm_handle A, size_t n_a, const int* a_bi, const int* a_bj, const void* a_tiles, int tA,
                           hbsm_handle B, size_t n_b, const int* b_bi, const int* b_bj, const void* b_tiles, int tB,
                           hbsm_handle C, int spamm, double tau, int n_slabs, void* host_c_tiles, size_t cap_tiles,
                           int* c_bi, int* c_bj, size_t* n_block_multiplies, size_t* n_resizes) {
    return guarded([&] {
        ProductOpts o;
        o.spamm = spamm != 0;
        o.tau = tau;
        HostTiles ha{n_a, a_bi, a_bj, a_tiles}, hb{n_b, b_bi, b_bj, b_tiles};
        try {
            op_product_from_host(M(A), ha, tA != 0, M(B), hb, tB != 0, M(C), o, n_slabs, host_c_tiles, cap_tiles, c_bi, c_bj,
                                 n_block_multiplies, n_resizes);
        } catch (...) {
            op_product_abort();
            throw;
        }
    });
}
int hbsm_worth_to_multiply(hbsm_handle A, int tA, hbsm_handle B, int tB, int* out) {
    return guarded([&] { *out = worth_product(M(A), tA != 0, M(B), tB != 0, false, 0.0) ? 1 : 0; });
}
int hbsm_worth_to_spamm(hbsm_handle A, int tA, hbsm_handle B, int tB, double tau, int* out) {
    return guarded([&] { *out = worth_product(M(A), tA != 0, M(B), tB != 0, true, tau) ? 1 : 0; });
}

int hbsm_add(hbsm_handle A, hbsm_handle B, hbsm_handle C) {
    return guarded([&] {
        if (C == A || C == B) throw Error(HBSM_E_ARG, "hbsm_b200: add: C must not alias an operand");
        op_add(M(A), M(B), M(C));
    });
}
int hbsm_transpose(hbsm_handle A, hbsm_handle C) {
    return guarded([&] { op_transpose(M(A), M(C)); });
}
int hbsm_upper_triangle(hbsm_handle A, hbsm_handle C) {
    return guarded([&] {
        if (C == A) throw Error(HBSM_E_ARG, "hbsm_b200: get_upper_triangle: target must not alias the source");
        op_upper(M(A), M(C));
    });
}
int hbsm_rescale(hbsm_handle C, hbsm_handle A, double alpha) {
    return guarded([&] { op_rescale(M(C), M(A), alpha); });
}
int hbsm_copy(hbsm_handle C, hbsm_handle A) {
    return guarded([&] { op_copy(M(C), M(A)); });
}

int hbsm_frob_block_trunc(hbsm_handle A, hbsm_handle C, double trunc_value, int* removed) {
    return guarded([&] {
        const bool r = op_trunc(M(A), M(C), trunc_value);
        if (removed) *removed = r ? 1 : 0;
    });
}
int hbsm_leaf_norms(hbsm_handle h, size_t cap, void* out, size_t* n) {
    return guarded([&] {
        Matrix& A = M(h);
        *n = A.L;
        if (cap < A.L || A.L == 0) return;
        DevBuf<char> fresh(A.L * A.esize());
        compute_leaf_norms(A, fresh.p);
        HB_CUDA(cudaMemcpyAsync(out, fresh.p, A.L * A.esize(), cudaMemcpyDeviceToHost, engine().stream));
        sync_stream();
    });
}
int hbsm_serialized_size(hbsm_handle h, size_t* out) {
    return guarded([&] { *out = serialized_size(M(h)); });
}
int hbsm_serialize(hbsm_handle h, char* buffer, size_t capacity) {
    return guarded([&] { serialize(M(h), buffer, capacity); });
}
int hbsm_deserialize(hbsm_handle h, const char* buffer, size_t size) {
    return guarded([&] { deserialize(M(h), buffer, size); });
}
int hbsm_count_skips(hbsm_handle A, int tA, hbsm_handle B, int tB, size_t n, const double* taus, int apply_truncation, int apply_spamm,
                     unsigned long* out) {
    return guarded([&] { count_skips(M(A), tA != 0, M(B), tB != 0, n, taus, apply_truncation != 0, apply_spamm != 0, out); });
}
int hbsm_spamm_errors(hbsm_handle A, int tA, hbsm_handle B, int tB, size_t n, const double* taus, double* out, size_t* n_out) {
    return guarded([&] { *n_out = spamm_errors(M(A), tA != 0, M(B), tB != 0, n, taus, out); });
}
int hbsm_extract_quadrant(hbsm_handle A, int q, hbsm_handle C, int* exists) {
    return guarded([&] {
        const bool e = op_extract_quadrant(M(A), q, M(C));
        if (exists) *exists = e ? 1 : 0;
    });
}
int hbsm_assemble_quadrants(hbsm_handle C, int n_rows, int n_cols, hbsm_handle q0, hbsm_handle q1, hbsm_handle q2, hbsm_handle q3) {
    return guarded([&] {
        const Matrix* quads[4] = {q0 ? &q0->m : nullptr, q1 ? &q1->m : nullptr, q2 ? &q2->m : nullptr, q3 ? &q3->m : nullptr};
        op_assemble_quadrants(M(C), n_rows, n_cols, quads);
    });
}
int hbsm_symm_multiply(hbsm_handle A, int sA, hbsm_handle B, int sB, hbsm_handle C) {
    return guarded([&] {
        if (!sA && !sB)   // H:3264
            throw_ref("Error in hbsm::symm_multiply, Neither A nor B are symmetric, one and only one of them should be symmetric.");
        if (sA && sB)     // H:3266
            throw_ref("Error in hbsm::symm_multiply, Both A and B are symmetric, one and only one of them should be symmetric.");
        if (!M(C).empty()) throw_ref("Error in HierarchicalBlockSparseMatrix::symm_multiply(): non-empty matrix to write result!");
        if (M(A).N != M(B).M) throw_ref("Error in HierarchicalBlockSparseMatrix::symm_multiply(): matrices have bad sizes!");
        Matrix S;
        ProductOpts o;
        if (sA) { sym_expand(M(A), S); op_product(S, false, M(B), false, M(C), o, nullptr, nullptr); }
        else    { sym_expand(M(B), S); op_product(M(A), false, S, false, M(C), o, nullptr, nullptr); }
    });
}
int hbsm_symm_square(hbsm_handle A, hbsm_handle C) {
    return guarded([&] {
        if (!M(C).empty()) throw_ref("Error in HierarchicalBlockSparseMatrix::symm_square(): non-empty matrix to write result!");
        if (M(A).N != M(A).M) throw_ref("Error in HierarchicalBlockSparseMatrix::symm_square(): matrix has bad sizes!");
        Matrix S;
        sym_expand(M(A), S);
        ProductOpts o;
        o.upper_only = true;
        op_product(S, false, S, false, M(C), o, nullptr, nullptr);
        sync_stream();
    });
}
int hbsm_symm_rk(hbsm_handle A, int transposed, hbsm_handle C) {
    return guarded([&] {
        if (!M(C).empty()) throw_ref("Error in HierarchicalBlockSparseMatrix::symm_rk(): non-empty matrix to write result!");
        ProductOpts o;
        o.upper_only = true;
        if (transposed) op_product(M(A), true, M(A), false, M(C), o, nullptr, nullptr);
        else op_product(M(A), false, M(A), true, M(C), o, nullptr, nullptr);
        sync_stream();
    });
}
int hbsm_symm_square_spamm(hbsm_handle A, hbsm_handle C, double tau, size_t* n_block_multiplies, size_t* n_resizes) {
    return guarded([&] {
        if (!M(C).empty()) throw_ref("Error in HierarchicalBlockSparseMatrix::symm_square(): non-empty matrix to write result!");
        if (M(A).N != M(A).M) throw_ref("Error in HierarchicalBlockSparseMatrix::symm_square(): matrix has bad sizes!");
        Matrix S;
        sym_expand(M(A), S);
        update_norms(S);
        ProductOpts o;
        o.spamm = true;
        o.tau = tau;
        o.upper_only = true;
        op_product(S, false, S, false, M(C), o, n_block_multiplies, n_resizes);
        sync_stream();
    });
}

int hbsm_multiply_dense(hbsm_handle A, int op, int m, const void* X, int ldx, void* Y, int ldy, double alpha, double beta) {
    return guarded([&] { dense_product_host(M(A), op, m, X, ldx, Y, ldy, alpha, beta); });
}
int hbsm_multiply_dense_device(hbsm_handle A, int op, int m, const void* d_X, int ldx, void* d_Y, int ldy, double alpha,
                               double beta, void* cuda_stream) {
    return guarded([&] {
        Matrix& a = M(A);
        validate_dense(a, op, m, ldx, ldy, d_X, d_Y);   // before either stream is touched
        if (m == 0) return;
        ensure_engine();
        // the caller's stream -> engine stream -> the caller's stream, by events: no host synchronisation
        static thread_local cudaEvent_t ev_in = nullptr, ev_out = nullptr;
        if (!ev_in) HB_CUDA(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
        if (!ev_out) HB_CUDA(cudaEventCreateWithFlags(&ev_out, cudaEventDisableTiming));
        const cudaStream_t s = (cudaStream_t)cuda_stream;
        HB_CUDA(cudaEventRecord(ev_in, s));
        HB_CUDA(cudaStreamWaitEvent(engine().stream, ev_in, 0));
        dense_product_device(a, op, m, d_X, ldx, d_Y, ldy, alpha, beta);
        HB_CUDA(cudaEventRecord(ev_out, engine().stream));
        HB_CUDA(cudaStreamWaitEvent(s, ev_out, 0));
    });
}
int hbsm_spectral_norm(hbsm_handle A, int symmetric_upper, int max_iter, double rel_tol, double* norm, double* lambda_min,
                       double* lambda_max, int* n_iter) {
    return guarded([&] {
        const SpectralResult r = spectral_norm(M(A), symmetric_upper != 0, max_iter, rel_tol);
        if (norm) *norm = r.norm;
        if (lambda_min) *lambda_min = r.lambda_min;
        if (lambda_max) *lambda_max = r.lambda_max;
        if (n_iter) *n_iter = r.n_iter;
    });
}

int hbsm_spectral_block_trunc(hbsm_handle A, int symmetric_upper, double eps, int max_iter, hbsm_handle C, hbsm_trunc_info* info) {
    return guarded([&] {
        if (C == A) throw Error(HBSM_E_ARG, "hbsm_b200: spectral_block_trunc: target must not alias the source");
        const TruncInfo t = spectral_block_trunc(M(A), symmetric_upper != 0, eps, max_iter, M(C));
        if (info) {
            info->n_dropped = t.n_dropped;
            info->drop_nsq = t.drop_nsq;
            info->n_frob = t.n_frob;
            info->err_bound = t.err_bound;
            info->certified_by_lanczos = t.certified_by_lanczos ? 1 : 0;
            info->n_decisions = t.n_decisions;
            info->lanczos_steps = t.lanczos_steps;
        }
    });
}
int hbsm_truncation_spectral_errors(hbsm_handle A, int symmetric_upper, size_t n, const double* taus, int max_iter, double rel_tol,
                                    double* out_norms, int* out_iters) {
    return guarded([&] { truncation_spectral_errors(M(A), symmetric_upper != 0, n, taus, max_iter, rel_tol, out_norms, out_iters); });
}

int hbsm_spamm_error_bounds(hbsm_handle A, int tA, hbsm_handle B, int tB, int symm_square, int updated, size_t n, const double* taus,
                            double* bounds, size_t* n_skipped) {
    return guarded([&] { spamm_error_bounds(M(A), tA != 0, M(B), tB != 0, symm_square != 0, updated != 0, n, taus, bounds, n_skipped); });
}
int hbsm_spamm_tau_for_error(hbsm_handle A, int tA, hbsm_handle B, int tB, int symm_square, int updated, double eps,
                             hbsm_spamm_tol_info* info) {
    return guarded([&] {
        const SpammTol t = spamm_tau_for_error(M(A), tA != 0, M(B), tB != 0, symm_square != 0, updated != 0, eps);
        if (info) {
            info->tau = t.tau;
            info->bound = t.bound;
            info->level = t.level;
            info->n_candidates = t.n_candidates;
            info->n_skipped = t.n_skipped;
            info->n_levels = t.n_levels;
        }
    });
}

int hbsm_export_tasks(hbsm_handle Ch, size_t cap, int64_t* ci, int64_t* cj, int64_t* k, size_t* n) {
    return guarded([&] {
        Matrix& C = M(Ch);
        *n = C.n_tasks;
        if (cap < C.n_tasks || C.n_tasks == 0) return;
        std::vector<uint64_t> keys = C.keys.to_host();
        std::vector<uint64_t> begin = C.task_begin.to_host();
        std::vector<uint32_t> tk = C.task_k.to_host();
        for (size_t t = 0; t < C.L; ++t)
            for (uint64_t p = begin[t]; p < begin[t + 1]; ++p) {
                ci[p] = morton_row(keys[t]);
                cj[p] = morton_col(keys[t]);
                k[p] = tk[p];
            }
    });
}

int hbsm_task_checksum(hbsm_handle Ch, uint64_t* out) {
    return guarded([&] { *out = task_checksum(M(Ch)); });
}
int hbsm_export_tile_tasks(hbsm_handle Ch, int bi, int bj, size_t cap, int64_t* k, size_t* n, int* found) {
    return guarded([&] {
        if (bi < 0 || bj < 0) throw Error(HBSM_E_ARG, "hbsm_b200: export_tile_tasks: negative block coordinate");
        const long long r = tile_tasks(M(Ch), (uint32_t)bi, (uint32_t)bj, cap, k);
        *found = r >= 0 ? 1 : 0;
        *n = r >= 0 ? (size_t)r : 0;
    });
}

int hbsm_export_leaves(hbsm_handle h, size_t cap, int64_t* bi, int64_t* bj, void* norms_cached, void* tiles, size_t* n) {
    return guarded([&] {
        Matrix& A = M(h);
        *n = A.L;
        if (cap < A.L || A.L == 0) return;
        if (bi || bj) {
            std::vector<uint64_t> keys = A.keys.to_host();
            for (size_t t = 0; t < A.L; ++t) {
                if (bi) bi[t] = morton_row(keys[t]);
                if (bj) bj[t] = morton_col(keys[t]);
            }
        }
        if (norms_cached) HB_CUDA(cudaMemcpyAsync(norms_cached, A.norms.p, A.L * A.esize(), cudaMemcpyDeviceToHost, engine().stream));
        if (tiles) HB_CUDA(cudaMemcpyAsync(tiles, A.tiles.p, A.L * A.tile_bytes(), cudaMemcpyDeviceToHost, engine().stream));
        sync_stream();
    });
}

int hbsm_stage_times_last(hbsm_stage_times* out) {
    return guarded([&] { *out = engine().last; });
}
int hbsm_set_gemm_variant(int variant) {
    return guarded([&] {
        if (variant != 0 && variant != 1 && variant != 3)
            throw Error(HBSM_E_ARG, "hbsm_b200: gemm variant " + std::to_string(variant) + " does not exist (0, 1 or 3)");
        shared().gemm_variant.store(variant);
    });
}

int hbsm_device_table(hbsm_handle h, size_t* n_tiles, const uint64_t** d_morton_keys, const void** d_norms,
                      const void** d_tiles) {
    return guarded([&] {
        Matrix& A = M(h);
        if (n_tiles) *n_tiles = A.L;
        if (d_morton_keys) *d_morton_keys = A.keys.p;
        if (d_norms) *d_norms = A.norms.p;
        if (d_tiles) *d_tiles = A.tiles.p;
    });
}
int hbsm_assign_device_tiles(hbsm_handle h, size_t n_tiles, const uint64_t* d_morton_keys, const void* d_tiles,
                             const void* d_norms_or_null) {
    return guarded([&] {
        // caller's arrays live on another stream: order them before ours
        HB_CUDA(cudaDeviceSynchronize());
        assign_tiles_device(M(h), n_tiles, d_morton_keys, d_tiles, d_norms_or_null);
    });
}
int hbsm_halo_reserve(hbsm_handle h, size_t capacity, uint64_t** d_keys, void** d_norms, void** d_tiles) {
    return guarded([&] { reserve_halo(M(h), capacity, d_keys, d_norms, d_tiles); });
}
int hbsm_halo_commit(hbsm_handle h, size_t n_halo) {
    return guarded([&] {
        HB_CUDA(cudaDeviceSynchronize());   // the tail was filled on the caller's (transport) stream: order it before ours
        commit_halo(M(h), n_halo);
    });
}
int hbsm_generate_decay(hbsm_handle h, int n, const double* table, int W, uint64_t seed, int symmetric, int row_tile_lo,
                        int row_tile_hi) {
    return guarded([&] { generate_decay(M(h), n, table, W, seed, symmetric != 0, row_tile_lo, row_tile_hi); });
}
uint64_t hbsm_morton_encode(uint32_t bi, uint32_t bj) { return morton_encode(bi, bj); }
void hbsm_morton_decode(uint64_t key, uint32_t* bi, uint32_t* bj) {
    if (bi) *bi = morton_row(key);
    if (bj) *bj = morton_col(key);
}
void* hbsm_stream(void) { return (void*)engine().stream; }

int hbsm_leaf_inv_chol(hbsm_handle A, hbsm_handle Z, int zdim, int valid) {
    return guarded([&] { op_leaf_inv_chol(M(A), M(Z), zdim, valid); });
}

// ---- multi-GPU (sharded.cu) ----
int hbsm_comm_set_library(const char* path) { return guarded([&] { comm_set_library(path); }); }
int hbsm_comm_unique_id(void* id_out) {
    return guarded([&] {
        if (!id_out) throw Error(HBSM_E_ARG, "hbsm_b200: comm_unique_id: null buffer");
        comm_unique_id(id_out);
    });
}
int hbsm_comm_init(const void* id, int rank, int world) {
    return guarded([&] {
        if (!id) throw Error(HBSM_E_ARG, "hbsm_b200: comm_init: null id");
        comm_init(id, rank, world);
    });
}
int hbsm_comm_finalize(void) { return guarded([&] { comm_finalize(); }); }
int hbsm_comm_info(int* rank, int* world, int* nccl_version) { return guarded([&] { comm_info(rank, world, nccl_version); }); }
int hbsm_comm_barrier(void) { return guarded([&] { comm_barrier(); }); }
int hbsm_comm_allreduce_f64(double* vals, int n, int take_max) { return guarded([&] { comm_allreduce_f64(vals, n, take_max != 0); }); }
int hbsm_comm_allgather_u64(const uint64_t* mine, size_t n, uint64_t* all) { return guarded([&] { comm_allgather_u64(mine, n, all); }); }
int hbsm_shard_rows(int grid_side, int world, int rank, int* lo, int* hi) {
    return guarded([&] {
        if (grid_side < 1 || world < 1 || rank < 0 || rank >= world || !lo || !hi) throw Error(HBSM_E_ARG, "hbsm_b200: shard_rows: bad arguments");
        *lo = (int)((long long)grid_side * rank / world);
        *hi = (int)((long long)grid_side * (rank + 1) / world);
    });
}
int hbsm_shard_rows_balanced(const uint64_t* w, int grid_side, int world, int* bounds) {
    return guarded([&] {
        if (!w || grid_side < 1 || world < 1 || !bounds) throw Error(HBSM_E_ARG, "hbsm_b200: shard_rows_balanced: bad arguments");
        double total = 0;
        for (int i = 0; i < grid_side; ++i) total += (double)w[i];
        bounds[0] = 0;
        double acc = 0;
        int row = 0;
        for (int r = 1; r < world; ++r) {   // boundary r: first row at which the prefix reaches r/world of the total (nearest side)
            const double want = total * r / world;
            while (row < grid_side && acc + (double)w[row] <= want) acc += (double)w[row++];
            if (row < grid_side && want - acc > acc + (double)w[row] - want) acc += (double)w[row++];
            bounds[r] = std::max(row, bounds[r - 1]);
        }
        bounds[world] = grid_side;
    });
}
int hbsm_publish(hbsm_handle h) { return guarded([&] { publish(M(h)); }); }
int hbsm_sharded_product(hbsm_handle A, int tA, hbsm_handle B, int tB, hbsm_handle C, int spamm, double tau, int upper_only,
                         size_t* n_block_multiplies, size_t* n_resizes) {
    return guarded([&] {
        ProductOpts o;
        o.spamm = spamm != 0; o.tau = tau; o.updated = true; o.upper_only = upper_only != 0;
        sharded_product(M(A), tA != 0, M(B), tB != 0, M(C), o, n_block_multiplies, n_resizes);
    });
}
int hbsm_sharded_row_weights(hbsm_handle A, int tA, hbsm_handle B, int tB, int spamm, double tau, int upper_only, int grid_side,
                             uint64_t* weights) {
    return guarded([&] {
        if (!weights) throw Error(HBSM_E_ARG, "hbsm_b200: row weights: null output");
        ProductOpts o;
        o.spamm = spamm != 0; o.tau = tau; o.updated = true; o.upper_only = upper_only != 0;
        sharded_row_weights(M(A), tA != 0, M(B), tB != 0, o, grid_side, weights);
    });
}
int hbsm_shard_stats_last(hbsm_shard_stats* out) {
    return guarded([&] {
        if (!out) throw Error(HBSM_E_ARG, "hbsm_b200: shard_stats_last: null");
        *out = shard_stats_last();
    });
}

}  // extern "C"

/* HierarchicalBlockSparseMatrix.h -- drop-in host class for the hot path of toxaart/hierarchical_block_sparse_lib.
 *
 * Same namespace, class name, public method names, argument order and exception behaviour as the public section of
 * the reference's header-only template (reference source/HierarchicalBlockSparseMatrix.h:166-428, cited H:<line>),
 * but the object is a thin owner of an opaque handle of the B200 engine: every method forwards to the C ABI in
 * include/hbsm_b200.h (libhbsm_b200.so, hand-written sm_100a CUDA).  There is no host fallback -- when no B200 is
 * usable every call that touches data throws std::runtime_error("hbsm_b200: no CUDA device ...").
 *
 * Differences a caller can observe (all documented in INTEGRATION.md):
 *   - Treal must be double or float (the reference's BLAS shim offers exactly these, gblas.h:85-143);
 *   - copy construction / assignment is a deep copy (the reference's implicit copy shares children by shared_ptr);
 *   - spamm(..., updated=false) tests against freshly computed leaf norms and leaves the operands' cached norms
 *     untouched, which is what the reference intends (it refreshes COPIES of A and B, H:3990-4005) but cannot deliver
 *     in its batched build (use-after-free, H:6294-6307);
 *   - the dead recursive multiply (compiled out by the reference's own flags) and adjust_sizes throw
 *     "not provided by hbsm_b200"; the a-priori estimators, inv_chol, serialisation, truncation and the small
 *     utilities are implemented.
 */
#ifndef HBSM_B200_HIERARCHICAL_BLOCK_SPARSE_MATRIX_H
#define HBSM_B200_HIERARCHICAL_BLOCK_SPARSE_MATRIX_H

#include <cmath>
#include <cstddef>
#include <cstdint>
#include <iostream>
#include <stdexcept>
#include <string>
#include <vector>

#include "../hbsm_b200.h"

namespace hbsm {

namespace detail {
template <class T> struct dtype_of;
template <> struct dtype_of<double> { enum { value = HBSM_F64 }; };
template <> struct dtype_of<float> { enum { value = HBSM_F32 }; };
inline void check(int rc) {
    if (rc != HBSM_OK) throw std::runtime_error(hbsm_last_error());
}
}  // namespace detail

template <class Treal>
class HierarchicalBlockSparseMatrix {
public:
    typedef Treal real;   // H:40
    typedef HierarchicalBlockSparseMatrix<Treal> Self;

    struct Params {       // H:167-169
        int blocksize;
    };

    HierarchicalBlockSparseMatrix() : h_(NULL) { detail::check(hbsm_create(detail::dtype_of<Treal>::value, &h_)); }   // H:171
    ~HierarchicalBlockSparseMatrix() { if (h_) hbsm_destroy(h_); }                                                   // H:175
    HierarchicalBlockSparseMatrix(const HierarchicalBlockSparseMatrix& o) : h_(NULL) {
        detail::check(hbsm_create(detail::dtype_of<Treal>::value, &h_));
        copy(o);
    }
    HierarchicalBlockSparseMatrix& operator=(const HierarchicalBlockSparseMatrix& o) {
        if (this != &o) copy(o);
        return *this;
    }

    int get_n_rows() const { int r = 0, c = 0; detail::check(hbsm_dims(h_, &r, &c)); return r; }   // H:181
    int get_n_cols() const { int r = 0, c = 0; detail::check(hbsm_dims(h_, &r, &c)); return c; }   // H:184

    void set_params(Params const& param) { detail::check(hbsm_set_blocksize(h_, param.blocksize)); }   // H:186, H:450
    Params get_params() const { Params p; detail::check(hbsm_get_blocksize(h_, &p.blocksize)); return p; }   // H:188

    bool children_exist() const { int v = 0; detail::check(hbsm_children_exist(h_, &v)); return v != 0; }   // H:190
    bool empty() const { int v = 0; detail::check(hbsm_is_empty(h_, &v)); return v != 0; }                   // H:192

    void resize(int nRows_, int nCols_, size_t* no_of_resizes = NULL) {   // H:194, H:544
        detail::check(hbsm_resize(h_, nRows_, nCols_));
        if (no_of_resizes) (*no_of_resizes)++;
    }
    void clear() { detail::check(hbsm_clear(h_)); }   // H:196

    void assign_from_vectors_general(const std::vector<int>& rows, const std::vector<int>& cols,
                                     const std::vector<Treal>& values, bool useMax, bool boundaries_checked) {   // H:198, H:668
        if (rows.size() != values.size() || cols.size() != values.size())   // H:677
            throw std::runtime_error("Error in HierarchicalBlockSparseMatrix<Treal>::assign_from_vectors: bad sizes.");
        detail::check(hbsm_assign_coo(h_, values.size(), rows.data(), cols.data(), values.data(), useMax ? 1 : 0,
                                      boundaries_checked ? 1 : 0));
    }
    void assign_from_vectors(const std::vector<int>& rows, const std::vector<int>& cols, const std::vector<Treal>& values) {
        assign_from_vectors_general(rows, cols, values, false, false);   // H:838
    }
    void assign_from_vectors_max(const std::vector<int>& rows, const std::vector<int>& cols, const std::vector<Treal>& values) {
        assign_from_vectors_general(rows, cols, values, true, false);    // H:845
    }

    Treal get_frob_squared() const { Treal v = 0; detail::check(hbsm_frob_squared(h_, &v)); return v; }   // H:214, H:641
    Treal get_frob_norm_squared_internal() const { Treal v = 0; detail::check(hbsm_frob_squared_cached(h_, &v)); return v; }   // H:216
    size_t get_n_block_multiplications() const { size_t n = 0; detail::check(hbsm_get_n_block_multiplications(h_, &n)); return n; }   // H:218
    void set_n_block_multiplicaitons(size_t n) { detail::check(hbsm_set_n_block_multiplications(h_, n)); }   // H:220 (sic)
    void update_internal_info() { detail::check(hbsm_update_norms(h_)); }   // H:223, H:3905
    size_t get_nnz() const { size_t n = 0; detail::check(hbsm_nnz(h_, &n)); return n; }   // H:225
    int get_depth() const { int d = 0; detail::check(hbsm_depth(h_, &d)); return d; }     // H:228
    int expected_depth() const { int d = 0; detail::check(hbsm_expected_depth(h_, &d)); return d; }   // H:230

    void get_values(const std::vector<int>& rows, const std::vector<int>& cols, std::vector<Treal>& values) const {   // H:233, H:1012
        if (rows.size() != cols.size())
            throw std::runtime_error("Error in HierarchicalBlockSparseMatrix<Treal>::get_values: bad sizes.");
        values.resize(rows.size());
        detail::check(hbsm_get_values(h_, rows.size(), rows.data(), cols.data(), values.data()));
    }
    void get_all_values(std::vector<int>& rows, std::vector<int>& cols, std::vector<Treal>& values) const {   // H:237, H:1034
        size_t n = 0;
        detail::check(hbsm_get_all_values(h_, 0, NULL, NULL, NULL, &n));
        rows.resize(n); cols.resize(n); values.resize(n);
        if (n) detail::check(hbsm_get_all_values(h_, n, rows.data(), cols.data(), values.data(), &n));
    }

    static void allocate_work_buffers(int /*max_dimension*/, int /*max_blocksize*/) {}   // H:248

    void copy(const HierarchicalBlockSparseMatrix<Treal>& other, size_t* no_of_resizes = NULL) {   // H:251, H:1490
        detail::check(hbsm_copy(h_, other.h_));
        if (no_of_resizes) (*no_of_resizes)++;
    }

    static void add(HierarchicalBlockSparseMatrix<Treal> const& A, HierarchicalBlockSparseMatrix<Treal> const& B,
                    HierarchicalBlockSparseMatrix<Treal>& C, size_t* no_of_resizes = NULL) {   // H:255, H:1644
        detail::check(hbsm_add(A.h_, B.h_, C.h_));
        if (no_of_resizes) (*no_of_resizes)++;
    }

    static void multiply(HierarchicalBlockSparseMatrix<Treal> const& A, bool tA, HierarchicalBlockSparseMatrix<Treal> const& B,
                         bool tB, HierarchicalBlockSparseMatrix<Treal>& C, size_t* no_of_block_multiplies = NULL,
                         size_t* no_of_resizes = NULL) {   // H:260, H:2142
        size_t nm = 0, nr = 0;
        detail::check(hbsm_multiply(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, C.h_, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;   // H:2186-2190
        if (no_of_resizes) *no_of_resizes = nr;
    }

    void rescale(HierarchicalBlockSparseMatrix<Treal> const& other, Treal alpha) {   // H:265, H:3078
        detail::check(hbsm_rescale(h_, other.h_, (double)alpha));
    }

    static void symm_multiply(HierarchicalBlockSparseMatrix<Treal> const& A, bool sA, HierarchicalBlockSparseMatrix<Treal> const& B,
                              bool sB, HierarchicalBlockSparseMatrix<Treal>& C) {   // H:274, H:3244
        detail::check(hbsm_symm_multiply(A.h_, sA ? 1 : 0, B.h_, sB ? 1 : 0, C.h_));
    }
    static void symm_square(HierarchicalBlockSparseMatrix<Treal> const& A, HierarchicalBlockSparseMatrix<Treal>& C) {   // H:277, H:3563
        detail::check(hbsm_symm_square(A.h_, C.h_));
    }
    static void symm_rk(HierarchicalBlockSparseMatrix<Treal> const& A, bool transposed, HierarchicalBlockSparseMatrix<Treal>& C) {   // H:280, H:3711
        detail::check(hbsm_symm_rk(A.h_, transposed ? 1 : 0, C.h_));
    }
    static void transpose(HierarchicalBlockSparseMatrix<Treal> const& A, HierarchicalBlockSparseMatrix<Treal>& C) {   // H:282, H:3733
        detail::check(hbsm_transpose(A.h_, C.h_));
    }
    void get_upper_triangle(HierarchicalBlockSparseMatrix<Treal>& A) const {   // H:284, H:3515: A = triu(*this)
        detail::check(hbsm_upper_triangle(h_, A.h_));
    }

    void print() const {   // H:295
        std::vector<int> rows, cols;
        std::vector<Treal> vals;
        get_all_values(rows, cols, vals);
        for (size_t i = 0; i < rows.size(); ++i) std::cout << rows[i] << " " << cols[i] << " " << vals[i] << std::endl;
    }

    static void spamm(HierarchicalBlockSparseMatrix<Treal> const& A, bool tA, HierarchicalBlockSparseMatrix<Treal> const& B, bool tB,
                      HierarchicalBlockSparseMatrix<Treal>& C, const Treal tau, bool updated,
                      size_t* no_of_block_multiplies = NULL, size_t* no_of_resizes = NULL) {   // H:305, H:3931
        size_t nm = 0, nr = 0;
        detail::check(hbsm_spamm(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, C.h_, (double)tau, updated ? 1 : 0, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;   // H:3976-3982
        if (no_of_resizes) *no_of_resizes = nr;
    }

    // engine extras: C <- alpha * op(A) * op(B) + beta * C in one call (hbsm_multiply_accumulate); C may be A and/or B, or empty.
    // The out-parameters are those of multiply / spamm: products executed, and C's block count.
    static void multiply_accumulate(HierarchicalBlockSparseMatrix<Treal> const& A, bool tA, HierarchicalBlockSparseMatrix<Treal> const& B,
                                    bool tB, HierarchicalBlockSparseMatrix<Treal>& C, Treal alpha, Treal beta,
                                    size_t* no_of_block_multiplies = NULL, size_t* no_of_resizes = NULL) {
        size_t nm = 0, nr = 0;
        detail::check(hbsm_multiply_accumulate(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, C.h_, (double)alpha, (double)beta, 0, 0.0, 1, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;
        if (no_of_resizes) *no_of_resizes = nr;
    }
    static void spamm_accumulate(HierarchicalBlockSparseMatrix<Treal> const& A, bool tA, HierarchicalBlockSparseMatrix<Treal> const& B,
                                 bool tB, HierarchicalBlockSparseMatrix<Treal>& C, Treal alpha, Treal beta, const Treal tau,
                                 bool updated = true, size_t* no_of_block_multiplies = NULL, size_t* no_of_resizes = NULL) {
        size_t nm = 0, nr = 0;
        detail::check(hbsm_multiply_accumulate(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, C.h_, (double)alpha, (double)beta, 1, (double)tau,
                                               updated ? 1 : 0, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;
        if (no_of_resizes) *no_of_resizes = nr;
    }

    static int get_blocksize(Params const& param, int /*max_dimension*/) { return param.blocksize; }   // H:315

    bool check_if_matrix_is_consistent() const { int v = 0; detail::check(hbsm_is_consistent(h_, &v)); return v != 0; }   // H:396

    static bool worth_to_multiply(HierarchicalBlockSparseMatrix<Treal> const& A, const bool tA,
                                  HierarchicalBlockSparseMatrix<Treal> const& B, const bool tB) {   // H:399, H:1873
        int v = 0;
        detail::check(hbsm_worth_to_multiply(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, &v));
        return v != 0;
    }
    static bool worth_to_spamm(HierarchicalBlockSparseMatrix<Treal> const& A, const bool tA,
                               HierarchicalBlockSparseMatrix<Treal> const& B, const bool tB, const Treal tau) {   // H:402, H:2006
        int v = 0;
        detail::check(hbsm_worth_to_spamm(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, (double)tau, &v));
        return v != 0;
    }

    // ---- engine extras (not in the reference): executed-product list, tile count, SpAMM-pruned symmetric square ----
    size_t get_n_blocks() const { size_t n = 0; detail::check(hbsm_n_blocks(h_, &n)); return n; }   // reference: private, H:7311
    static void symm_square_spamm(HierarchicalBlockSparseMatrix<Treal> const& A, HierarchicalBlockSparseMatrix<Treal>& C,
                                  const Treal tau, size_t* no_of_block_multiplies = NULL, size_t* no_of_resizes = NULL) {
        size_t nm = 0, nr = 0;
        detail::check(hbsm_symm_square_spamm(A.h_, C.h_, (double)tau, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;
        if (no_of_resizes) *no_of_resizes = nr;
    }
    hbsm_handle handle() const { return h_; }
    // Y = alpha * op(A) * X + beta * Y on host arrays (column-major, leading dimensions ldx / ldy); op is HBSM_OP_N,
    // HBSM_OP_T or HBSM_OP_SYM_UPPER (triu(A) + striu(A)^T); leaf sizes up to 256.  The reference's get_row_sums / get_col_sums stubs below still
    // throw; A*1 and A^T*1 are multiply_dense with X = ones.
    static void multiply_dense(Self const& A, int op, int m, const Treal* X, int ldx, Treal* Y, int ldy, Treal alpha, Treal beta) {
        detail::check(hbsm_multiply_dense(A.h_, op, m, X, ldx, Y, ldy, (double)alpha, (double)beta));
    }
    // ||A||_2 by Lanczos, on A^T A, or on triu(A) + striu(A)^T when symmetric_upper.  lambda_min / lambda_max receive the
    // extreme Ritz values of that operator: the eigenvalue bounds of triu(A) + striu(A)^T, or those of A^T A (squared
    // singular values) without symmetric_upper.  The reference's spectral_norm() stub below still throws.
    Treal spectral_norm_estimate(bool symmetric_upper, int max_iter, Treal rel_tol, int* n_iter = NULL, Treal* lambda_min = NULL,
                                 Treal* lambda_max = NULL) const {
        double nrm = 0, lo = 0, hi = 0;
        int it = 0;
        detail::check(hbsm_spectral_norm(h_, symmetric_upper ? 1 : 0, max_iter, (double)rel_tol, &nrm, &lo, &hi, &it));
        if (n_iter) *n_iter = it;
        if (lambda_min) *lambda_min = (Treal)lo;
        if (lambda_max) *lambda_max = (Treal)hi;
        return (Treal)nrm;
    }
    // C = *this without the leaves of the largest ||.||_F^2 level whose error matrix E (triu(E) + striu(E)^T when
    // symmetric_upper) has ||E||_2 <= eps by the search of hbsm_spectral_block_trunc; info (may be NULL) receives its record.
    // The reference's get_spectral_squared_of_error_matrix / spectral_norm stubs below still throw.
    void spectral_block_trunc(HierarchicalBlockSparseMatrix<Treal>& C, Treal eps, bool symmetric_upper, int max_iter,
                              hbsm_trunc_info* info = NULL) const {
        hbsm_trunc_info t;
        detail::check(hbsm_spectral_block_trunc(h_, symmetric_upper ? 1 : 0, (double)eps, max_iter, C.h_, &t));
        if (info) *info = t;
    }
    // out[i] = Lanczos estimate of ||E_i||_2, E_i = the leaves frob_block_trunc(taus[i]) would drop (hbsm_truncation_spectral_errors)
    void get_spectral_errors_of_truncation(std::vector<Treal>& out, std::vector<Treal> const& taus, bool symmetric_upper, int max_iter,
                                           Treal rel_tol) const {
        std::vector<double> t(taus.begin(), taus.end()), nrm(taus.size());
        std::vector<int> it(taus.size());
        detail::check(hbsm_truncation_spectral_errors(h_, symmetric_upper ? 1 : 0, t.size(), t.empty() ? NULL : &t[0], max_iter,
                                                      (double)rel_tol, nrm.empty() ? NULL : &nrm[0], it.empty() ? NULL : &it[0]));
        out.assign(nrm.begin(), nrm.end());
    }
    // ---- multi-GPU extras (not in the reference; one process per GPU, see hbsm::comm below and INTEGRATION.md) ----
    // Every rank holds matrices with the FULL logical dimensions but only the tiles of its slab of block rows (C row for
    // op(A), contraction index for op(B)) and receives the same slab of C.  publish() is the distributed half of
    // update_internal_info() for a right operand; the sharded_* statics are collective and mirror multiply (H:260) /
    // spamm (H:305) / symm_square (H:277) argument for argument; the counters they return are this rank's.
    void publish() { detail::check(hbsm_publish(h_)); }
    static void sharded_multiply(HierarchicalBlockSparseMatrix<Treal> const& A, bool tA, HierarchicalBlockSparseMatrix<Treal>& B, bool tB,
                                 HierarchicalBlockSparseMatrix<Treal>& C, size_t* no_of_block_multiplies = NULL,
                                 size_t* no_of_resizes = NULL) {
        size_t nm = 0, nr = 0;
        detail::check(hbsm_sharded_product(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, C.h_, 0, 0.0, 0, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;
        if (no_of_resizes) *no_of_resizes = nr;
    }
    static void sharded_spamm(HierarchicalBlockSparseMatrix<Treal> const& A, bool tA, HierarchicalBlockSparseMatrix<Treal>& B, bool tB,
                              HierarchicalBlockSparseMatrix<Treal>& C, const Treal tau, size_t* no_of_block_multiplies = NULL,
                              size_t* no_of_resizes = NULL) {
        size_t nm = 0, nr = 0;
        detail::check(hbsm_sharded_product(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, C.h_, 1, (double)tau, 0, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;
        if (no_of_resizes) *no_of_resizes = nr;
    }
    // F: a symmetric matrix in FULL storage, row-sharded and published; C = this rank's block rows of triu(F*F), SpAMM-pruned
    // with tau (prune = false: exact, symm_square H:3563 of F's upper triangle)
    static void sharded_symm_square(HierarchicalBlockSparseMatrix<Treal>& F, HierarchicalBlockSparseMatrix<Treal>& C, bool prune,
                                    const Treal tau, size_t* no_of_block_multiplies = NULL, size_t* no_of_resizes = NULL) {
        size_t nm = 0, nr = 0;
        detail::check(hbsm_sharded_product(F.h_, 0, F.h_, 0, C.h_, prune ? 1 : 0, (double)tau, 1, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;
        if (no_of_resizes) *no_of_resizes = nr;
    }
    // Host-to-host multiply / SpAMM in one pipelined call (hbsm_product_from_host): A and B are sized matrices without
    // tiles; their dense column-major tiles come from host arrays (tile t at block (a_bi[t], a_bj[t])), C's tiles go to
    // c_tiles (room for cap_tiles tiles; c_bi/c_bj receive their block coordinates).  PCIe upload, norm refresh, leaf
    // GEMMs and download overlap slab by slab; afterwards A, B (norms fresh) and C live on the device as usual.
    static void product_from_host_tiles(HierarchicalBlockSparseMatrix<Treal>& A, size_t n_a, const int* a_bi, const int* a_bj,
                                        const Treal* a_tiles, bool tA, HierarchicalBlockSparseMatrix<Treal>& B, size_t n_b,
                                        const int* b_bi, const int* b_bj, const Treal* b_tiles, bool tB,
                                        HierarchicalBlockSparseMatrix<Treal>& C, bool use_spamm, const Treal tau, Treal* c_tiles,
                                        size_t cap_tiles, int* c_bi, int* c_bj, size_t* no_of_block_multiplies = NULL,
                                        size_t* no_of_resizes = NULL) {
        size_t nm = 0, nr = 0;
        detail::check(hbsm_product_from_host(A.h_, n_a, a_bi, a_bj, a_tiles, tA ? 1 : 0, B.h_, n_b, b_bi, b_bj, b_tiles, tB ? 1 : 0,
                                             C.h_, use_spamm ? 1 : 0, (double)tau, 0, c_tiles, cap_tiles, c_bi, c_bj, &nm, &nr));
        if (no_of_block_multiplies) *no_of_block_multiplies = nm;
        if (no_of_resizes) *no_of_resizes = nr;
    }

    // ---- host-side utilities around the hot path (SURVEY 8f "next"), built on the calls above ----
    // add_scaled_identity H:1532: *this = other + alpha * I.  (The reference also writes alpha onto the diagonal of the
    // zero padding of boundary leaves; that region is invisible through the element API and is left zero here.)
    void add_scaled_identity(HierarchicalBlockSparseMatrix<Treal> const& other, Treal alpha) {
        if (other.empty()) throw std::runtime_error("Error in HierarchicalBlockSparseMatrix::add_scaled_identity(): empty matrix as input!");
        HierarchicalBlockSparseMatrix<Treal> I;
        I.set_params(other.get_params());
        const int n = other.get_n_rows() < other.get_n_cols() ? other.get_n_rows() : other.get_n_cols();
        I.resize(other.get_n_rows(), other.get_n_cols());
        std::vector<int> idx(n);
        std::vector<Treal> v(n, alpha);
        for (int i = 0; i < n; ++i) idx[i] = i;
        I.assign_from_vectors(idx, idx, v);
        add(other, I, *this);
        set_n_block_multiplicaitons(0);
    }

    // set_to_identity H:3805 (params of A must be set)
    static void set_to_identity(HierarchicalBlockSparseMatrix<Treal>& A, int nRows) {
        A.clear();
        A.resize(nRows, nRows);
        std::vector<int> idx(nRows);
        std::vector<Treal> v(nRows, (Treal)1);
        for (int i = 0; i < nRows; ++i) idx[i] = i;
        A.assign_from_vectors(idx, idx, v);
    }

    // get_trace H:3782: leaf diagonals summed in order, quadrants combined as child0 + child3 -- same summation tree here
    Treal get_trace() const {
        const int n = get_n_rows() < get_n_cols() ? get_n_rows() : get_n_cols();
        if (n <= 0) return (Treal)0;
        std::vector<int> idx(n);
        for (int i = 0; i < n; ++i) idx[i] = i;
        std::vector<Treal> d;
        get_values(idx, idx, d);
        const int b = get_params().blocksize;
        long long vsize = b;
        for (int l = expected_depth(); l > 0; --l) vsize *= 2;
        return trace_rec(d, 0, vsize, b);
    }

    // get_nnz_diag_lowest_level H:3843: blocksize^2 per EXISTING diagonal leaf (zeros count, absent leaves do not)
    size_t get_nnz_diag_lowest_level() const {
        std::vector<int64_t> bi, bj;
        leaf_coordinates(bi, bj);
        const size_t b = (size_t)get_params().blocksize;
        size_t n = 0;
        for (size_t i = 0; i < bi.size(); ++i) n += (bi[i] == bj[i]) ? b * b : 0;
        return n;
    }

    // get_max_abs_value H:5177
    Treal get_max_abs_value() const {
        std::vector<int> r, c;
        std::vector<Treal> v;
        get_all_values(r, c, v);
        Treal m = 0;
        for (size_t i = 0; i < v.size(); ++i) { Treal a = v[i] < 0 ? -v[i] : v[i]; if (a > m) m = a; }
        return m;
    }

    // random_blocks H:3005: nnz_blocks distinct leaf blocks filled with uniform [-1,1) values (matrix must be resized, and
    // empty of elements: assembly is one-shot, H:793)
    void random_blocks(size_t nnz_blocks) {
        const int b = get_params().blocksize, M = get_n_rows(), N = get_n_cols();
        const int nb1 = M / b + (M % b > 0), nb2 = N / b + (N % b > 0);
        const size_t total = (size_t)nb1 * nb2;
        if (nnz_blocks > total) throw std::runtime_error("Error in HierarchicalBlockSparseMatrix::random_blocks():too many blocks!");
        std::vector<size_t> order(total);
        for (size_t i = 0; i < total; ++i) order[i] = i;
        uint64_t state = 0x9E3779B97F4A7C15ull ^ (uint64_t)(uintptr_t)this ^ ((uint64_t)nnz_blocks << 32);
        for (size_t i = total; i > 1; --i) { size_t j = (size_t)(next_random(state) % i); size_t t = order[i - 1]; order[i - 1] = order[j]; order[j] = t; }
        std::vector<int> rows, cols;
        std::vector<Treal> vals;
        for (size_t k = 0; k < nnz_blocks; ++k) {
            const int r0 = b * (int)(order[k] % nb1), c0 = b * (int)(order[k] / nb1);
            for (int j = 0; j < b; ++j)
                for (int i = 0; i < b; ++i) {
                    if (r0 + i >= M || c0 + j >= N) continue;
                    rows.push_back(r0 + i); cols.push_back(c0 + j);
                    vals.push_back((Treal)(2.0 * ((double)(next_random(state) >> 11) * (1.0 / 9007199254740992.0)) - 1.0));
                }
        }
        assign_from_vectors(rows, cols, vals);
    }

    // frob_block_trunc H:4935 (device): matrix_truncated = *this without the blocks of Frobenius norm < trunc_value
    bool frob_block_trunc(HierarchicalBlockSparseMatrix<Treal>& matrix_truncated, Treal trunc_value) const {
        int removed = 0;
        detail::check(hbsm_frob_block_trunc(h_, matrix_truncated.h_, (double)trunc_value, &removed));
        return removed != 0;
    }

    // get_frob_squared_of_error_matrix H:3863: entry i = norm^2 of the part that truncation at trunc_values[i] would drop,
    // i.e. the sum over leaves with ||leaf||_F < trunc_values[i], added up the quadtree in child order 0..3
    void get_frob_squared_of_error_matrix(std::vector<Treal>& frob_squared_of_error_matrix, std::vector<Treal> const& trunc_values) const {
        std::vector<int64_t> bi, bj;
        leaf_coordinates(bi, bj);
        std::vector<Treal> nsq(bi.size());
        size_t n = 0;
        if (!bi.empty()) detail::check(hbsm_leaf_norms(h_, nsq.size(), nsq.data(), &n));
        frob_squared_of_error_matrix.assign(trunc_values.size(), (Treal)0);
        if (bi.empty()) return;
        std::vector<uint64_t> key(bi.size());
        for (size_t i = 0; i < bi.size(); ++i) key[i] = hbsm_morton_encode((uint32_t)bi[i], (uint32_t)bj[i]);
        for (size_t t = 0; t < trunc_values.size(); ++t)
            frob_squared_of_error_matrix[t] = error_rec(key, nsq, 0, key.size(), expected_depth(), trunc_values[t]);
    }

    // wire format of the reference (H:1124-1487), byte-compatible: what the Chunks-and-Tasks runtime ships
    size_t get_size() const { size_t n = 0; detail::check(hbsm_serialized_size(h_, &n)); return n; }                       // H:241
    void write_to_buffer(char* dataBuffer, size_t const bufferSize) const { detail::check(hbsm_serialize(h_, dataBuffer, bufferSize)); }   // H:244
    void assign_from_buffer(const char* dataBuffer, size_t const bufferSize) { detail::check(hbsm_deserialize(h_, dataBuffer, bufferSize)); }   // H:245

    // a-priori estimators from the cached norms (count_skips H:4945, get_errors_of_approx_multiplication H:5193,
    // get_spamm_errors H:5236): host recursion over the per-level norm tables inside the engine
    static std::vector<unsigned long int> count_skips(HierarchicalBlockSparseMatrix<Treal> const& A, const bool tA,
                                                      HierarchicalBlockSparseMatrix<Treal> const& B, const bool tB,
                                                      std::vector<Treal> const& taus, const bool& apply_truncation, const bool& apply_spamm) {
        std::vector<double> t(taus.begin(), taus.end());
        std::vector<unsigned long int> out(taus.size(), 0);
        detail::check(hbsm_count_skips(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, t.size(), t.data(), apply_truncation ? 1 : 0, apply_spamm ? 1 : 0, out.data()));
        return out;
    }
    static std::vector<Treal> get_errors_of_approx_multiplication(HierarchicalBlockSparseMatrix<Treal> const& A, const bool tA,
                                                                  HierarchicalBlockSparseMatrix<Treal> const& B, const bool tB,
                                                                  std::vector<Treal> const& taus, const bool& apply_truncation, const bool& apply_spamm) {
        std::vector<unsigned long int> skips = count_skips(A, tA, B, tB, taus, apply_truncation, apply_spamm);
        std::vector<Treal> errors(skips.size(), (Treal)0);
        const Treal c1 = A.get_max_abs_value(), c2 = B.get_max_abs_value(), cm = c1 > c2 ? c1 : c2;
        for (size_t i = 0; i < errors.size(); ++i) {
            const Treal base = std::sqrt(taus[i] * taus[i] * skips[i]);
            if (apply_truncation && !apply_spamm) errors[i] = cm * base;
            else if (!apply_truncation && apply_spamm) errors[i] = base;
            else if (apply_truncation && apply_spamm) errors[i] = (cm > (Treal)1 ? cm : (Treal)1) * base;
        }
        return errors;
    }
    static std::vector<Treal> get_spamm_errors(HierarchicalBlockSparseMatrix<Treal> const& A, const bool tA,
                                               HierarchicalBlockSparseMatrix<Treal> const& B, const bool tB, std::vector<Treal> const& taus) {
        std::vector<double> t(taus.begin(), taus.end()), out(taus.size(), 0.0);
        size_t n = 0;
        detail::check(hbsm_spamm_errors(A.h_, tA ? 1 : 0, B.h_, tB ? 1 : 0, t.size(), t.data(), out.data(), &n));
        return std::vector<Treal>(out.begin(), out.begin() + n);
    }

    // inv_chol H:3110: inverse Cholesky factor Z (upper triangular, Z^T A Z = I) by the reference's block recursion
    //   Z00 = invchol(A00);  X = -Z00 (Z00^T A01);  Z11 = invchol(A10 X + A11);  Z01 = X Z11
    // The recursion runs on the host over quadrant matrices; every product / sum in it is the engine's multiply / add /
    // rescale on the GPU, and the b x b leaf factor (the scalar loop of H:3118-3140) is one device kernel, hbsm_leaf_inv_chol.
    static void inv_chol(HierarchicalBlockSparseMatrix<Treal> const& A, HierarchicalBlockSparseMatrix<Treal>& Z) {
        if (!Z.empty()) throw std::runtime_error("Error in HierarchicalBlockSparseMatrix::inv_chol(): non-empty matrix to write result!");
        if (A.get_n_rows() != A.get_n_cols()) throw std::runtime_error("Error in HierarchicalBlockSparseMatrix::inv_chol(): call for non-square matrix!");
        Z.set_params(A.get_params());
        inv_chol_rec(A, Z, A.get_n_rows(), A.get_n_rows());
    }

    // ---- members outside the multiply / SpAMM / add path (SURVEY 2 "OUT OF SCOPE", 8f "next"): declared, throwing ----
#define HBSM_B200_NOT_PROVIDED(name) \
    throw std::runtime_error("Error in HierarchicalBlockSparseMatrix<Treal>::" name ": not provided by hbsm_b200 (outside the multiply/SpAMM/add path).")
    static void adjust_sizes(HierarchicalBlockSparseMatrix<Treal>&, const int, const int) { HBSM_B200_NOT_PROVIDED("adjust_sizes"); }   // H:286
#undef HBSM_B200_NOT_PROVIDED

    // ---- the reference's own "dummy function, for compatibility" stubs (H:271, H:317-427): same throwing behaviour ----
#define HBSM_B200_STUB(name) \
    throw std::runtime_error("Error in HierarchicalBlockSparseMatrix<Treal>::" name ": function not yet implemented.")
    static void inv_chol_trunc(HierarchicalBlockSparseMatrix<Treal> const&, HierarchicalBlockSparseMatrix<Treal>&, Treal) { HBSM_B200_STUB("inv_chol_trunc"); }
    void get_col_sums(std::vector<Treal>&) const { HBSM_B200_STUB("get_col_sums"); }
    void get_col_sums_part(std::vector<Treal>&, const int, const int) const { HBSM_B200_STUB("get_col_sums_part"); }
    void get_row_sums(std::vector<Treal>&) const { HBSM_B200_STUB("get_row_sums"); }
    void get_row_sums_part(std::vector<Treal>&, const int, const int) const { HBSM_B200_STUB("get_row_sums_part"); }
    void get_diag(std::vector<Treal>&) const { HBSM_B200_STUB("get_diag"); }
    void get_diag_part(std::vector<Treal>&, int, int) const { HBSM_B200_STUB("get_diag_part"); }
    void get_spectral_squared_of_error_matrix(std::vector<Treal>&, std::vector<Treal> const&, int, bool) const { HBSM_B200_STUB("get_spectral_squared_of_error_matrix"); }
    Treal get_frob_squared_symm() const { HBSM_B200_STUB("get_frob_squared_symm"); }
    void get_frob_squared_of_error_matrix_symm(std::vector<Treal>&, std::vector<Treal> const&) const { HBSM_B200_STUB("get_frob_squared_of_error_matrix_symm"); }
    bool frob_block_trunc_symm(HierarchicalBlockSparseMatrix<Treal>&, Treal) const { HBSM_B200_STUB("frob_block_trunc_symm"); }
    void set_neg_to_zero(const HierarchicalBlockSparseMatrix<Treal>&) { HBSM_B200_STUB("get_row_sums_part"); }
    static void max(HierarchicalBlockSparseMatrix<Treal> const&, HierarchicalBlockSparseMatrix<Treal> const&, HierarchicalBlockSparseMatrix<Treal>&) { HBSM_B200_STUB("max"); }
    Treal spectral_norm(int = 0, bool = false) const { HBSM_B200_STUB("spectral_norm"); }
    void get_nnz_in_submatrix(std::vector<int>&, std::vector<int>&, std::vector<Treal>&, int, int, int, int) const { HBSM_B200_STUB("spectral_norm"); }
    static void symm_rk_TN(HierarchicalBlockSparseMatrix<Treal> const&, HierarchicalBlockSparseMatrix<Treal>&) { HBSM_B200_STUB("symm_rk_TN"); }
    static void symm_rk_NT(HierarchicalBlockSparseMatrix<Treal> const&, HierarchicalBlockSparseMatrix<Treal>&) { HBSM_B200_STUB("symm_rk_NT"); }
    void symm_to_nosymm() { HBSM_B200_STUB("symm_to_nosymm"); }
    void nosymm_to_symm() { HBSM_B200_STUB("nosymm_to_symm"); }
    static void submatrix_inv_chol(std::vector<real> const&, std::vector<real>&, int, int) { HBSM_B200_STUB("submatrix_inv_chol"); }
    static void anticommutator(HierarchicalBlockSparseMatrix<Treal> const&, HierarchicalBlockSparseMatrix<Treal> const&, HierarchicalBlockSparseMatrix<Treal>&) {
        throw std::runtime_error("Error in HierarchicalBlockSparseMatrix<Treal>::anticommutator: function not applicable.");
    }
    static void symm_product(HierarchicalBlockSparseMatrix<Treal> const&, HierarchicalBlockSparseMatrix<Treal> const&, const bool, HierarchicalBlockSparseMatrix<Treal>&) {
        throw std::runtime_error("Error in HierarchicalBlockSparseMatrix<Treal>::symm_product: function not applicable.");
    }
#undef HBSM_B200_STUB

private:
    hbsm_handle h_;

    bool quadrant(int q, Self& out) const {
        int e = 0;
        out.set_params(get_params());
        detail::check(hbsm_extract_quadrant(h_, q, out.h_, &e));
        return e != 0;
    }
    // A: node of virtual size v (dims = v unless it is the root); `valid` = rows/cols of it inside the real matrix;
    // Z receives dims (zdim, zdim)
    static void inv_chol_rec(Self const& A, Self& Z, int zdim, int valid) {
        const int b = A.get_params().blocksize;
        if (A.expected_depth() == 0) {   // leaf factor, H:3118-3147: one kernel on the leaf where it lies (hbsm_leaf_inv_chol)
            detail::check(hbsm_leaf_inv_chol(A.h_, Z.h_, zdim, valid));
            return;
        }
        long long v = b;
        for (int l = A.expected_depth(); l > 0; --l) v *= 2;
        const int half = (int)(v / 2);
        Self A00, A01, A10, A11;
        const bool h00 = A.quadrant(0, A00), h10 = A.quadrant(1, A10), h01 = A.quadrant(2, A01), h11 = A.quadrant(3, A11);
        if (!h00) throw std::runtime_error("Error in HierarchicalBlockSparseMatrix::inv_chol(): smth went wrong since Z_00 is NULL!");
        Self Z00, Z01, Z11, X;
        Z00.set_params(A.get_params()); Z01.set_params(A.get_params()); Z11.set_params(A.get_params());
        inv_chol_rec(A00, Z00, half, valid < half ? valid : half);
        bool hX = false, hQ = false, hZ11 = false, hZ01 = false;
        Self Q;
        if (h01) {
            Self R, T;
            multiply(Z00, true, A01, false, R);     // R = Z00^T A01
            multiply(Z00, false, R, false, T);      // T = Z00 R
            X.rescale(T, (Treal)-1);                // X = -T
            hX = true;
        }
        if (h10 && hX) {
            Self Y;
            multiply(A10, false, X, false, Y);      // Y = A10 X
            if (h11) add(Y, A11, Q); else Q.copy(Y);
            hQ = true;
        } else if (h11) {
            Q.copy(A11);
            hQ = true;
        }
        if (hQ && valid > half) {
            inv_chol_rec(Q, Z11, half, valid - half);
            hZ11 = !Z11.empty() && Z11.get_n_blocks() > 0;
        }
        if (hX && hZ11) {
            multiply(X, false, Z11, false, Z01);    // Z01 = X Z11
            hZ01 = true;
        }
        detail::check(hbsm_assemble_quadrants(Z.h_, zdim, zdim, Z00.h_, NULL, hZ01 ? Z01.h_ : NULL, hZ11 ? Z11.h_ : NULL));
    }

    static uint64_t next_random(uint64_t& s) {   // splitmix64
        s += 0x9E3779B97F4A7C15ull;
        uint64_t z = s;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    void leaf_coordinates(std::vector<int64_t>& bi, std::vector<int64_t>& bj) const {
        size_t n = 0;
        detail::check(hbsm_n_blocks(h_, &n));
        bi.resize(n); bj.resize(n);
        if (n) detail::check(hbsm_export_leaves(h_, n, bi.data(), bj.data(), NULL, NULL, &n));
    }
    // diagonal d[lo, lo+size) of the virtual matrix (entries past the end are zero padding)
    static Treal trace_rec(const std::vector<Treal>& d, long long lo, long long size, int b) {
        if (lo >= (long long)d.size()) return (Treal)0;
        if (size <= b) {
            Treal t = 0;
            for (long long i = lo; i < lo + size && i < (long long)d.size(); ++i) t += d[(size_t)i];
            return t;
        }
        Treal t = 0;
        t += trace_rec(d, lo, size / 2, b);
        t += trace_rec(d, lo + size / 2, size / 2, b);
        return t;
    }
    // leaves [lo,hi) of the Morton-sorted table below a node at `level` levels above the leaves
    static Treal error_rec(const std::vector<uint64_t>& key, const std::vector<Treal>& nsq, size_t lo, size_t hi, int level, Treal trunc) {
        if (lo >= hi) return (Treal)0;
        if (level == 0) return (std::sqrt(nsq[lo]) < trunc) ? nsq[lo] : (Treal)0;
        Treal child[4] = {0, 0, 0, 0};
        size_t p = lo;
        for (int q = 0; q < 4; ++q) {
            size_t e = p;
            while (e < hi && ((key[e] >> (2 * (level - 1))) & 3u) == (uint64_t)q) ++e;
            child[q] = error_rec(key, nsq, p, e, level - 1, trunc);
            p = e;
        }
        return child[0] + child[1] + child[2] + child[3];
    }
};

// One communicator per process (NCCL inside libhbsm_b200.so).  Rank 0 makes the id and hands its bytes to the other ranks by
// whatever the host program has (MPI_Bcast, a file, a socket); then every rank calls init after hbsm_init(device).
namespace comm {
inline std::vector<unsigned char> unique_id() {
    std::vector<unsigned char> id(HBSM_COMM_ID_BYTES);
    detail::check(hbsm_comm_unique_id(id.data()));
    return id;
}
inline void init(const std::vector<unsigned char>& id, int rank, int world) {
    if (id.size() != HBSM_COMM_ID_BYTES) throw std::runtime_error("hbsm::comm::init: the id must have HBSM_COMM_ID_BYTES bytes");
    detail::check(hbsm_comm_init(id.data(), rank, world));
}
inline void finalize() { detail::check(hbsm_comm_finalize()); }
inline void barrier() { detail::check(hbsm_comm_barrier()); }
inline void rows_of(int grid_side, int world, int rank, int& lo, int& hi) { detail::check(hbsm_shard_rows(grid_side, world, rank, &lo, &hi)); }
inline double sum(double v) { detail::check(hbsm_comm_allreduce_f64(&v, 1, 0)); return v; }
inline double max(double v) { detail::check(hbsm_comm_allreduce_f64(&v, 1, 1)); return v; }
}  // namespace comm

}  // namespace hbsm

#endif

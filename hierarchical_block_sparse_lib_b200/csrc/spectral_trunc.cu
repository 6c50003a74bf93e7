// spectral_trunc.cu -- block truncation with spectral-norm error control, and spectral norms of truncation error matrices.
//
// A truncation at level v drops exactly the leaves whose fresh ||.||_F^2 (nsq) is <= v; E_v is the dropped part, and the
// error operator is E_v, or sym(E_v) = triu(E_v) + striu(E_v)^T with symmetric_upper (tiles below the diagonal then play no
// part: they are never dropped).  Both are applied without materialising E_v: a masked line index selects E_v's entries out
// of A's own row and column line indices, and the dense product (dense.cu) walks it over A's tiles, so one Lanczos step
// reads E_v's tiles only.  The search over the distinct nsq levels and its brackets are described in DESIGN section 10.
#include "matrix.cuh"
#include <cmath>

namespace hbsm_b200 {
namespace {

inline unsigned blocks_for(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// a decision accepts only once the extreme Ritz pairs have converged to this relative residual bound
constexpr double ACCEPT_REL_TOL = 1e-3;

// sort key of leaf i: its nsq bits (non-negative IEEE values order as unsigned integers), or ~0 for a leaf the operator
// ignores (below the diagonal with symmetric_upper), which sorts behind every level
template <typename T>
__global__ void k_level_keys(const uint64_t* __restrict__ keys, const T* __restrict__ nsq, size_t n, int symmetric_upper,
                             uint64_t* __restrict__ skey, uint32_t* __restrict__ sidx) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t bits;
    if (sizeof(T) == 8) bits = (uint64_t)__double_as_longlong((double)nsq[i]);
    else bits = (uint64_t)(uint32_t)__float_as_uint((float)nsq[i]);
    skey[i] = (symmetric_upper && morton_row(keys[i]) > morton_col(keys[i])) ? ~0ull : bits;
    sidx[i] = (uint32_t)i;
}

// flag[order[i]] = (i < e) xor flip: the leaves of the first e sorted positions (flip = 0: dropped; flip = 1: kept)
__global__ void k_rank_flags(const uint32_t* __restrict__ order, size_t n, size_t e, uint32_t flip, uint32_t* __restrict__ flag) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[order[i]] = (i < e ? 1u : 0u) ^ flip;
}

// Masked line index.  The row index's L entries and the column index's L entries, concatenated, are flagged with
// sel[tile] xor flip; one exclusive scan of the 2L flags compacts both stably, so every line stays contiguous and ascending.
__global__ void k_mask_flags(const uint32_t* __restrict__ rtile, const uint32_t* __restrict__ ctile, size_t L,
                             const uint32_t* __restrict__ sel, uint32_t flip, uint32_t* __restrict__ flag) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 2 * L) flag[i] = sel[i < L ? rtile[i] : ctile[i - L]] ^ flip;
}
__global__ void k_mask_scatter(const uint32_t* __restrict__ rother, const uint32_t* __restrict__ rtile,
                               const uint32_t* __restrict__ cother, const uint32_t* __restrict__ ctile, size_t L,
                               const uint32_t* __restrict__ flag, const uint64_t* __restrict__ pos, uint32_t* __restrict__ mother,
                               uint32_t* __restrict__ mtile) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 2 * L || !flag[i]) return;
    const bool row = i < L;
    mother[pos[i]] = row ? rother[i] : cother[i - L];
    mtile[pos[i]] = row ? rtile[i] : ctile[i - L];
}
// ptr of the masked row lines = pos[row ptr]; of the masked column lines = pos[L + column ptr] - nd (they start at nd)
__global__ void k_mask_ptr(const uint32_t* __restrict__ rptr, const uint32_t* __restrict__ cptr, uint32_t n_lines, size_t L,
                           const uint64_t* __restrict__ pos, uint64_t nd, uint32_t* __restrict__ mptr) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t np = (size_t)n_lines + 1;
    if (i < np) mptr[i] = (uint32_t)pos[rptr[i]];
    else if (i < 2 * np) mptr[i] = (uint32_t)(pos[L + cptr[i - np]] - nd);
}

// The masked index of one matrix: buffers allocated once, rebuilt for each selection in O(L) (four launches and the scan's
// one read of its total)
struct MaskedIndex {
    const Matrix& A;
    OpView own, view;
    DevBuf<uint32_t> flag, other, tile, ptr;
    DevBuf<uint64_t> pos;
    explicit MaskedIndex(const Matrix& a) : A(a), own(own_view(a)) {
        flag.alloc(2 * A.L);
        other.alloc(2 * A.L);
        tile.alloc(2 * A.L);
        ptr.alloc(2 * ((size_t)A.grid_side() + 1));
    }
    // E's view: the leaves t with sel[t] xor flip != 0; returns how many
    size_t build(const uint32_t* sel, uint32_t flip) {
        const size_t L = A.L;
        const uint32_t nl = A.grid_side();
        HB_LAUNCH(k_mask_flags, blocks_for(2 * L, 256), 256, 0, own.row.tile, own.col.tile, L, sel, flip, flag.p);
        const size_t nd = scan_flags(flag, 2 * L, pos) / 2;   // every leaf sits in one row line and one column line
        HB_LAUNCH(k_mask_scatter, blocks_for(2 * L, 256), 256, 0, own.row.other, own.row.tile, own.col.other, own.col.tile, L, flag.p,
                  pos.p, other.p, tile.p);
        HB_LAUNCH(k_mask_ptr, blocks_for(2 * ((size_t)nl + 1), 256), 256, 0, own.row.ptr, own.col.ptr, nl, L, pos.p, (uint64_t)nd, ptr.p);
        view.row = LineView{ptr.p, other.p, tile.p};
        view.col = LineView{ptr.p + nl + 1, other.p + nd, tile.p + nd};
        return nd;
    }
};

void validate_common(const Matrix& A, bool symmetric_upper, int max_iter, const char* fn) {
    const std::string f = std::string("hbsm_b200: ") + fn + ": ";
    if (max_iter < 1) throw Error(HBSM_E_ARG, f + "max_iter < 1");
    if (symmetric_upper && A.M != A.N) throw Error(HBSM_E_ARG, f + "symmetric_upper needs a square A");
    if (A.b > 256) throw Error(HBSM_E_ARG, f + "leaf sizes above 256 have no kernel");
}

}  // namespace

// The search (DESIGN section 10).  Levels are the distinct nsq values of the leaves the operator uses, ascending.
//   lower bracket kF: the largest level whose Frobenius bound sum w * nsq (w = 2 with symmetric_upper, else 1) is <= eps^2:
//     ||E||_2 <= ||E||_F, and ||sym(T)||_F^2 <= 2 ||T||_F^2 for every tile, diagonal ones included.
//   upper bracket: the level of the first leaf that can never go -- an off-diagonal leaf (any leaf without symmetric_upper)
//     with nsq > b * eps^2, since ||E||_2 >= ||T||_2 >= ||T||_F / sqrt(b) -- and every level above it; a non-finite nsq
//     also ends the candidates.
//   between: the highest candidate first, then bisection keeping "lo accepted, hi rejected or excluded"; each test is a
//     decision-mode Lanczos run on E_level.  Monotonicity of ||E_v||_2 in v is not assumed.
TruncInfo spectral_block_trunc(const Matrix& A, bool symmetric_upper, double eps, int max_iter, Matrix& C) {
    if (&C == &A) throw Error(HBSM_E_ARG, "hbsm_b200: spectral_block_trunc: target must not alias the source");
    if (!(eps >= 0.0)) throw Error(HBSM_E_ARG, "hbsm_b200: spectral_block_trunc: eps must be >= 0 (and not NaN)");
    validate_common(A, symmetric_upper, max_iter, "spectral_block_trunc");
    TruncInfo info{};
    info.drop_nsq = -1.0;
    if (!trunc_begin(A, C)) return info;
    const size_t L = A.L;
    const bool f64 = A.dtype == HBSM_F64;
    DevBuf<char> nsq(L * A.esize());
    compute_leaf_norms(A, nsq.p);
    DevBuf<uint64_t> skey(L);
    DevBuf<uint32_t> sidx(L);
    if (f64) HB_LAUNCH(k_level_keys<double>, blocks_for(L, 256), 256, 0, A.keys.p, (const double*)nsq.p, L, symmetric_upper ? 1 : 0, skey.p, sidx.p);
    else HB_LAUNCH(k_level_keys<float>, blocks_for(L, 256), 256, 0, A.keys.p, (const float*)nsq.p, L, symmetric_upper ? 1 : 0, skey.p, sidx.p);
    radix_sort_pairs(skey.p, sidx.p, L, 64);   // stable
    const std::vector<uint64_t> hkey = skey.to_host();
    const std::vector<uint32_t> hidx = sidx.to_host();
    const std::vector<uint64_t> keys = A.keys.to_host();

    // levels below the upper bracket: value[g], end[g] = sorted positions with nsq <= value[g], frob[g] = the Frobenius
    // bound of dropping them (summed in ascending order)
    const double w = symmetric_upper ? 2.0 : 1.0, e2 = eps * eps, hard = (double)A.b * e2;
    auto nsq_at = [&](size_t i) {
        if (f64) { double x; memcpy(&x, &hkey[i], sizeof x); return x; }
        const uint32_t u = (uint32_t)hkey[i];
        float f;
        memcpy(&f, &u, sizeof f);
        return (double)f;
    };
    std::vector<size_t> end;
    std::vector<double> value, frob;
    double acc = 0.0;
    for (size_t i = 0; i < L && hkey[i] != ~0ull;) {
        const double x = nsq_at(i);
        if (!std::isfinite(x)) break;
        size_t j = i;
        bool never = false;   // the level holds a leaf that can never be dropped
        double s = acc;
        for (; j < L && hkey[j] == hkey[i]; ++j) {
            const uint64_t k = keys[hidx[j]];
            never = never || ((!symmetric_upper || morton_row(k) != morton_col(k)) && x > hard);
            s += w * x;
        }
        if (never) break;
        acc = s;
        value.push_back(x);
        end.push_back(j);
        frob.push_back(acc);
        i = j;
    }
    int hi = (int)value.size();   // first excluded level
    int lo = -1;
    while (lo + 1 < hi && frob[lo + 1] <= e2) ++lo;
    const int kF = lo;
    info.n_frob = kF >= 0 ? end[kF] : 0;
    info.err_bound = kF >= 0 ? std::sqrt(frob[kF]) : 0.0;

    if (lo + 1 < hi) {
        MaskedIndex mi(A);
        DevBuf<uint32_t> drop(L);
        double lo_bound = info.err_bound;
        auto test = [&](int g) {
            HB_LAUNCH(k_rank_flags, blocks_for(L, 256), 256, 0, sidx.p, L, end[g], 0u, drop.p);
            mi.build(drop.p, 0u);
            LanczosDecision d{eps, false, 0.0};
            const SpectralResult r = lanczos(A, mi.view, symmetric_upper, max_iter, ACCEPT_REL_TOL, &d);
            ++info.n_decisions;
            info.lanczos_steps += r.n_iter;
            if (d.feasible) lo_bound = d.bound;
            return d.feasible;
        };
        if (test(hi - 1)) lo = hi - 1;   // a large eps often drops everything droppable
        else hi = hi - 1;
        while (hi - lo > 1) {
            const int mid = lo + (hi - lo) / 2;
            if (test(mid)) lo = mid; else hi = mid;
        }
        if (lo > kF) { info.certified_by_lanczos = true; info.err_bound = lo_bound; }   // the last accepted test is level lo
    }

    const size_t e = lo >= 0 ? end[lo] : 0;
    info.n_dropped = e;
    info.drop_nsq = lo >= 0 ? value[lo] : -1.0;
    DevBuf<uint32_t> keep(L);
    HB_LAUNCH(k_rank_flags, blocks_for(L, 256), 256, 0, sidx.p, L, e, 1u, keep.p);
    trunc_compact(A, keep, C);
    return info;
}

// ||E_tau||_2 for each tau: E_tau = the leaves frob_block_trunc(A, tau) drops (nsq < tau^2 in Treal), by the
// full-convergence Lanczos run hbsm_spectral_norm makes on a matrix holding exactly those tiles (same walk, same bits)
void truncation_spectral_errors(const Matrix& A, bool symmetric_upper, size_t n, const double* taus, int max_iter, double rel_tol,
                                double* out_norms, int* out_iters) {
    if (!(rel_tol > 0.0)) throw Error(HBSM_E_ARG, "hbsm_b200: truncation_spectral_errors: rel_tol must be > 0");
    validate_common(A, symmetric_upper, max_iter, "truncation_spectral_errors");
    if (n > 0 && (!taus || !out_norms || !out_iters)) throw Error(HBSM_E_ARG, "hbsm_b200: truncation_spectral_errors: null taus or outputs");
    for (size_t i = 0; i < n; ++i) { out_norms[i] = 0.0; out_iters[i] = 0; }
    if (n == 0 || !A.sized || A.L == 0 || A.vdepth() == 0 || A.M == 0 || A.N == 0) return;   // nothing is ever dropped
    ensure_engine();
    DevBuf<char> nsq(A.L * A.esize());
    compute_leaf_norms(A, nsq.p);
    DevBuf<uint32_t> keep(A.L);
    MaskedIndex mi(A);
    for (size_t i = 0; i < n; ++i) {
        trunc_keep_flags(A, nsq.p, taus[i], keep.p);
        if (mi.build(keep.p, 1u) == 0) continue;
        const SpectralResult r = lanczos(A, mi.view, symmetric_upper, max_iter, rel_tol, nullptr);
        out_norms[i] = r.norm;
        out_iters[i] = r.n_iter;
    }
}

}  // namespace hbsm_b200

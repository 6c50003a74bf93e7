// spamm_error.cu -- SpAMM error control: a rigorous bound on the error of the leaf products SpAMM skips, at every threshold
// at once, and the threshold whose bound meets an error budget (DESIGN section 12).
//
// The candidates are the leaf pairs of the exact product, grouped by C tile (product_candidates).  Candidate i has the level
// p_i = fl(nsq_A * nsq_B) in Treal -- the number the product compares with fl(tau * tau) -- and s_i >= ||A_ik||_F ||B_kj||_F.
// At any tau the skipped candidates of C tile t are a prefix of t's candidates in p order; with S_t their sum of s,
// ||E||_F^2 <= w * sum_t S_t^2.  One pass gives that sum at every level:
//   sort by p, then stably by C tile: each tile's candidates in p order;
//   per tile, in that order, delta_i = s_i (2 S_prev + s_i): the exact growth of S_t^2 when i joins the skipped set;
//   back in p order, the prefix sums of delta: at the last candidate of a level they are sum_t S_t(level)^2.
// Every operation rounds upward and grows with its inputs, so each value bounds its exact counterpart from above.  The
// prefix sum runs sequentially at each of its three levels (items of a thread, threads of a block, blocks): bitwise
// repeatable and non-decreasing along the p order.
#include "matrix.cuh"
#include <cmath>

namespace hbsm_b200 {
namespace {

inline unsigned blocks_for(size_t n, unsigned threads) { return (unsigned)((n + threads - 1) / threads); }

// Sort keys of the levels: an IEEE value orders as an unsigned integer once a negative one is complemented and a positive
// one gets its sign bit set; NaN takes the largest key, behind every number.  fp32 keys use the low 32 bits.
template <typename T> struct LevelKey;
template <> struct LevelKey<double> {
    static constexpr uint64_t NAN_KEY = ~0ull;
    static constexpr int BITS = 64;
    __host__ __device__ static uint64_t of(double p) {
        if (p != p) return NAN_KEY;
        uint64_t u;
        memcpy(&u, &p, sizeof u);
        return (u >> 63) ? ~u : (u | (1ull << 63));
    }
    static double value(uint64_t k) {
        const uint64_t u = (k >> 63) ? (k & ~(1ull << 63)) : ~k;
        double p;
        memcpy(&p, &u, sizeof p);
        return p;
    }
};
template <> struct LevelKey<float> {
    static constexpr uint64_t NAN_KEY = 0xffffffffull;
    static constexpr int BITS = 32;
    __host__ __device__ static uint64_t of(float p) {
        if (p != p) return NAN_KEY;
        uint32_t u;
        memcpy(&u, &p, sizeof u);
        return (uint64_t)((u >> 31) ? ~u : (u | 0x80000000u));
    }
    static double value(uint64_t k) {
        const uint32_t u = (k >> 31) ? ((uint32_t)k & 0x7fffffffu) : ~(uint32_t)k;
        float p;
        memcpy(&p, &u, sizeof p);
        return (double)p;
    }
};

// Per candidate: its level key (fl(na * nb) in Treal, as spamm_keep in product.cu computes it), and
// s = sqrt(na) sqrt(nb) / (1 - gamma) rounded up, gamma covering the rounding of the sequential sums behind na and nb;
// a NaN s (a NaN or negative norm) becomes +Inf
template <typename T>
__global__ void k_cand_levels(const uint2* __restrict__ ab, size_t q, const T* __restrict__ an, const T* __restrict__ bn,
                              double one_minus_gamma, uint64_t* __restrict__ key, uint32_t* __restrict__ order,
                              double* __restrict__ s) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= q) return;
    const uint2 p = ab[i];
    const T na = an[p.x], nb = bn[p.y];
    key[i] = LevelKey<T>::of(DT<T>::mul(na, nb));
    const double si = __ddiv_ru(__dmul_ru(__dsqrt_ru((double)na), __dsqrt_ru((double)nb)), one_minus_gamma);
    s[i] = isnan(si) ? INFINITY : si;
    order[i] = (uint32_t)i;
}

// the C tile of every candidate (candidates are grouped by C tile: begin[t] .. begin[t + 1])
__global__ void k_tile_of(const uint64_t* __restrict__ begin, size_t nct, uint32_t* __restrict__ tile) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nct) return;
    for (uint64_t j = begin[t]; j < begin[t + 1]; ++j) tile[j] = (uint32_t)t;
}

__global__ void k_tile_keys(const uint32_t* __restrict__ order, const uint32_t* __restrict__ tile, size_t q,
                            uint64_t* __restrict__ tkey, uint32_t* __restrict__ by_tile) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= q) return;
    tkey[j] = tile[order[j]];
    by_tile[j] = order[j];
}

// per C tile, its candidates in p order: delta = s (2 S_prev + s), S_prev the running sum of s before, all rounded up
__global__ void k_tile_deltas(const uint64_t* __restrict__ begin, size_t nct, const uint32_t* __restrict__ by_tile,
                              const double* __restrict__ s, double* __restrict__ delta) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nct) return;
    double S = 0.0;
    for (uint64_t j = begin[t]; j < begin[t + 1]; ++j) {
        const uint32_t c = by_tile[j];
        const double x = s[c];
        delta[c] = x == 0.0 ? 0.0 : __dmul_ru(x, __dadd_ru(2.0 * S, x));
        S = __dadd_ru(S, x);
    }
}

// Inclusive prefix sum of delta in p order, rounded up.  A thread sums its PS_ITEMS consecutive items in order; thread 0 of
// the block chains the thread totals; a single thread chains the block totals.  Each level's last value is the next level's
// start, which keeps the result non-decreasing.
constexpr int PS_THREADS = 256, PS_ITEMS = 8, PS_TILE = PS_THREADS * PS_ITEMS;

__global__ void __launch_bounds__(PS_THREADS) k_prefix_local(const uint32_t* __restrict__ order, const double* __restrict__ delta,
                                                             size_t q, double* __restrict__ out, double* __restrict__ block_total) {
    __shared__ double tot[PS_THREADS], excl[PS_THREADS + 1];
    const size_t base = (size_t)blockIdx.x * PS_TILE + (size_t)threadIdx.x * PS_ITEMS;
    double run[PS_ITEMS];
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < PS_ITEMS; ++i) {
        if (base + i < q) acc = __dadd_ru(acc, delta[order[base + i]]);
        run[i] = acc;
    }
    tot[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double e = 0.0;
        for (int t = 0; t < PS_THREADS; ++t) {
            excl[t] = e;
            e = __dadd_ru(e, tot[t]);
        }
        excl[PS_THREADS] = e;
        block_total[blockIdx.x] = e;
    }
    __syncthreads();
    const double e = excl[threadIdx.x];
#pragma unroll
    for (int i = 0; i < PS_ITEMS; ++i)
        if (base + i < q) out[base + i] = __dadd_ru(e, run[i]);
}

__global__ void k_prefix_blocks(double* __restrict__ total, size_t nb) {   // in place: block totals -> block starts
    double e = 0.0;
    for (size_t b = 0; b < nb; ++b) {
        const double t = total[b];
        total[b] = e;
        e = __dadd_ru(e, t);
    }
}

__global__ void k_prefix_add(double* __restrict__ out, size_t q, const double* __restrict__ start) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < q) out[j] = __dadd_ru(start[j / PS_TILE], out[j]);
}

__global__ void k_level_heads(const uint64_t* __restrict__ key, size_t q, uint32_t* __restrict__ head) {
    const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < q) head[j] = (j == 0 || key[j] != key[j - 1]) ? 1u : 0u;
}

__device__ size_t lower_bound_key(const uint64_t* key, size_t n, uint64_t k) {
    size_t lo = 0, hi = n;
    while (lo < hi) {
        const size_t mid = lo + (hi - lo) / 2;
        if (key[mid] < k) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ double bound_at(const double* prefix, size_t j, double w) { return __dsqrt_ru(__dmul_ru(w, prefix[j])); }

// per tau: the candidates it skips (tkey = the key of fl(tau * tau) in Treal; NaN skips everything, and NaN levels are skipped
// at every tau) and their bound (+Inf when any level is NaN)
__global__ void k_eval(const uint64_t* __restrict__ key, const double* __restrict__ prefix, size_t q, uint64_t nan_key,
                       const uint64_t* __restrict__ tkey, size_t m, double w, uint64_t* __restrict__ count, double* __restrict__ bound) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const size_t finite = lower_bound_key(key, q, nan_key);
    const size_t c = tkey[i] == nan_key ? q : lower_bound_key(key, finite, tkey[i] + 1) + (q - finite);
    count[i] = c;
    bound[i] = finite < q ? INFINITY : (c ? bound_at(prefix, c - 1, w) : 0.0);
}

// out[0] = the number of candidates NaN levels hold; out[1] = the first position (p order) whose bound exceeds eps, or q
__global__ void k_first_over(const uint64_t* __restrict__ key, const double* __restrict__ prefix, size_t q, uint64_t nan_key,
                             double w, double eps, uint64_t* __restrict__ out) {
    size_t lo = 0, hi = q;
    while (lo < hi) {
        const size_t mid = lo + (hi - lo) / 2;
        if (bound_at(prefix, mid, w) <= eps) lo = mid + 1; else hi = mid;
    }
    out[0] = q - lower_bound_key(key, q, nan_key);
    out[1] = lo;
}

// out[0] = the first position of the level that holds position j
__global__ void k_level_start(const uint64_t* __restrict__ key, size_t j, uint64_t* __restrict__ out) {
    out[0] = lower_bound_key(key, j, key[j]);
}

// The curve of one product: its candidates' level keys in p order and the prefix of sum_t S_t^2 along that order
struct Curve {
    bool f64 = true;
    double w = 1.0;
    size_t q = 0, n_levels = 0;
    uint64_t nan_key = 0;
    DevBuf<uint64_t> key;
    DevBuf<double> prefix;
    double value(uint64_t k) const { return f64 ? LevelKey<double>::value(k) : LevelKey<float>::value(k); }
    uint64_t tau_key(double tau) const {   // fl(tau * tau) in Treal, tau rounded to Treal first (build_tasks)
        if (f64) return LevelKey<double>::of(tau * tau);
        const float t = (float)tau;
        return LevelKey<float>::of(t * t);
    }
};

void validate(const Matrix& A, bool tA, const Matrix& B, bool tB, bool symm_square, bool updated, const char* fn) {
    const std::string f = std::string("hbsm_b200: ") + fn + ": ";
    if (symm_square) {
        if (&B != &A || tA || tB) throw Error(HBSM_E_ARG, f + "symm_square needs B = A and no transpose");
        if (A.sized && A.M != A.N) throw Error(HBSM_E_ARG, f + "symm_square needs a square A");
        check_spamm_operands(A, false, A, false, true);
    } else {
        check_spamm_operands(A, tA, B, tB, updated);
    }
}

void build_curve(const Matrix& A, bool tA, const Matrix& B, bool tB, bool symm_square, bool updated, Curve& cv) {
    ensure_engine();
    cv.f64 = A.dtype == HBSM_F64;
    cv.w = symm_square ? 2.0 : 1.0;
    cv.nan_key = cv.f64 ? LevelKey<double>::NAN_KEY : LevelKey<float>::NAN_KEY;
    // the operands the product reads: symm_square joins sym_expand(A) with its norms refreshed (hbsm_symm_square_spamm)
    Matrix S;
    const Matrix* a = &A;
    const Matrix* b = &B;
    if (symm_square) {
        sym_expand(A, S);
        update_norms(S);
        a = b = &S;
    }
    const void* an = a->norms.p;
    const void* bn = b->norms.p;
    DevBuf<char> fresh_a, fresh_b;   // updated = false: fresh norms in temporaries, the caches untouched (hbsm_spamm)
    if (!symm_square && !updated) {
        fresh_a.alloc(std::max<size_t>(A.L, 1) * A.esize());
        compute_leaf_norms(A, fresh_a.p);
        an = fresh_a.p;
        bn = an;
        if (&B != &A) {
            fresh_b.alloc(std::max<size_t>(B.L, 1) * B.esize());
            compute_leaf_norms(B, fresh_b.p);
            bn = fresh_b.p;
        }
    }
    DevBuf<uint64_t> begin;
    DevBuf<uint2> ab;
    size_t nct = 0;
    const size_t q = product_candidates(*a, symm_square ? false : tA, *b, symm_square ? false : tB, symm_square, begin, ab, &nct);
    cv.q = q;
    if (q == 0) return;

    // gamma = n u / (1 - n u), n = b^2 terms per nsq, u = Treal's unit roundoff (n u is exact); rounded so 1 - gamma is low
    const double nu = std::ldexp((double)A.b * (double)A.b, cv.f64 ? -53 : -24);
    const double gamma_up = std::nextafter(nu / (1.0 - nu), INFINITY);
    const double one_minus_gamma = std::max(std::nextafter(1.0 - gamma_up, 0.0), 0.0);
    cv.key.alloc(q);
    DevBuf<uint32_t> order(q);
    DevBuf<double> s(q);
    if (cv.f64)
        HB_LAUNCH(k_cand_levels<double>, blocks_for(q, 256), 256, 0, ab.p, q, (const double*)an, (const double*)bn, one_minus_gamma,
                  cv.key.p, order.p, s.p);
    else
        HB_LAUNCH(k_cand_levels<float>, blocks_for(q, 256), 256, 0, ab.p, q, (const float*)an, (const float*)bn, one_minus_gamma,
                  cv.key.p, order.p, s.p);
    ab.release();
    radix_sort_pairs(cv.key.p, order.p, q, cv.f64 ? LevelKey<double>::BITS : LevelKey<float>::BITS);   // stable: p order

    DevBuf<double> delta(q);
    {
        DevBuf<uint32_t> tile(q), by_tile(q);
        DevBuf<uint64_t> tkey(q);
        HB_LAUNCH(k_tile_of, blocks_for(nct, 256), 256, 0, begin.p, nct, tile.p);
        HB_LAUNCH(k_tile_keys, blocks_for(q, 256), 256, 0, order.p, tile.p, q, tkey.p, by_tile.p);
        int tbits = 1;
        while (tbits < 64 && (1ull << tbits) < (uint64_t)nct) ++tbits;
        radix_sort_pairs(tkey.p, by_tile.p, q, tbits);   // stable: (C tile, p) order
        HB_LAUNCH(k_tile_deltas, blocks_for(nct, 128), 128, 0, begin.p, nct, by_tile.p, s.p, delta.p);
    }
    s.release();
    begin.release();

    cv.prefix.alloc(q);
    const size_t nb = (q + PS_TILE - 1) / PS_TILE;
    DevBuf<double> start(nb);
    HB_LAUNCH(k_prefix_local, (unsigned)nb, PS_THREADS, 0, order.p, delta.p, q, cv.prefix.p, start.p);
    HB_LAUNCH(k_prefix_blocks, 1, 1, 0, start.p, nb);
    HB_LAUNCH(k_prefix_add, blocks_for(q, 256), 256, 0, cv.prefix.p, q, start.p);

    DevBuf<uint32_t> head(q);
    HB_LAUNCH(k_level_heads, blocks_for(q, 256), 256, 0, cv.key.p, q, head.p);
    DevBuf<uint64_t> pos;
    cv.n_levels = scan_flags(head, q, pos);
}

// a tau whose fl(tau * tau) in Treal (tau rounded to Treal first) lies in [v, next) -- next absent at the top level --
// among sqrt(v) and its neighbours; NaN when none does (squares do not hit every value)
double tau_for_level(bool f64, double v, bool has_next, double next) {
    auto sq = [&](double t) {
        if (f64) return t * t;
        const float f = (float)t;
        return (double)(f * f);
    };
    auto step = [&](double t, double dir) { return f64 ? std::nextafter(t, dir) : (double)std::nextafterf((float)t, (float)dir); };
    const double t0 = f64 ? std::sqrt(v) : (double)(float)std::sqrt(v);
    double up = t0, dn = t0;
    for (int k = 0; k < 4; ++k) {
        for (double t : {up, dn})
            if (t >= 0.0 && sq(t) >= v && (!has_next || sq(t) < next)) return t;
        up = step(up, INFINITY);
        dn = step(dn, 0.0);
    }
    return NAN;
}

void eval_taus(const Curve& cv, size_t n, const double* taus, double* bounds, size_t* n_skipped) {
    std::vector<uint64_t> tk(n), cnt(n);
    for (size_t i = 0; i < n; ++i) tk[i] = cv.tau_key(taus[i]);
    DevBuf<uint64_t> dk(n), dc(n);
    DevBuf<double> db(n);
    dk.upload(tk.data(), n);
    HB_LAUNCH(k_eval, blocks_for(n, 128), 128, 0, cv.key.p, cv.prefix.p, cv.q, cv.nan_key, dk.p, n, cv.w, dc.p, db.p);
    dc.download(cnt.data(), n);
    db.download(bounds, n);
    sync_stream();
    if (n_skipped)
        for (size_t i = 0; i < n; ++i) n_skipped[i] = (size_t)cnt[i];
}

}  // namespace

void spamm_error_bounds(const Matrix& A, bool tA, const Matrix& B, bool tB, bool symm_square, bool updated, size_t n,
                        const double* taus, double* bounds, size_t* n_skipped) {
    validate(A, tA, B, tB, symm_square, updated, "spamm_error_bounds");
    if (n > 0 && (!taus || !bounds)) throw Error(HBSM_E_ARG, "hbsm_b200: spamm_error_bounds: null taus or bounds");
    for (size_t i = 0; i < n; ++i) {
        bounds[i] = 0.0;
        if (n_skipped) n_skipped[i] = 0;
    }
    if (n == 0) return;
    Curve cv;
    build_curve(A, tA, B, tB, symm_square, updated, cv);
    if (cv.q > 0) eval_taus(cv, n, taus, bounds, n_skipped);
}

// The highest level whose bound is <= eps, found on the non-decreasing curve by bisection, then a tau for it; a level no tau
// can single out gives way to the one below it, whose bound is smaller.
SpammTol spamm_tau_for_error(const Matrix& A, bool tA, const Matrix& B, bool tB, bool symm_square, bool updated, double eps) {
    if (!(eps >= 0.0) || std::isinf(eps))
        throw Error(HBSM_E_ARG, "hbsm_b200: spamm_tau_for_error: eps must be >= 0 and finite");
    validate(A, tA, B, tB, symm_square, updated, "spamm_tau_for_error");
    SpammTol r{};
    r.level = -1.0;
    Curve cv;
    build_curve(A, tA, B, tB, symm_square, updated, cv);
    r.n_candidates = cv.q;
    r.n_levels = cv.n_levels;
    if (cv.q == 0) return r;
    DevBuf<uint64_t> out(2);
    HB_LAUNCH(k_first_over, 1, 1, 0, cv.key.p, cv.prefix.p, cv.q, cv.nan_key, cv.w, eps, out.p);
    auto o = read_scalars(out.p, out.p + 1);
    if (o.first > 0) throw Error(HBSM_E_ARG, "hbsm_b200: spamm_tau_for_error: a leaf pair has a NaN level, every bound is +Inf");
    auto level_start = [&](size_t j) {
        HB_LAUNCH(k_level_start, 1, 1, 0, cv.key.p, j, out.p);
        return (size_t)read_scalars(out.p, nullptr).first;
    };
    size_t e = (size_t)o.second;   // the skipped candidates: positions [0, e) of the p order, e at a level boundary
    if (e < cv.q) e = level_start(e);
    while (e > 0) {
        const auto k = read_scalars(cv.key.p + e - 1, e < cv.q ? cv.key.p + e : nullptr);
        const double v = cv.value(k.first);
        const double t = tau_for_level(cv.f64, v, e < cv.q, e < cv.q ? cv.value(k.second) : 0.0);
        if (!std::isnan(t)) {
            r.tau = t;
            r.level = v;
            break;
        }
        e = level_start(e - 1);
    }
    eval_taus(cv, 1, &r.tau, &r.bound, &r.n_skipped);
    // tau = 0 still skips the pairs whose level is 0; their bound exceeds eps only when a norm product underflowed
    if (r.bound > eps)
        throw Error(HBSM_E_ARG, "hbsm_b200: spamm_tau_for_error: no tau meets eps (leaf pairs whose norm product underflows to 0 "
                                "are skipped at every tau)");
    return r;
}

}  // namespace hbsm_b200

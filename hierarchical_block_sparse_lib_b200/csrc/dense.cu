// dense.cu -- block-sparse matrix times dense multivector, Y = alpha*op(A)*X + beta*Y, and the Lanczos spectral-norm
// estimate built on it.  X (K x m) and Y (M x m) are dense column-major arrays in A's dtype with leading dimensions
// ldx >= K, ldy >= M.  op(A) is A (HBSM_OP_N), A^T (HBSM_OP_T) or triu(A) + striu(A)^T (HBSM_OP_SYM_UPPER, the symmetric
// storage of sym_expand / symm_*; tiles below the diagonal and the strict lower part of diagonal tiles are ignored).
//
// Kernel (k_dense): C-stationary.  A work unit is (block row r of Y, column chunk of MC columns of X and Y); a persistent
// grid claims units from an atomic counter.  The CTA that owns a unit walks the tiles of op(A)'s block row r in a fixed
// order -- the row line r of A for N, the column line r (tiles used transposed) for T, and for SYM_UPPER the column line
// r's tiles (k, r), k < r, transposed, then the diagonal tile, then the row line r's tiles (r, k), k > r -- and keeps the
// b x MC accumulators of the unit on chip, so every tile crosses HBM once per column chunk and Y is written once, with no
// atomics on data.  Tiles stream through a 4-stage cp.async ring in chunks of KL contraction indices (the whole tile when it
// takes at most DN_CHUNK_BYTES, else the largest multiple of 8 that does and whose ring fits the shared memory), together
// with the KL x MC slab of X they multiply; the copies are element-wise, so any leaf size up to 256 works and X / Y rows
// outside the matrix are never touched.  The diagonal tile of SYM_UPPER is applied in
// two masked passes (as stored on i <= l, transposed on i > l); the second pass reads the tile from L2.
// fp64 multiplies with DMMA (mma.sync m8n8k4), fp32 with FFMA.
#include "gemm_common.cuh"
#include <cfloat>
#include <cmath>

namespace hbsm_b200 {
namespace {

constexpr int DN_THREADS = 256;
constexpr int DN_NST = 4;                    // cp.async ring stages
constexpr int DN_CHUNK_BYTES = 40 * 1024;    // most tile bytes per stage, in either layout (a whole 64-leaf in both dtypes)

template <typename T>
struct DenseArgs {
    const T* tiles;
    const uint32_t *rptr, *rother, *rtile;   // row lines of A (N, SYM_UPPER)
    const uint32_t *cptr, *cother, *ctile;   // column lines of A (T, SYM_UPPER)
    const T* X;
    T* Y;
    long long ldx, ldy;
    int b, Mop, K, m, op;
    int n_brows, n_units;
    int KL, nchunk, KLP;     // contraction indices per stage, stages per tile, KL rounded up to 4
    int SA_N, SA_T, MCP;     // shared-memory strides: A chunk as stored, A chunk transposed, X slab row
    int a_elems, stage_elems;
    T alpha, beta;
    unsigned* counter;
};

// shared-memory strides that make the fragment loads conflict-free: fp64 (DMMA, 4 x 4 index patches per half warp) wants a
// stride of 4 mod 16 doubles, fp32 (one row per lane) an odd stride
template <typename T> __host__ __device__ inline int pad_stride(int x);
template <> __host__ __device__ inline int pad_stride<double>(int x) { return x + (((4 - x) % 16) + 16) % 16; }
template <> __host__ __device__ inline int pad_stride<float>(int x) { return x | 1; }

template <typename T>
__device__ __forceinline__ void cp_async_elem(T* dst, const T* src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(smem_u32(dst)), "l"(src), "n"((int)sizeof(T)) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// e = tid, tid + 256, ... < total over a 2-D range with `inner` fastest: f(inner index, outer index) without a division
// per element
template <typename F>
__device__ __forceinline__ void for_2d(int inner, int total, F&& f) {
    int a = (int)threadIdx.x % inner, o = (int)threadIdx.x / inner;
    const int da = DN_THREADS % inner, dout = DN_THREADS / inner;
    for (int e = threadIdx.x; e < total; e += DN_THREADS) {
        f(a, o);
        a += da;
        o += dout;
        if (a >= inner) { a -= inner; ++o; }
    }
}

// the walk of one block row: column-line entries [c_lo, c_hi) (used transposed), then row-line entries [r_lo, r_hi) (used
// as stored); under SYM_UPPER a leading diagonal row entry (diag = 1) is applied twice, masked
struct Walk { uint32_t c_lo, c_hi, r_lo, r_hi, diag; };
struct Step { uint32_t tile, k; int trans, mask; };   // mask 1: keep i <= l, 2: keep i > l (i, l: row / contraction in the tile)

__device__ __forceinline__ uint32_t lower_bound_u32(const uint32_t* v, uint32_t lo, uint32_t hi, uint32_t x) {
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (v[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

template <typename T>
__device__ __forceinline__ Walk make_walk(const DenseArgs<T>& g, uint32_t r) {
    Walk w{0, 0, 0, 0, 0};
    if (g.op == HBSM_OP_N) {
        w.r_lo = g.rptr[r]; w.r_hi = g.rptr[r + 1];
    } else if (g.op == HBSM_OP_T) {
        w.c_lo = g.cptr[r]; w.c_hi = g.cptr[r + 1];
    } else {
        w.c_lo = g.cptr[r];
        w.c_hi = lower_bound_u32(g.cother, w.c_lo, g.cptr[r + 1], r);                 // (k, r), k < r
        w.r_hi = g.rptr[r + 1];
        w.r_lo = lower_bound_u32(g.rother, g.rptr[r], w.r_hi, r);                     // (r, k), k >= r
        w.diag = (w.r_lo < w.r_hi && g.rother[w.r_lo] == r) ? 1u : 0u;
    }
    return w;
}
__device__ __forceinline__ int walk_steps(const Walk& w) { return (int)(w.c_hi - w.c_lo + w.r_hi - w.r_lo + w.diag); }

template <typename T>
__device__ __forceinline__ Step step_at(const DenseArgs<T>& g, const Walk& w, int s) {
    const int nc = (int)(w.c_hi - w.c_lo);
    if (s < nc) return Step{g.ctile[w.c_lo + s], g.cother[w.c_lo + s], 1, 0};
    s -= nc;
    if (w.diag) {
        if (s < 2) return Step{g.rtile[w.r_lo], g.rother[w.r_lo], s, s + 1};
        s -= 1;
    }
    return Step{g.rtile[w.r_lo + s], g.rother[w.r_lo + s], 0, 0};
}

// stage one item (chunk c of step s): the chunk of the tile and the KLP x MC slab of X it multiplies (zeros outside X)
template <typename T, int MC>
__device__ __forceinline__ void issue_item(const DenseArgs<T>& g, const Step& st, int c, T* As, int c0) {
    const int b = g.b, l0 = c * g.KL, nl = min(g.KL, b - l0);
    const T* tile = g.tiles + (size_t)st.tile * (size_t)b * (size_t)b;
    if (!st.trans)   // tile columns l0 .. l0+nl, contiguous: As[i + l*SA_N]
        for_2d(b, nl * b, [&](int i, int l) { cp_async_elem(As + i + l * g.SA_N, tile + (size_t)(l0 + l) * b + i); });
    else             // tile rows l0 .. l0+nl of every column i: As[l + i*SA_T]
        for_2d(nl, nl * b, [&](int l, int i) { cp_async_elem(As + l + i * g.SA_T, tile + (size_t)i * b + l0 + l); });
    T* Xs = As + g.a_elems;
    const long long row0 = (long long)st.k * b + l0;
    for_2d(g.KLP, g.KLP * MC, [&](int l, int j) {
        T* d = Xs + l * g.MCP + j;
        const long long row = row0 + l;
        const int col = c0 + j;
        if (l < nl && row < g.K && col < g.m) cp_async_elem(d, g.X + row + (long long)col * g.ldx);
        else *d = (T)0;
    });
}

// element (i, l) of op(tile) from a staged chunk (l relative to the chunk, la absolute); 0 outside the tile or the mask
template <typename T>
__device__ __forceinline__ T chunk_elem(const DenseArgs<T>& g, const T* As, const Step& st, int i, int l, int la, int nl) {
    const bool ok = i < g.b && l < nl && (st.mask == 0 || (st.mask == 1 ? i <= la : i > la));
    return ok ? (st.trans ? As[l + i * g.SA_T] : As[i + l * g.SA_N]) : (T)0;
}

// Per-thread accumulators and the per-dtype inner product of one staged chunk.
//   fp64: warps own m-fragments (8 rows) round-robin, G = min(8, ceil(b/8)) of them at a time, and the remaining 8/G warp
//         groups split the contraction; each warp keeps all MC/8 n-fragments of its rows.
//   fp32: thread t owns row t % RP (RP = b rounded up to a power of two) and every KS = 256/RP-th contraction index.
template <typename T, int MC> struct Core;

template <int MC>
struct Core<double, MC> {
    static constexpr int NF = MC / 8, MFW = 4;   // n-fragments, m-fragments per warp (b <= 256)
    double acc[MFW][NF][2];
    int nmf, G, KS, fg, ks;
    bool active;
    __device__ void init(int b) {
        nmf = (b + 7) / 8;
        G = nmf < 8 ? nmf : 8;
        KS = 8 / G;
        const int w = threadIdx.x >> 5;
        fg = w % G; ks = w / G;
        active = ks < KS;
    }
    __device__ void zero() {
#pragma unroll
        for (int t = 0; t < MFW; ++t)
#pragma unroll
            for (int n = 0; n < NF; ++n) acc[t][n][0] = acc[t][n][1] = 0.0;
    }
    __device__ void run(const DenseArgs<double>& g, const double* As, const Step& st, int l0, int nl) {
        if (!active) return;
        const int lane = threadIdx.x & 31, lr = lane & 3, lc = lane >> 2;
        const double* Xs = As + g.a_elems;
        for (int kk = ks * 4; kk < nl; kk += 4 * KS) {
            const int l = kk + lr;
            double x[NF];
#pragma unroll
            for (int n = 0; n < NF; ++n) x[n] = Xs[l * g.MCP + n * 8 + lc];
#pragma unroll
            for (int t = 0; t < MFW; ++t) {
                const int mf = fg + t * G;
                if (mf < nmf) {
                    const double a = chunk_elem(g, As, st, mf * 8 + lc, l, l0 + l, nl);
#pragma unroll
                    for (int n = 0; n < NF; ++n) dmma884(acc[t][n][0], acc[t][n][1], a, x[n]);
                }
            }
        }
    }
    static __host__ __device__ int rows_padded(int b) { return (b + 7) / 8 * 8; }
    static __host__ __device__ int ksplit(int b) { const int nmf = (b + 7) / 8; return 8 / (nmf < 8 ? nmf : 8); }
    // partial sums -> P[(ks * MC + col) * BP + row]
    __device__ void store(double* P, int BP) const {
        if (!active) return;
        const int lane = threadIdx.x & 31;
#pragma unroll
        for (int t = 0; t < MFW; ++t) {
            const int mf = fg + t * G;
            if (mf < nmf)
#pragma unroll
                for (int n = 0; n < NF; ++n)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int row = mf * 8 + (lane >> 2), col = n * 8 + 2 * (lane & 3) + e;
                        P[(size_t)(ks * MC + col) * BP + row] = acc[t][n][e];
                    }
        }
    }
};

template <int MC>
struct Core<float, MC> {
    float acc[MC];
    int RP, KS, i, ks;
    static __host__ __device__ int rp_of(int b) { int r = 1; while (r < b) r <<= 1; return r; }
    __device__ void init(int b) {
        RP = rp_of(b);
        KS = DN_THREADS / RP;
        i = threadIdx.x & (RP - 1);
        ks = threadIdx.x / RP;
    }
    __device__ void zero() {
#pragma unroll
        for (int j = 0; j < MC; ++j) acc[j] = 0.f;
    }
    __device__ void run(const DenseArgs<float>& g, const float* As, const Step& st, int l0, int nl) {
        const float* Xs = As + g.a_elems;
        for (int l = ks; l < nl; l += KS) {
            const float a = chunk_elem(g, As, st, i, l, l0 + l, nl);
            const float4* xv = reinterpret_cast<const float4*>(Xs + l * g.MCP);
#pragma unroll
            for (int q = 0; q < MC / 4; ++q) {
                const float4 x = xv[q];
                acc[4 * q + 0] = fmaf(a, x.x, acc[4 * q + 0]);
                acc[4 * q + 1] = fmaf(a, x.y, acc[4 * q + 1]);
                acc[4 * q + 2] = fmaf(a, x.z, acc[4 * q + 2]);
                acc[4 * q + 3] = fmaf(a, x.w, acc[4 * q + 3]);
            }
        }
    }
    static __host__ __device__ int rows_padded(int b) { return rp_of(b); }
    static __host__ __device__ int ksplit(int b) { return DN_THREADS / rp_of(b); }
    __device__ void store(float* P, int BP) const {
#pragma unroll
        for (int j = 0; j < MC; ++j) P[(size_t)(ks * MC + j) * BP + i] = acc[j];
    }
};

template <typename T, int MC>
__global__ void __launch_bounds__(DN_THREADS) k_dense(const DenseArgs<T> g) {
    extern __shared__ __align__(16) unsigned char dn_smem[];
    T* ring = reinterpret_cast<T*>(dn_smem);
    __shared__ unsigned s_unit;
    __shared__ Walk s_walk;
    Core<T, MC> core;
    core.init(g.b);
    const int BP = Core<T, MC>::rows_padded(g.b), KS = Core<T, MC>::ksplit(g.b);
    for (;;) {
        if (threadIdx.x == 0) s_unit = atomicAdd(g.counter, 1u);   // scheduler only: data is never combined atomically
        __syncthreads();
        const unsigned unit = s_unit;
        if (unit >= (unsigned)g.n_units) break;
        const uint32_t r = unit % (unsigned)g.n_brows;
        const int c0 = (int)(unit / (unsigned)g.n_brows) * MC;
        if (threadIdx.x == 0) s_walk = make_walk(g, r);
        __syncthreads();
        const Walk w = s_walk;
        const int n_items = walk_steps(w) * g.nchunk;
        core.zero();
#pragma unroll
        for (int q = 0; q < DN_NST - 1; ++q) {
            if (q < n_items) issue_item<T, MC>(g, step_at(g, w, q / g.nchunk), q % g.nchunk, ring + q * g.stage_elems, c0);
            cp_async_commit();
        }
        for (int q = 0; q < n_items; ++q) {
            cp_async_wait<DN_NST - 2>();
            __syncthreads();
            const int c = q % g.nchunk, l0 = c * g.KL;
            core.run(g, ring + (q % DN_NST) * g.stage_elems, step_at(g, w, q / g.nchunk), l0, min(g.KL, g.b - l0));
            const int qn = q + DN_NST - 1;   // refills the stage consumed in the previous round
            if (qn < n_items) issue_item<T, MC>(g, step_at(g, w, qn / g.nchunk), qn % g.nchunk, ring + (qn % DN_NST) * g.stage_elems, c0);
            cp_async_commit();
        }
        cp_async_wait<0>();
        __syncthreads();
        // epilogue: partial sums through shared memory, added in a fixed order, then Y = alpha * sum + beta * Y
        core.store(ring, BP);
        __syncthreads();
        const int row0 = (int)r * g.b;
        const int nrows = min(g.b, g.Mop - row0), ncols = min(MC, g.m - c0);
        for_2d(nrows, nrows * ncols, [&](int i, int j) {
            T s = ring[(size_t)j * BP + i];
            for (int k = 1; k < KS; ++k) s += ring[(size_t)(k * MC + j) * BP + i];
            T* y = g.Y + (row0 + i) + (long long)(c0 + j) * g.ldy;
            *y = g.beta == (T)0 ? g.alpha * s : g.alpha * s + g.beta * *y;
        });
        __syncthreads();
    }
}

// ---- Lanczos helpers: fixed-grid, fixed-order reductions in double (bitwise reproducible) ----
constexpr int LZ_BLOCKS = 256;

__device__ __forceinline__ double block_sum(double v, double* red) {
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int k = 0; k < DN_THREADS / 32; ++k) s += red[k];
    __syncthreads();
    return s;
}

template <typename T>
__global__ void __launch_bounds__(DN_THREADS) k_lz_start(T* v, size_t n, uint64_t seed) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        v[i] = (T)((double)(splitmix64(seed ^ splitmix64(i)) >> 11) * (1.0 / 9007199254740992.0) - 0.5);
}

// part[blockIdx.x] = sum over this block's strided share of a[i] * b[i]
template <typename T>
__global__ void __launch_bounds__(DN_THREADS) k_lz_dot(const T* a, const T* b, size_t n, double* part) {
    __shared__ double red[DN_THREADS / 32];
    double s = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        s += (double)a[i] * (double)b[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) part[blockIdx.x] = s;
}

// w -= alpha * v + beta_prev * vp  (alpha from the device scalar), then the partial sums of |w|^2
template <typename T>
__global__ void __launch_bounds__(DN_THREADS) k_lz_update(T* w, const T* v, const T* vp, size_t n, const double* alpha,
                                                          double beta_prev, double* part) {
    __shared__ double red[DN_THREADS / 32];
    const T a = (T)*alpha, bp = (T)beta_prev;
    double s = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const T x = w[i] - a * v[i] - bp * vp[i];
        w[i] = x;
        s += (double)x * (double)x;
    }
    s = block_sum(s, red);
    if (threadIdx.x == 0) part[blockIdx.x] = s;
}

__global__ void __launch_bounds__(DN_THREADS) k_lz_finish(const double* part, int n, double* out) {
    __shared__ double red[DN_THREADS / 32];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += DN_THREADS) s += part[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) *out = s;
}

template <typename T>
__global__ void __launch_bounds__(DN_THREADS) k_lz_scale(T* dst, const T* src, size_t n, double s) {
    const T f = (T)s;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i] * f;
}

// Eigenvalues of the symmetric tridiagonal matrix (d, e) -- d[0..n), e[i] couples i and i+1 -- by implicit QL with
// Wilkinson shifts; z (in: e_{n-1}) receives the last components of the eigenvectors.  d, z come back in ascending order.
void tridiag_eig(int n, std::vector<double>& d, std::vector<double> e, std::vector<double>& z) {
    z.assign(n, 0.0);
    z[n - 1] = 1.0;
    e.resize(n, 0.0);
    e[n - 1] = 0.0;
    for (int l = 0; l < n; ++l) {
        for (int iter = 0;; ++iter) {
            int m = l;
            for (; m < n - 1; ++m)
                if (std::fabs(e[m]) <= DBL_EPSILON * (std::fabs(d[m]) + std::fabs(d[m + 1]))) break;
            if (m == l) break;
            if (iter == 100) throw Error(HBSM_E_RUNTIME, "hbsm_b200: spectral_norm: tridiagonal QL did not converge");
            double g = (d[l + 1] - d[l]) / (2.0 * e[l]);
            double r = std::hypot(g, 1.0);
            g = d[m] - d[l] + e[l] / (g + std::copysign(r, g));   // shift: the eigenvalue of the leading 2 x 2 nearer d[l]
            double s = 1.0, c = 1.0, p = 0.0;
            bool deflated = false;
            for (int i = m - 1; i >= l; --i) {   // chase the bulge from the bottom of the block up to l
                const double f = s * e[i], bb = c * e[i];
                r = std::hypot(f, g);
                e[i + 1] = r;
                if (r == 0.0) {   // underflow: the block splits at i + 1
                    d[i + 1] -= p;
                    e[m] = 0.0;
                    deflated = true;
                    break;
                }
                s = f / r;
                c = g / r;
                g = d[i + 1] - p;
                r = (d[i] - g) * s + 2.0 * c * bb;
                p = s * r;
                d[i + 1] = g + p;
                g = c * r - bb;
                const double zf = z[i + 1];
                z[i + 1] = s * z[i] + c * zf;
                z[i] = c * z[i] - s * zf;
            }
            if (deflated) continue;
            d[l] -= p;
            e[l] = g;
            e[m] = 0.0;
        }
    }
    std::vector<int> ord(n);
    for (int i = 0; i < n; ++i) ord[i] = i;
    std::sort(ord.begin(), ord.end(), [&](int a, int b) { return d[a] < d[b] || (d[a] == d[b] && a < b); });
    std::vector<double> d2(n), z2(n);
    for (int i = 0; i < n; ++i) { d2[i] = d[ord[i]]; z2[i] = z[ord[i]]; }
    d.swap(d2);
    z.swap(z2);
}

struct DenseOp {   // op(A) of a validated call
    int Mop, K;
};

DenseOp dense_shape(const Matrix& A, int op) {
    if (!A.sized) throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: A is empty (not sized)");
    if (op != HBSM_OP_N && op != HBSM_OP_T && op != HBSM_OP_SYM_UPPER)
        throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: unknown op " + std::to_string(op));
    if (op == HBSM_OP_SYM_UPPER && A.M != A.N) throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: SYM_UPPER needs a square A");
    if (A.b > 256) throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: leaf sizes above 256 have no kernel");
    return op == HBSM_OP_T ? DenseOp{A.N, A.M} : DenseOp{A.M, A.N};
}

LineView line_view(const LineIndex& ix) { return LineView{ix.ptr.p, ix.other.p, ix.tile.p}; }

OpView view_for(const Matrix& A, int op) {   // A's own line indices that op walks
    OpView v;
    if (op != HBSM_OP_T) v.row = line_view(line_index(A, false));
    if (op != HBSM_OP_N) v.col = line_view(line_index(A, true));
    return v;
}

template <typename T, int MC>
void launch_dense_mc(const Matrix& A, const OpView& v, int op, int m, const T* X, long long ldx, T* Y, long long ldy, double alpha,
                     double beta) {
    Engine& e = engine();
    const DenseOp s = dense_shape(A, op);
    DenseArgs<T> g{};
    g.tiles = (const T*)A.tiles.p;
    g.rptr = v.row.ptr; g.rother = v.row.other; g.rtile = v.row.tile;
    g.cptr = v.col.ptr; g.cother = v.col.other; g.ctile = v.col.tile;
    g.X = X; g.Y = Y; g.ldx = ldx; g.ldy = ldy;
    g.b = A.b; g.Mop = s.Mop; g.K = s.K; g.m = m; g.op = op;
    g.n_brows = (s.Mop + A.b - 1) / A.b;
    const int n_cchunks = (m + MC - 1) / MC;
    if ((long long)g.n_brows * n_cchunks > INT32_MAX) throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: too many work units");
    g.n_units = g.n_brows * n_cchunks;
    const int b = A.b;
    const int align = 16 / (int)sizeof(T);
    g.SA_N = pad_stride<T>(b);
    g.MCP = sizeof(T) == 8 ? MC + 4 : MC;
    g.alpha = (T)alpha;
    g.beta = (T)beta;
    const size_t part = (size_t)Core<T, MC>::ksplit(b) * MC * Core<T, MC>::rows_padded(b) * sizeof(T);
    auto geometry = [&](int KL) {   // stage layout for KL contraction indices per stage; returns the dynamic shared memory
        g.KL = KL;
        g.nchunk = (b + KL - 1) / KL;
        g.KLP = (KL + 3) / 4 * 4;
        g.SA_T = pad_stride<T>(KL);
        g.a_elems = (std::max(KL * g.SA_N, b * g.SA_T) + align - 1) / align * align;   // room for either layout
        g.stage_elems = (g.a_elems + g.KLP * g.MCP + align - 1) / align * align;
        return std::max((size_t)DN_NST * g.stage_elems * sizeof(T), part);
    };
    // KL = b, or the largest multiple of 8 below it, whose chunk takes at most DN_CHUNK_BYTES in the larger of its two
    // layouts and whose whole ring (chunks and X slabs) fits the per-block opt-in shared memory
    int optin = 0;
    HB_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, e.device));
    size_t smem = 0;
    for (int KL = b;; KL = (KL - 1) & ~7) {
        smem = geometry(KL);
        if ((g.a_elems * sizeof(T) <= (size_t)DN_CHUNK_BYTES && smem <= (size_t)optin) || KL <= 8) break;
    }
    if (smem > (size_t)optin)
        throw Error(HBSM_E_CUDA, "hbsm_b200: multiply_dense: " + std::to_string(smem) + " B of shared memory needed, the device offers " +
                                     std::to_string(optin));
    auto kfn = k_dense<T, MC>;
    HB_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    HB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kfn, DN_THREADS, smem));
    const unsigned grid = (unsigned)std::max(1, std::min(g.n_units, std::max(per_sm, 1) * e.sm_count));
    DevBuf<unsigned> counter(1);
    counter.zero();
    g.counter = counter.p;
    HB_LAUNCH(kfn, grid, DN_THREADS, smem, g);
}

template <typename T>
void launch_dense(const Matrix& A, const OpView& v, int op, int m, const T* X, long long ldx, T* Y, long long ldy, double alpha,
                  double beta) {
    if (m <= 8) launch_dense_mc<T, 8>(A, v, op, m, X, ldx, Y, ldy, alpha, beta);
    else if (m <= 16) launch_dense_mc<T, 16>(A, v, op, m, X, ldx, Y, ldy, alpha, beta);
    else launch_dense_mc<T, 32>(A, v, op, m, X, ldx, Y, ldy, alpha, beta);
}

// Decision tests of one Lanczos step (decision mode).  theta_lo / theta_hi: extreme Ritz values; r_lo / r_hi: the residual
// bounds of their pairs (0 on breakdown: the Ritz values are exact).  For the symmetric operator the Ritz values lie inside
// [lambda_min, lambda_max], so |theta| > eps proves ||op|| > eps.  Acceptance needs theta_hi + r_hi <= eps and
// theta_lo - r_lo >= -eps with the extreme pairs converged (r <= conv * max|theta|): a residual bound only places an
// eigenvalue near theta, and before the pair has converged a larger eigenvalue may not have entered the Krylov space yet.
// For E^T E the same holds with eps^2 and theta_hi alone.  Returns true when decided.
bool decide(LanczosDecision& d, bool symmetric_upper, double theta_lo, double theta_hi, double r_lo, double r_hi, double conv) {
    const double scale = std::max(std::fabs(theta_lo), std::fabs(theta_hi));
    if (symmetric_upper) {
        const double up = std::max(theta_hi + r_hi, r_lo - theta_lo);
        d.bound = up;
        if (scale > d.eps) { d.feasible = false; return true; }
        if (up <= d.eps && r_hi <= conv * scale && r_lo <= conv * scale) { d.feasible = true; return true; }
    } else {
        const double e2 = d.eps * d.eps;
        d.bound = std::sqrt(std::max(theta_hi + r_hi, 0.0));
        if (theta_hi > e2) { d.feasible = false; return true; }
        if (theta_hi + r_hi <= e2 && r_hi <= conv * scale) { d.feasible = true; return true; }
    }
    return false;
}

}  // namespace

void validate_dense(const Matrix& A, int op, int m, long long ldx, long long ldy, const void* X, const void* Y) {
    const DenseOp s = dense_shape(A, op);
    if (m < 0) throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: m < 0");
    if (ldx < std::max(1, s.K)) throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: ldx < max(1, rows of X)");
    if (ldy < std::max(1, s.Mop)) throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: ldy < max(1, rows of Y)");
    if (m > 0 && ((s.K > 0 && !X) || (s.Mop > 0 && !Y))) throw Error(HBSM_E_ARG, "hbsm_b200: multiply_dense: null X or Y");
}


// Y (device) = alpha * op(A) * X + beta * Y on the engine stream
void dense_product_device(const Matrix& A, int op, int m, const void* d_X, long long ldx, void* d_Y, long long ldy, double alpha,
                          double beta) {
    validate_dense(A, op, m, ldx, ldy, d_X, d_Y);
    const DenseOp s = dense_shape(A, op);
    if (m == 0 || s.Mop == 0) return;
    ensure_engine();
    const OpView v = view_for(A, op);
    if (A.dtype == HBSM_F64) launch_dense<double>(A, v, op, m, (const double*)d_X, ldx, (double*)d_Y, ldy, alpha, beta);
    else launch_dense<float>(A, v, op, m, (const float*)d_X, ldx, (float*)d_Y, ldy, alpha, beta);
}

void dense_product_host(const Matrix& A, int op, int m, const void* X, long long ldx, void* Y, long long ldy, double alpha,
                        double beta) {
    validate_dense(A, op, m, ldx, ldy, X, Y);
    const DenseOp s = dense_shape(A, op);
    if (m == 0 || s.Mop == 0) return;
    ensure_engine();
    const size_t es = A.esize();
    const size_t kx = (size_t)std::max(1, s.K);
    DevBuf<char> dX(kx * m * es), dY((size_t)s.Mop * m * es);
    Engine& e = engine();
    if (s.K > 0)
        HB_CUDA(cudaMemcpy2DAsync(dX.p, s.K * es, X, (size_t)ldx * es, s.K * es, m, cudaMemcpyHostToDevice, e.stream));
    if (beta != 0.0)   // beta == 0 never reads Y
        HB_CUDA(cudaMemcpy2DAsync(dY.p, s.Mop * es, Y, (size_t)ldy * es, s.Mop * es, m, cudaMemcpyHostToDevice, e.stream));
    dense_product_device(A, op, m, dX.p, (long long)kx, dY.p, s.Mop, alpha, beta);
    HB_CUDA(cudaMemcpy2DAsync(Y, (size_t)ldy * es, dY.p, s.Mop * es, s.Mop * es, m, cudaMemcpyDeviceToHost, e.stream));
    sync_stream();
}

// Plain Lanczos on S = triu(A) + striu(A)^T (symmetric_upper) or on A^T A, without reorthogonalisation: loss of
// orthogonality only adds copies of converged extreme Ritz values.  Stops when the residual bound |beta_j s_j(last)| of the
// extreme Ritz pair (for S: of both extreme pairs) is <= rel_tol * max|theta|, on breakdown (beta_j at round-off level:
// the Krylov space is invariant and the Ritz values are exact), or after max_iter steps (at most the dimension).
SpectralResult spectral_norm(const Matrix& A, bool symmetric_upper, int max_iter, double rel_tol) {
    if (!A.sized) throw Error(HBSM_E_ARG, "hbsm_b200: spectral_norm: A is empty (not sized)");
    if (symmetric_upper && A.M != A.N) throw Error(HBSM_E_ARG, "hbsm_b200: spectral_norm: symmetric_upper needs a square A");
    if (max_iter < 1) throw Error(HBSM_E_ARG, "hbsm_b200: spectral_norm: max_iter < 1");
    if (!(rel_tol > 0.0)) throw Error(HBSM_E_ARG, "hbsm_b200: spectral_norm: rel_tol must be > 0");
    if (A.b > 256) throw Error(HBSM_E_ARG, "hbsm_b200: spectral_norm: leaf sizes above 256 have no kernel");
    SpectralResult res{};
    if (A.L == 0 || A.M == 0 || A.N == 0) return res;
    ensure_engine();
    return lanczos(A, own_view(A), symmetric_upper, max_iter, rel_tol, nullptr);
}

OpView own_view(const Matrix& A) { return view_for(A, HBSM_OP_SYM_UPPER); }

// The Lanczos core of spectral_norm on any operator view.  In decision mode (dec != nullptr) the run stops when decide()
// settles ||op|| <= dec->eps (with the extreme pairs converged to rel_tol) or > dec->eps, on breakdown (decided with the exact
// Ritz values), or at max_iter / the dimension, where an undecided run counts as infeasible.
SpectralResult lanczos(const Matrix& A, const OpView& view, bool symmetric_upper, int max_iter, double rel_tol, LanczosDecision* dec) {
    SpectralResult res{};
    if (dec) { dec->feasible = false; dec->bound = 0.0; }
    const size_t n = (size_t)A.N, es = A.esize();
    DevBuf<char> V(n * es), P(n * es), W(n * es), tmp(symmetric_upper ? 1 : (size_t)A.M * es);
    DevBuf<double> part(LZ_BLOCKS), scal(2);
    P.zero();
    const double eps = A.dtype == HBSM_F64 ? DBL_EPSILON : (double)FLT_EPSILON;
    const unsigned grid = (unsigned)std::min<size_t>(LZ_BLOCKS, (n + DN_THREADS - 1) / DN_THREADS);
    char* v = V.p; char* vp = P.p;
    auto run = [&](auto z) {
        using T = decltype(z);
        auto dot = [&](const char* a, const char* b, double* out) {
            HB_LAUNCH(k_lz_dot<T>, grid, DN_THREADS, 0, (const T*)a, (const T*)b, n, part.p);
            HB_LAUNCH(k_lz_finish, 1, DN_THREADS, 0, part.p, (int)grid, out);
        };
        auto read2 = [&](double* h) {
            HB_CUDA(cudaMemcpyAsync(h, scal.p, 2 * sizeof(double), cudaMemcpyDeviceToHost, engine().stream));
            sync_stream();
        };
        double h[2];
        HB_LAUNCH(k_lz_start<T>, grid, DN_THREADS, 0, (T*)v, n, (uint64_t)0x5D4E3C2B1A09F8E7ull);
        dot(v, v, scal.p + 1);
        read2(h);
        HB_LAUNCH(k_lz_scale<T>, grid, DN_THREADS, 0, (T*)v, (const T*)v, n, 1.0 / std::sqrt(h[1]));
        std::vector<double> alpha, beta, theta, zl;
        double beta_prev = 0.0, tnorm = 0.0;
        for (int j = 0;; ++j) {
            if (symmetric_upper) {
                launch_dense<T>(A, view, HBSM_OP_SYM_UPPER, 1, (const T*)v, (long long)n, (T*)W.p, (long long)n, 1.0, 0.0);
            } else {
                launch_dense<T>(A, view, HBSM_OP_N, 1, (const T*)v, (long long)n, (T*)tmp.p, (long long)A.M, 1.0, 0.0);
                launch_dense<T>(A, view, HBSM_OP_T, 1, (const T*)tmp.p, (long long)A.M, (T*)W.p, (long long)n, 1.0, 0.0);
            }
            dot(v, W.p, scal.p);
            HB_LAUNCH(k_lz_update<T>, grid, DN_THREADS, 0, (T*)W.p, (const T*)v, (const T*)vp, n, scal.p, beta_prev, part.p);
            HB_LAUNCH(k_lz_finish, 1, DN_THREADS, 0, part.p, (int)grid, scal.p + 1);
            read2(h);
            const double bj = std::sqrt(h[1]);
            alpha.push_back(h[0]);
            tnorm = std::max(tnorm, std::fabs(h[0]) + beta_prev + bj);   // Gershgorin bound of the tridiagonal matrix
            theta = alpha;
            tridiag_eig((int)alpha.size(), theta, beta, zl);
            const int k = (int)theta.size();
            const double scale = std::max(std::fabs(theta[0]), std::fabs(theta[k - 1]));
            const double bound_hi = std::fabs(bj * zl[k - 1]), bound_lo = std::fabs(bj * zl[0]);
            res.n_iter = j + 1;
            const bool converged = bound_hi <= rel_tol * scale && (!symmetric_upper || bound_lo <= rel_tol * scale);
            const bool breakdown = bj <= 16.0 * std::sqrt((double)n) * eps * tnorm;
            const bool decided = dec && (breakdown ? decide(*dec, symmetric_upper, theta[0], theta[k - 1], 0.0, 0.0, rel_tol)
                                                   : decide(*dec, symmetric_upper, theta[0], theta[k - 1], bound_lo, bound_hi, rel_tol));
            if ((dec ? decided : converged) || breakdown || res.n_iter >= max_iter || (size_t)res.n_iter >= n) {
                res.lambda_min = theta[0];
                res.lambda_max = theta[k - 1];
                break;
            }
            beta.push_back(bj);
            HB_LAUNCH(k_lz_scale<T>, grid, DN_THREADS, 0, (T*)vp, (const T*)W.p, n, 1.0 / bj);   // v_{j+1} = w / beta_j
            std::swap(v, vp);
            beta_prev = bj;
        }
    };
    if (A.dtype == HBSM_F64) run(double{}); else run(float{});
    res.norm = symmetric_upper ? std::max(std::fabs(res.lambda_min), std::fabs(res.lambda_max)) : std::sqrt(std::max(res.lambda_max, 0.0));
    return res;
}

}  // namespace hbsm_b200

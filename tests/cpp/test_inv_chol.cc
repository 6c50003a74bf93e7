// test_inv_chol.cc -- runs the drop-in class's inv_chol (include/hbsm/HierarchicalBlockSparseMatrix.h) on matrices read
// from a file and writes the factors back; tests/test_gpu_inv_chol.py writes the inputs and checks the results against
// its reference, so the numerics live in one place.
//
// Usage: test_inv_chol IN OUT.  All values little-endian.
//   IN:  int32 n_cases, then per case: int32 dtype (0 = double, 1 = float), int32 b, int32 n, int64 nnz,
//        int32 rows[nnz], int32 cols[nnz], float64 vals[nnz]
//   OUT: per case: int64 get_n_blocks(Z), int64 gemm_kernel of the last product (hbsm_stage_times_last; -1 if none has
//        run in this process), int64 get_n_rows(Z), int64 get_n_cols(Z), int64 count, int32 rows[count],
//        int32 cols[count], float64 vals[count] (get_all_values)
#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>

#include "hbsm/hierarchical_block_sparse_lib.h"

template <class V>
static void get(std::FILE* f, V* p, size_t n) {
    if (n && std::fread(p, sizeof(V), n, f) != n) throw std::runtime_error("short input file");
}
template <class V>
static void put(std::FILE* f, const V* p, size_t n) {
    if (n && std::fwrite(p, sizeof(V), n, f) != n) throw std::runtime_error("short write");
}

template <class T>
static void run_case(int b, int n, const std::vector<int>& r, const std::vector<int>& c, const std::vector<double>& v, std::FILE* out) {
    typedef hbsm::HierarchicalBlockSparseMatrix<T> M;
    typename M::Params p;
    p.blocksize = b;
    M A, Z;
    A.set_params(p);
    A.resize(n, n);
    std::vector<T> tv(v.begin(), v.end());
    A.assign_from_vectors(r, c, tv);
    M::inv_chol(A, Z);
    hbsm_stage_times st;
    const int64_t kernel = hbsm_stage_times_last(&st) == HBSM_OK ? (int64_t)st.gemm_kernel : -1;
    std::vector<int> zr, zc;
    std::vector<T> zv;
    Z.get_all_values(zr, zc, zv);
    const int64_t head[5] = {(int64_t)Z.get_n_blocks(), kernel, (int64_t)Z.get_n_rows(), (int64_t)Z.get_n_cols(), (int64_t)zv.size()};
    std::vector<double> zd(zv.begin(), zv.end());
    put(out, head, 5);
    put(out, zr.data(), zr.size());
    put(out, zc.data(), zc.size());
    put(out, zd.data(), zd.size());
}

int main(int argc, char** argv) {
    if (argc != 3) { std::fprintf(stderr, "usage: %s IN OUT\n", argv[0]); return 2; }
    try {
        if (hbsm_init(0) != HBSM_OK) { std::fprintf(stderr, "hbsm_init: %s\n", hbsm_last_error()); return 2; }
        std::FILE* in = std::fopen(argv[1], "rb");
        std::FILE* out = std::fopen(argv[2], "wb");
        if (!in || !out) throw std::runtime_error("cannot open the input or the output file");
        int32_t n_cases = 0;
        get(in, &n_cases, 1);
        for (int k = 0; k < n_cases; ++k) {
            int32_t hd[3];
            int64_t nnz = 0;
            get(in, hd, 3);
            get(in, &nnz, 1);
            std::vector<int> r(nnz), c(nnz);
            std::vector<double> v(nnz);
            get(in, r.data(), nnz);
            get(in, c.data(), nnz);
            get(in, v.data(), nnz);
            if (hd[0] == 0) run_case<double>(hd[1], hd[2], r, c, v, out);
            else run_case<float>(hd[1], hd[2], r, c, v, out);
        }
        std::fclose(in);
        if (std::fclose(out) != 0) throw std::runtime_error("cannot write the output file");
        std::printf("test_inv_chol: %d cases\n", n_cases);
        return 0;
    } catch (const std::exception& e) {
        std::fprintf(stderr, "test_inv_chol: %s\n", e.what());
        return 1;
    }
}

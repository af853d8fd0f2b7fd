// cu_lanczos.h — host mirror of the reference's lanczosDecomp<T> (parallel-final/lib/cu_lanczos.h:30-108).
// The constructor does all the work, as in the reference: it uploads the CSR, normalises the start vector and runs the
// k-step Lanczos decomposition on the GPU through the C ABI (include/lz.h). Differences that follow from the B200 design:
//   * the basis Q never leaves the device (no per-step D2H copy, cu_lanczos.cu:126), so the `Q` member stays nullptr;
//     `get_basis(j, out)` fetches a vector on demand;
//   * `cuda == false` is refused: there is no CPU path in this library (the reference's CPU decompose() lives on as the
//     test oracle under oracle/);
//   * optional 5th/6th constructor arguments select full reorthogonalisation and the GPU.
#ifndef LZ_CU_LANCZOS_H
#define LZ_CU_LANCZOS_H

#include <cmath>
#include <cstdlib>
#include <iostream>
#include <string>
#include <vector>

#include "../../include/lz.h"
#include "adjMatrix.h"

template <typename T, typename U>
T norm(const T* v, U n) {  // cu_lanczos.h:18-24
  T s{0.0};
  for (U i = 0; i < n; i++) s += v[i] * v[i];
  return std::sqrt(s);
}

template <typename U, typename V> void check_ans(lanczosDecomp<U>&, lanczosDecomp<V>&);
template <typename U> void write_ans(std::string filename, lanczosDecomp<U>&);
template <typename T> class ritzPairs;

template <typename T>
class lanczosDecomp {
 private:
  adjMatrix& A;
  unsigned krylov_dim;
  T* alpha;           // diagonal of the tridiagonal matrix      [krylov]
  T* beta;            // sub-diagonal                              [krylov - 1]
  T* Q = nullptr;     // not materialised on the host (basis is device-resident)
  T* x;               // starting vector                           [n]
  T* ans;             // e^A x, filled by multOut                  [n]
  T x_norm;
  lz_ctx* ctx = nullptr;
  int reorth = LZ_REORTH_NONE;

  void cu_decompose();
  [[noreturn]] static void fail(const char* where) {
    std::cerr << where << ": " << lz_last_error() << '\n';
    std::abort();
  }

 public:
  lanczosDecomp() = delete;
  lanczosDecomp(adjMatrix& adj, const unsigned krylov, T* starting_vec, bool cuda, int reorth_mode = LZ_REORTH_NONE, int device = 0)
      : A{adj}, krylov_dim{krylov}, alpha(new T[krylov]), beta(new T[krylov > 1 ? krylov - 1 : 1]), x(new T[adj.get_n()]),
        ans(new T[adj.get_n()]), x_norm{norm(starting_vec, adj.get_n())}, reorth{reorth_mode} {
    for (unsigned i = 0; i < A.n; i++) x[i] = starting_vec[i];
    if (!cuda) {
      std::cerr << "lanczosDecomp: cuda=false requested, but this library has no CPU fallback "
                   "(the reference's serial decompose() is kept only as the test oracle)\n";
      std::abort();
    }
    if (lz_create(device, &ctx) != LZ_OK) fail("lanczosDecomp: lz_create");
    cu_decompose();
  }
  lanczosDecomp(lanczosDecomp&) = delete;
  lanczosDecomp& operator=(lanczosDecomp&) = delete;
  ~lanczosDecomp() { free_mem(); delete[] ans; ans = nullptr; }

  void free_mem() {  // cu_lanczos.h:78-86 (without its stdout chatter and its cudaFree of a host pointer)
    delete[] alpha; alpha = nullptr;
    delete[] beta; beta = nullptr;
    delete[] x; x = nullptr;
    if (ctx) { lz_destroy(ctx); ctx = nullptr; }
  }

  unsigned get_n() const { return A.get_n(); }
  unsigned get_krylov() const { return krylov_dim; }
  const T* get_alpha() const { return alpha; }
  const T* get_beta() const { return beta; }
  const T* get_ans_ptr() const { return ans; }
  void get_basis(unsigned j, T* out) const;
  // Centrality ranking (valid after multOut): the m largest entries of e^A x, descending, ties -> lower vertex id. Selected on
  // the device (lz_top_k); returns the number of pairs written. The reference has no ranking call — its users sort write_ans output.
  unsigned top_k(unsigned m, unsigned* idx_out, T* val_out) const {
    std::vector<double> v(m);
    uint32_t cnt = 0;
    static_assert(sizeof(unsigned) == sizeof(uint32_t), "32-bit vertex ids");
    if (lz_top_k(ctx, m, reinterpret_cast<uint32_t*>(idx_out), v.data(), &cnt) != LZ_OK) fail("lanczosDecomp: lz_top_k");
    for (unsigned i = 0; i < cnt; i++) val_out[i] = (T)v[i];
    return cnt;
  }
  lz_timings timings() const { lz_timings t{}; lz_timings_get(ctx, &t); return t; }

  friend class eigenDecomp<T>;
  friend class ritzPairs<T>;
  template <typename U> friend void multOut(lanczosDecomp<U>&, eigenDecomp<U>&, adjMatrix&, bool);
  template <typename U, typename V> friend void check_ans(lanczosDecomp<U>&, lanczosDecomp<V>&);
  template <typename U> friend void write_ans(std::string filename, lanczosDecomp<U>&);

  void check_ans(const T* analytic) const;   // lanczos.cu:69-84
};

// ---- implementation (double is the graded precision; float = fp32 basis on the device, fp64 arithmetic) ---------------
namespace lz_detail {
inline std::vector<double> widen(const float* p, size_t n) { return std::vector<double>(p, p + n); }
}

template <>
inline void lanczosDecomp<double>::cu_decompose() {
  if (lz_csr_upload(ctx, A.n, A.row_offset, A.col_idx) != LZ_OK) fail("lanczosDecomp: lz_csr_upload");
  if (lz_set_start_vector(ctx, x) != LZ_OK) fail("lanczosDecomp: lz_set_start_vector");
  if (lz_lanczos_run(ctx, krylov_dim, reorth) != LZ_OK) fail("lanczosDecomp: lz_lanczos_run");
  if (lz_get_tridiag(ctx, alpha, beta) != LZ_OK) fail("lanczosDecomp: lz_get_tridiag");
}
template <>
inline void lanczosDecomp<float>::cu_decompose() {
  // single precision maps to the fp32-basis mode of the library (V stored as floats, arithmetic fp64): it keeps the memory and
  // bandwidth saving that motivates the reference's float build (cu_lanczos.cu:144) without its 1e-6 error and nan hazards
  std::vector<double> xd = lz_detail::widen(x, A.n), a(krylov_dim), b(krylov_dim);
  if (lz_set_basis_precision(ctx, LZ_BASIS_F32) != LZ_OK) fail("lanczosDecomp: lz_set_basis_precision");
  if (lz_csr_upload(ctx, A.n, A.row_offset, A.col_idx) != LZ_OK) fail("lanczosDecomp: lz_csr_upload");
  if (lz_set_start_vector(ctx, xd.data()) != LZ_OK) fail("lanczosDecomp: lz_set_start_vector");
  if (lz_lanczos_run(ctx, krylov_dim, reorth) != LZ_OK) fail("lanczosDecomp: lz_lanczos_run");
  if (lz_get_tridiag(ctx, a.data(), b.data()) != LZ_OK) fail("lanczosDecomp: lz_get_tridiag");
  for (unsigned i = 0; i < krylov_dim; i++) alpha[i] = (float)a[i];
  for (unsigned i = 0; i + 1 < krylov_dim; i++) beta[i] = (float)b[i];
}
template <>
inline void lanczosDecomp<double>::get_basis(unsigned j, double* out) const {
  if (lz_get_basis(ctx, j, out) != LZ_OK) fail("lanczosDecomp: lz_get_basis");
}
template <>
inline void lanczosDecomp<float>::get_basis(unsigned j, float* out) const {
  std::vector<double> q(A.get_n());
  if (lz_get_basis(ctx, j, q.data()) != LZ_OK) fail("lanczosDecomp: lz_get_basis");
  for (unsigned i = 0; i < A.get_n(); i++) out[i] = (float)q[i];
}

template <typename T>
void lanczosDecomp<T>::check_ans(const T* analytic) const {
  const unsigned n = A.get_n();
  std::vector<double> diff(n);
  unsigned max_idx = 0;
  for (unsigned i = 0; i < n; i++) {
    diff[i] = std::abs((double)ans[i] - (double)analytic[i]);
    if (diff[i] > diff[max_idx]) max_idx = i;
  }
  std::cout << "\nMax difference of " << diff[max_idx] << " found at index\n\tlanczos[" << max_idx << "] \t\t\t= " << ans[max_idx]
            << "\n\tanalytic_ans[" << max_idx << "] \t\t= " << analytic[max_idx] << '\n';
  const double nd = norm(diff.data(), n);
  std::cout << "\nTotal norm of differences\t= " << nd << '\n';
  std::cout << "Relative norm of differences\t= " << nd / (double)norm(analytic, n) << '\n';
}
#endif

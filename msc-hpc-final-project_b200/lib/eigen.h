// eigen.h — host mirror of eigenDecomp<T> (parallel-final/lib/eigen.h:10-39, eigen.cu:17-21).
// The reference calls LAPACKE_dstevd on the host; here the k x k tridiagonal is solved on the device (lz_tridiag_expv),
// together with the coefficient vector multOut needs. eigenvalues are ascending; eigenvectors[i*k + j] = component i of
// eigenvector j — the layout LAPACK_ROW_MAJOR dstevd returns. Unlike the reference, L.beta is left intact.
// eigenDecomp(L, kind, param) first selects the matrix function multOut applies (lz_set_matfun: LZ_MATFUN_EXP with inverse
// temperature param, LZ_MATFUN_EXP_SCALED, LZ_MATFUN_RESOLVENT for Katz); the one-argument form keeps e^A.
#ifndef LZ_EIGEN_H
#define LZ_EIGEN_H

#include <vector>

#include "adjMatrix.h"
#include "cu_lanczos.h"

template <typename T>
class eigenDecomp {
 private:
  T* eigenvalues;
  T* eigenvectors;
  lanczosDecomp<T>& L;
  void decompose();

 public:
  eigenDecomp() = delete;
  eigenDecomp(lanczosDecomp<T>& _L)
      : eigenvalues(new T[_L.krylov_dim]), eigenvectors(new T[(size_t)_L.krylov_dim * _L.krylov_dim]), L{_L} {
    decompose();
  }
  eigenDecomp(lanczosDecomp<T>& _L, int kind, double param)
      : eigenvalues(new T[_L.krylov_dim]), eigenvectors(new T[(size_t)_L.krylov_dim * _L.krylov_dim]), L{_L} {
    if (lz_set_matfun(L.ctx, kind, param) != LZ_OK) lanczosDecomp<T>::fail("eigenDecomp: lz_set_matfun");
    decompose();
  }
  eigenDecomp(eigenDecomp<T>&) = delete;
  eigenDecomp& operator=(eigenDecomp<T>&) = delete;
  ~eigenDecomp() {
    delete[] eigenvalues;
    delete[] eigenvectors;
  }
  const T* get_eigenvalues() const { return eigenvalues; }
  const T* get_eigenvectors() const { return eigenvectors; }
  // f(A) x = ans * e^log_scale(): nonzero only for LZ_MATFUN_EXP_SCALED
  double log_scale() const {
    double ls = 0.0;
    if (lz_get_matfun_scale(L.ctx, &ls) != LZ_OK) lanczosDecomp<T>::fail("eigenDecomp: lz_get_matfun_scale");
    return ls;
  }
  template <typename U> friend void multOut(lanczosDecomp<U>&, eigenDecomp<U>&, adjMatrix&, bool);
};

template <typename T>
void eigenDecomp<T>::decompose() {
  const unsigned k = L.krylov_dim;
  if (lz_tridiag_expv(L.ctx) != LZ_OK) lanczosDecomp<T>::fail("eigenDecomp: lz_tridiag_expv");
  std::vector<double> w(k), z((size_t)k * k);
  if (lz_get_eigen(L.ctx, w.data(), z.data(), nullptr) != LZ_OK) lanczosDecomp<T>::fail("eigenDecomp: lz_get_eigen");
  for (unsigned i = 0; i < k; i++) eigenvalues[i] = (T)w[i];
  for (size_t i = 0; i < (size_t)k * k; i++) eigenvectors[i] = (T)z[i];
}
#endif

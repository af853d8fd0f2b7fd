// ritz.h — the top m Ritz pairs of a lanczosDecomp, checked against A on the device (lz_ritz). The reference has no such class; it
// follows eigenDecomp: the constructor does the work, accessors read the result. Values are largest first; [rayleigh_j - resid_j,
// rayleigh_j + resid_j] contains an eigenvalue of A. Afterwards L's answer is y_0 (eigenvector centrality: L.top_k ranks by it) until
// the next multOut. spectral_radius_bounds() gives lo <= lambda_max <= hi; alpha = f / hi with f < 1 is a certified Katz parameter.
#ifndef LZ_RITZ_H
#define LZ_RITZ_H

#include <vector>

#include "cu_lanczos.h"

template <typename T>
class ritzPairs {
 private:
  lanczosDecomp<T>& L;
  unsigned m;
  std::vector<double> theta, rho, res;

 public:
  ritzPairs() = delete;
  ritzPairs(lanczosDecomp<T>& _L, unsigned _m) : L{_L}, m{_m}, theta(_m), rho(_m), res(_m) {
    if (lz_ritz(L.ctx, m) != LZ_OK) lanczosDecomp<T>::fail("ritzPairs: lz_ritz");
    if (lz_get_ritz(L.ctx, theta.data(), rho.data(), res.data()) != LZ_OK) lanczosDecomp<T>::fail("ritzPairs: lz_get_ritz");
  }
  ritzPairs(ritzPairs<T>&) = delete;
  ritzPairs& operator=(ritzPairs<T>&) = delete;
  unsigned size() const { return m; }
  const std::vector<double>& values() const { return theta; }
  const std::vector<double>& rayleigh() const { return rho; }
  const std::vector<double>& residuals() const { return res; }
  // y_j, n entries in original vertex order, unit 2-norm, non-negative sum
  void vector(unsigned j, T* out) const {
    std::vector<double> y(L.get_n());
    if (lz_get_ritz_vector(L.ctx, j, y.data()) != LZ_OK) lanczosDecomp<T>::fail("ritzPairs: lz_get_ritz_vector");
    for (unsigned i = 0; i < L.get_n(); i++) out[i] = (T)y[i];
  }
  void spectral_radius_bounds(double& lo, double& hi) const {
    if (lz_spectral_radius_bounds(L.ctx, &lo, &hi) != LZ_OK) lanczosDecomp<T>::fail("ritzPairs: lz_spectral_radius_bounds");
  }
};
#endif

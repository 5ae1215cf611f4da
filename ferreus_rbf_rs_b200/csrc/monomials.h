// Monomial basis of the polynomial drift (polynomials.rs:15-62).  This is the one place that fixes the column order
// [1, x, y, z, x^2, xy, xz, y^2, yz, z^2]: 1, the dim linear terms, then the products s_a * s_b for a <= b.  The host
// evaluate_monomials (solver_host.cpp) and the interpolant finish kernel (device_io.cu) both call it.
#pragma once

#if defined(__CUDACC__)
#define FB_HOST_DEVICE __host__ __device__
#else
#define FB_HOST_DEVICE
#endif

namespace fb {

// s: scaled coordinates (p - translation) / scale; o: the basis row (1, 1 + dim or (dim + 1)(dim + 2) / 2 entries)
FB_HOST_DEVICE inline void monomial_row(const double *s, int dim, int degree, double *o) {
  o[0] = 1.0;
  if (degree >= 1)
    for (int d = 0; d < dim; ++d) o[1 + d] = s[d];
  if (degree == 2) {
    int k = 1 + dim;
    for (int a = 0; a < dim; ++a)
      for (int b = a; b < dim; ++b) o[k++] = s[a] * s[b];
  }
}

}  // namespace fb

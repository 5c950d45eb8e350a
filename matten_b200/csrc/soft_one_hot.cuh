// Radial modes 3-6 of mt_edge_radial / mt_edge_radial_bwd (include/matten_b200.h), used by edge_radial_kernel and
// edge_radial_bwd_kernel in graph_ops.cu.  Plain C++ apart from the function qualifiers, so that
// tests/test_radial_basis_host.py can compile it for the host and compare it with the reference.
#pragma once

namespace mt {

// Modes 3-6: e3nn soft_one_hot_linspace(r, start, end, nb, basis, cutoff) * sqrt(nb) for basis 3 gaussian,
// 4 cosine, 5 smooth_finite, 6 fourier: basis function k at r, or with DR its derivative with respect to r.  The
// masks have zero derivative, as under autograd through e3nn.
template <typename T, bool DR>
__device__ __forceinline__ T soft_one_hot(int mode, int k, int nb, T r, T start, T end, int cutoff) {
  const T pi = T(3.14159265358979323846);
  const T scale = sqrt(T(nb));
  // centres: linspace(start, end, n), or with cutoff the inner n of linspace(start, end, n + 2); d in steps
  const T step = (end - start) / T(cutoff ? nb + 1 : nb - 1);
  const T d = (r - (start + T(cutoff ? k + 1 : k) * step)) / step;
  if (mode == 3) {  // exp(-d^2) / 1.12
    const T v = exp(-(d * d)) / T(1.12) * scale;
    return DR ? T(-2) * d / step * v : v;
  }
  if (mode == 5) {
    // smooth_finite: C u(d + 1) u(1 - d) with u(t) = exp(-1/t) for t > 0, else 0.  C is e3nn's
    // 1.14136 * exp(2), which it evaluates in fp32.
    const T C = T(8.433573722839355);
    const T t1 = d + T(1), t2 = T(1) - d;
    const T u1 = t1 > T(0) ? exp(T(-1) / t1) : T(0);
    const T u2 = t2 > T(0) ? exp(T(-1) / t2) : T(0);
    if (!DR) return C * u1 * u2 * scale;
    // u'(t) = u(t) / t^2, taken as 0 wherever u(t) is 0 (t^2 may have underflowed there, and 0 / 0 is NaN)
    const T du1 = u1 > T(0) ? u1 / (t1 * t1) : T(0);
    const T du2 = u2 > T(0) ? u2 / (t2 * t2) : T(0);
    return C * (du1 * u2 - u1 * du2) / step * scale;
  }
  // the two trigonometric bases share one sincos (one call site of its slow argument reduction):
  //   cosine:  cos(pi/2 d) [-1 < d < 1]
  //   fourier: x = (r - start) / (end - start); cos(pi i x) for i = 0..n-1, or with cutoff sin(pi i x) [0 < x < 1]
  //            for i = 1..n; divided by sqrt(0.25 + n/2)
  T arg, darg, m;
  bool sine = false;
  if (mode == 4) {
    const T a = T(0.5) * pi;
    arg = a * d;
    darg = a / step;
    m = (d < T(1) && T(-1) < d) ? scale : T(0);
  } else {
    const T c = end - start, x = (r - start) / c;
    const T a = T(cutoff ? k + 1 : k) * pi;
    arg = a * x;
    darg = a / c;
    m = (!cutoff || (T(0) < x && x < T(1))) ? scale / sqrt(T(0.25) + T(nb) / T(2)) : T(0);
    sine = cutoff;
  }
  T s, c;
  sincos(arg, &s, &c);
  if (!DR) return (sine ? s : c) * m;
  return (sine ? c : -s) * darg * m;
}

}  // namespace mt

// Device math used by the elementwise and fused kernels.
//
// float32: libdevice expf/logf/powf (no fast-math), which is well inside the 1e-5 relative
// tolerance against numpy.
// float64: the reference's own tests compare exp/log results to numpy with `==`
// (test/test_autograd.py:90-96, 182-189), and numpy returns the correctly rounded value there.
// CUDA's exp()/log() are 1-ulp functions, so the f64 path evaluates exp in double-double
// arithmetic (~100 significant bits) and rounds once; log is one Newton step on top of it.
#pragma once
#include <math.h>
#if defined(__CUDACC__)
#include <cuda_runtime.h>
#define TNN_HD __host__ __device__ __forceinline__
#else
#define TNN_HD static inline
#endif

namespace tnn {

// Rounding-exact primitives.  On the device the intrinsics stop ptxas from contracting a*b+c
// into an FMA (which would break the error-free transformations); the host build (used by the
// CPU unit test of exp_cr/log_cr) is compiled with -ffp-contract=off.
#if defined(__CUDA_ARCH__)
TNN_HD double d_add(double a, double b) { return __dadd_rn(a, b); }
TNN_HD double d_sub(double a, double b) { return __dsub_rn(a, b); }
TNN_HD double d_mul(double a, double b) { return __dmul_rn(a, b); }
TNN_HD double d_div(double a, double b) { return __ddiv_rn(a, b); }
TNN_HD double d_fma(double a, double b, double c) { return __fma_rn(a, b, c); }
#else
TNN_HD double d_add(double a, double b) { return a + b; }
TNN_HD double d_sub(double a, double b) { return a - b; }
TNN_HD double d_mul(double a, double b) { return a * b; }
TNN_HD double d_div(double a, double b) { return a / b; }
TNN_HD double d_fma(double a, double b, double c) { return fma(a, b, c); }
#endif

struct dd {
  double hi, lo;
};

TNN_HD dd two_sum(double a, double b) {
  double s = d_add(a, b);
  double bb = d_sub(s, a);
  double e = d_add(d_sub(a, d_sub(s, bb)), d_sub(b, bb));
  return dd{s, e};
}
TNN_HD dd fast_two_sum(double a, double b) {  // |a| >= |b|
  double s = d_add(a, b);
  double e = d_sub(b, d_sub(s, a));
  return dd{s, e};
}
TNN_HD dd two_prod(double a, double b) {
  double p = d_mul(a, b);
  double e = d_fma(a, b, -p);
  return dd{p, e};
}
TNN_HD dd dd_add(dd a, dd b) {
  dd s = two_sum(a.hi, b.hi);
  dd t = two_sum(a.lo, b.lo);
  s.lo = d_add(s.lo, t.hi);
  s = fast_two_sum(s.hi, s.lo);
  s.lo = d_add(s.lo, t.lo);
  return fast_two_sum(s.hi, s.lo);
}
TNN_HD dd dd_add_d(dd a, double b) {
  dd s = two_sum(a.hi, b);
  s.lo = d_add(s.lo, a.lo);
  return fast_two_sum(s.hi, s.lo);
}
TNN_HD dd dd_mul(dd a, dd b) {
  dd p = two_prod(a.hi, b.hi);
  p.lo = d_add(p.lo, d_add(d_mul(a.hi, b.lo), d_mul(a.lo, b.hi)));
  return fast_two_sum(p.hi, p.lo);
}
TNN_HD dd dd_div_d(dd a, double n) {  // a / n
  double q1 = d_div(a.hi, n);
  dd p = two_prod(q1, n);
  // remainder r = a - q1*n, evaluated exactly enough in double-double
  double r = d_add(d_add(d_sub(a.hi, p.hi), -p.lo), a.lo);
  double q2 = d_div(r, n);
  return fast_two_sum(q1, q2);
}

// exp(x) as an unrounded double-double, |x| < 700
TNN_HD dd exp_dd(double x, int* k_out) {
  const double INV_LN2 = 1.4426950408889634074;
  const double LN2_HI = 0x1.62e42fefa39efp-1;
  const double LN2_LO = 0x1.abc9e3b39803fp-56;
  double k = rint(x * INV_LN2);
  // r = x - k*ln2 (double-double)
  dd t = two_prod(k, LN2_HI);
  dd u = two_prod(k, LN2_LO);
  dd kl = dd_add(t, u);
  dd r = dd_add(dd{x, 0.0}, dd{-kl.hi, -kl.lo});
  // s = r / 64, |s| <= 0.0055; exp(s) by a degree-11 Horner in double-double
  dd s = dd{r.hi * 0.015625, r.lo * 0.015625};
  dd acc = dd{1.0, 0.0};
#pragma unroll
  for (int i = 11; i >= 1; --i) {
    // acc = 1 + s/i * acc
    dd q = dd_div_d(dd_mul(s, acc), (double)i);
    acc = dd_add_d(q, 1.0);
  }
  // undo the scaling: six squarings
#pragma unroll
  for (int i = 0; i < 6; ++i) acc = dd_mul(acc, acc);
  *k_out = (int)k;
  return acc;
}

TNN_HD double exp_cr(double x) {
  if (!(fabs(x) < 700.0)) return exp(x);  // overflow / underflow / nan / inf: libdevice
  int k;
  dd e = exp_dd(x, &k);
  return ldexp(d_add(e.hi, e.lo), k);
}

TNN_HD double log_cr(double x) {
  if (!(x > 1e-300 && x < 1e300)) return log(x);  // <=0, nan, inf, subnormal range: libdevice
  double y0 = log(x);
  if (!(fabs(y0) < 690.0)) return y0;
  int k;
  dd e = exp_dd(y0, &k);  // exp(y0) = e * 2^k  ~ x
  // c = (x - exp(y0)) / x  evaluated on the scaled value to stay exact
  double xs = ldexp(x, -k);
  double c = d_div(d_sub(d_sub(xs, e.hi), e.lo), xs);
  return d_add(y0, c);
}

// numpy's `**` goes through libm pow(); small integral exponents are evaluated by repeated
// multiplication so integer-valued results stay exact (test_autograd.py:62-67).
template <typename T>
TNN_HD T pow_int(T a, int e) {
  bool neg = e < 0;
  unsigned u = neg ? (unsigned)(-e) : (unsigned)e;
  T r = T(1), b = a;
  while (u) {
    if (u & 1u) r *= b;
    b *= b;
    u >>= 1;
  }
  return neg ? T(1) / r : r;
}

TNN_HD float m_exp(float x) { return expf(x); }
TNN_HD double m_exp(double x) { return exp_cr(x); }
TNN_HD float m_log(float x) { return logf(x); }
TNN_HD double m_log(double x) { return log_cr(x); }
TNN_HD float m_pow(float a, float b) {
  float rb = rintf(b);
  if (rb == b && fabsf(b) <= 64.f) return pow_int<float>(a, (int)rb);
  return powf(a, b);
}
TNN_HD double m_pow(double a, double b) {
  double rb = rint(b);
  if (rb == b && fabs(b) <= 64.0) return pow_int<double>(a, (int)rb);
  return pow(a, b);
}
TNN_HD float m_sqrt(float x) { return sqrtf(x); }
TNN_HD double m_sqrt(double x) { return sqrt(x); }
// Plain libdevice functions in both precisions, for the activations (nothing there is compared
// with `==`, so exp needs no correctly rounded f64 path).
TNN_HD float m_exp_ld(float x) { return expf(x); }
TNN_HD double m_exp_ld(double x) { return exp(x); }
TNN_HD float m_expm1(float x) { return expm1f(x); }
TNN_HD double m_expm1(double x) { return expm1(x); }
TNN_HD float m_log1p(float x) { return log1pf(x); }
TNN_HD double m_log1p(double x) { return log1p(x); }
// np.maximum / np.minimum propagate NaN (fmax/fmin do not)
template <typename T>
TNN_HD T m_max(T a, T b) { return (a != a) ? a : ((b != b) ? b : (a > b ? a : b)); }
template <typename T>
TNN_HD T m_min(T a, T b) { return (a != a) ? a : ((b != b) ? b : (a < b ? a : b)); }

#if defined(__CUDACC__)  // (normcdf is a CUDA math function; the host build of this header has none)
// ---- activations (TNN_OP_LEAKY_RELU .. TNN_OP_SILU_BWD; formulas in include/tnn_b200.h) ----------
// The kink at 0 goes to the x >= 0 branch; NaN in gives NaN out; +-inf give the limits; every finite
// x gives a finite value and derivative.  A product x * w whose weight w has underflowed to 0 is
// taken as 0, so no inf * 0 reaches the output (x = -inf, or x^2, x^3 overflowed).

// the logistic function without overflow: s = sigma(v), sn = sigma(-v) = 1 - s (NaN for NaN v)
template <typename T>
struct Sigmoid2 {
  T s, sn;
};
template <typename T>
TNN_HD Sigmoid2<T> sigmoid2(T v) {
  const T e = m_exp_ld(-fabs(v));
  const T lo = e / (T(1) + e), hi = T(1) / (T(1) + e);
  return v >= T(0) ? Sigmoid2<T>{hi, lo} : Sigmoid2<T>{lo, hi};
}
template <typename T>
TNN_HD T mul_or_zero(T x, T w) { return w == T(0) ? T(0) : x * w; }

template <typename T>
TNN_HD T act_leaky_relu(T x, T slope) {
  if (!(x < T(0))) return x;                      // x >= 0 or NaN
  return mul_or_zero(x, slope);
}
template <typename T>
TNN_HD T act_leaky_relu_bwd(T g, T x, T slope) {
  if (!(x < T(0))) return x >= T(0) ? g : x;
  return g * slope;
}
template <typename T>
TNN_HD T act_elu(T x, T alpha) { return x >= T(0) ? x : alpha * m_expm1(x); }
template <typename T>
TNN_HD T act_elu_bwd(T g, T x, T alpha) { return x >= T(0) ? g : g * (alpha * m_exp_ld(x)); }

// Phi(x) = erfc(-x / sqrt 2) / 2 as libdevice's normcdf (x / sqrt 2 is not rounded first; with erfc
// written out, the f64 backward's flat vector kernel spills), phi(x) = exp(-x^2 / 2) / sqrt(2 pi)
TNN_HD float m_normcdf(float x) { return normcdff(x); }
TNN_HD double m_normcdf(double x) { return normcdf(x); }
template <typename T>
TNN_HD T act_gelu(T x) { return mul_or_zero(x, m_normcdf(x)); }
template <typename T>
TNN_HD T act_gelu_bwd(T g, T x) {
  const T pdf = m_exp_ld(T(-0.5) * (x * x)) * T(0.39894228040143267794);
  return g * (m_normcdf(x) + mul_or_zero(x, pdf));
}

// u = sqrt(2/pi) (x + 0.044715 x^3); y = x sigma(2u); x^3 = +-inf still gives sigma(2u) in {0, 1}
template <typename T>
TNN_HD Sigmoid2<T> gelu_tanh_sig(T x) {
  return sigmoid2(T(2) * (T(0.79788456080286535588) * (x + T(0.044715) * (x * x * x))));
}
template <typename T>
TNN_HD T act_gelu_tanh(T x) { return mul_or_zero(x, gelu_tanh_sig(x).s); }
template <typename T>
TNN_HD T act_gelu_tanh_bwd(T g, T x) {
  const Sigmoid2<T> q = gelu_tanh_sig(x);
  const T w = q.s * q.sn;                         // s (1 - s) without cancellation
  // where w has underflowed, the polynomial (which overflows first at |x| ~ 2e19 in f32) is not read
  const T t = w == T(0) ? T(0)
                        : (T(2) * x) * w * (T(0.79788456080286535588) * (T(1) + T(0.134145) * (x * x)));
  return g * (q.s + t);
}

template <typename T>
TNN_HD T act_softplus(T x) { return (x > T(0) ? x : T(0)) + m_log1p(m_exp_ld(-fabs(x))); }
template <typename T>
TNN_HD T act_softplus_bwd(T g, T x) { return g * sigmoid2(x).s; }

template <typename T>
TNN_HD T act_silu(T x) { return mul_or_zero(x, sigmoid2(x).s); }
template <typename T>
TNN_HD T act_silu_bwd(T g, T x) {
  const Sigmoid2<T> q = sigmoid2(x);
  return g * (q.s + mul_or_zero(x, q.s * q.sn));
}
#endif  // __CUDACC__

}  // namespace tnn

// Pointwise losses (new: no reference counterpart): MSE, MAE, Huber and sigmoid cross-entropy of a
// prediction p against a target t of the same shape (core/losses.py),
//
//   L = (1/m) * sum over all n elements of l(p, t),   m = rows of the global batch
//
//   tnn_pointwise_loss      ONE pass over (p, t): L, and -- given dp -- dL/dp for the upstream gradient 1
//                           (the seed of loss.backward()), so the loss's forward and default backward
//                           are one launch
//   tnn_pointwise_loss_bwd  dp = dl/dp * (g / m) for any other upstream gradient g, read on the device
//
// Memory pass: int64 indices, 16-byte vector accesses when n and every pointer allow it (scalar
// otherwise), a grid-stride loop over a grid fixed by n and the SM count (ew_grid).  Each term, its
// derivative and every sum are float64; the results are rounded once to the dtype.  Each thread sums
// its terms in a fixed order, each CTA folds its threads in a fixed tree, and the last CTA to arrive
// folds the CTA partials in CTA order (col_fold_last_arrival, the column reductions' counters).  No
// floating-point atomics, no host read: bit-identical results run to run and under graph replay.
#include "common.cuh"

namespace tnn {
namespace {

constexpr int kThreads = 256;

// sign(e) as numpy has it: 0 at e = 0 (keeping the zero's sign), NaN for NaN
__device__ __forceinline__ double sgn(double e) { return e > 0.0 ? 1.0 : (e < 0.0 ? -1.0 : e); }

// l(p, t) and dl/dp, both float64.  Sigmoid cross-entropy in its overflow-free form:
// max(z, 0) - z t + log1p(exp(-|z|)), sigmoid(z) = (z >= 0 ? 1 : exp(-|z|)) / (1 + exp(-|z|))
template <int KIND, bool WANT_L>
__device__ __forceinline__ void loss_term(double p, double t, double delta, double& l, double& d) {
  if constexpr (KIND == TNN_LOSS_SIGMOID_CE) {
    const double en = exp(-fabs(p));
    if (WANT_L) l = ((p < 0.0 ? 0.0 : p) - p * t) + log1p(en);
    d = (p >= 0.0 ? 1.0 : en) / (1.0 + en) - t;
  } else {
    const double e = p - t;
    if constexpr (KIND == TNN_LOSS_MSE) {
      if (WANT_L) l = e * e;
      d = 2.0 * e;
    } else if constexpr (KIND == TNN_LOSS_MAE) {
      if (WANT_L) l = fabs(e);
      d = sgn(e);
    } else {
      const double a = fabs(e);
      const bool quad = a < delta;
      if (WANT_L) l = quad ? 0.5 * e * e : delta * (a - 0.5 * delta);
      d = quad ? e : delta * sgn(e);
    }
  }
}

// the gradient one element receives, dl/dp * (g / m): the seeded output of the forward pass takes
// scale = 1.0 / m, the backward pass g / m with g read from the device -- the same expressions, so
// g = 1 gives the same bits.  (One division per thread, not per element: a float64 division is a
// subroutine of some twenty instructions.)
template <typename T>
__device__ __forceinline__ T grad_out(double d, double scale) { return (T)(d * scale); }

// one 16-byte access: 4 floats or 2 doubles
template <typename T>
struct alignas(16) Pack {
  static constexpr int W = 16 / sizeof(T);
  T e[W];
};

// sum of one double per thread over the CTA, in a fixed order; the result is valid in thread 0
__device__ __forceinline__ double cta_sum(double s, double* sm) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();                       // sm may still be read by a previous call
  if (lane == 0) sm[warp] = s;
  __syncthreads();
  if (threadIdx.x == 0)
    for (int w = 1; w < kThreads / 32; ++w) s += sm[w];
  return s;
}

// VEC: the body moves 16-byte packs (p, t and dp all aligned), the n % W tail is taken by the first
// threads of the grid
template <typename T, int KIND, bool VEC>
__global__ void __launch_bounds__(kThreads)
pointwise_loss_fwd_kernel(const T* __restrict__ p, const T* __restrict__ t, int64_t n, double m, double delta,
                          T* loss, T* __restrict__ dp, double* partials, unsigned int* counter) {
  __shared__ double sm[kThreads / 32];
  const int64_t tid = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  const double scale = 1.0 / m;
  double s = 0.0, l, d;
  int64_t done = 0;
  if constexpr (VEC) {
    constexpr int W = Pack<T>::W;
    using V = Pack<T>;
    const int64_t nv = n / W;
    for (int64_t i0 = tid; i0 < nv; i0 += 2 * stride) {
      V a[2], b[2], r;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < nv) {
          a[u] = reinterpret_cast<const V*>(p)[i];
          b[u] = reinterpret_cast<const V*>(t)[i];
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < nv) {
#pragma unroll
          for (int k = 0; k < W; ++k) {
            loss_term<KIND, true>((double)a[u].e[k], (double)b[u].e[k], delta, l, d);
            s += l;
            r.e[k] = grad_out<T>(d, scale);
          }
          if (dp) reinterpret_cast<V*>(dp)[i] = r;
        }
      }
    }
    done = nv * W;
  }
  for (int64_t i = done + tid; i < n; i += stride) {
    loss_term<KIND, true>((double)p[i], (double)t[i], delta, l, d);
    s += l;
    if (dp) dp[i] = grad_out<T>(d, scale);
  }
  s = cta_sum(s, sm);
  if (gridDim.x > 1) {
    if (threadIdx.x == 0) partials[blockIdx.x] = s;
    if (!col_fold_last_arrival(counter, gridDim.x)) return;
    s = 0.0;
    for (int64_t j = threadIdx.x; j < gridDim.x; j += kThreads) s += __ldcg(partials + j);
    s = cta_sum(s, sm);
  }
  if (threadIdx.x == 0) loss[0] = (T)(s / m);
}

template <typename T, int KIND, bool VEC>
__global__ void __launch_bounds__(kThreads)
pointwise_loss_bwd_kernel(T* __restrict__ dp, const T* __restrict__ p, const T* __restrict__ t, int64_t n,
                          double m, double delta, const T* gptr) {
  const int64_t tid = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  const double scale = (double)gptr[0] / m;
  double l, d;
  int64_t done = 0;
  if constexpr (VEC) {
    constexpr int W = Pack<T>::W;
    using V = Pack<T>;
    const int64_t nv = n / W;
    for (int64_t i0 = tid; i0 < nv; i0 += 2 * stride) {
      V a[2], b[2], r;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < nv) {
          a[u] = reinterpret_cast<const V*>(p)[i];
          b[u] = reinterpret_cast<const V*>(t)[i];
        }
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < nv) {
#pragma unroll
          for (int k = 0; k < W; ++k) {
            loss_term<KIND, false>((double)a[u].e[k], (double)b[u].e[k], delta, l, d);
            r.e[k] = grad_out<T>(d, scale);
          }
          reinterpret_cast<V*>(dp)[i] = r;
        }
      }
    }
    done = nv * W;
  }
  for (int64_t i = done + tid; i < n; i += stride) {
    loss_term<KIND, false>((double)p[i], (double)t[i], delta, l, d);
    dp[i] = grad_out<T>(d, scale);
  }
}

// ---- host side --------------------------------------------------------------------------------
bool aligned16(const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; }

// one grid for both passes of a given (n, vector path): the forward's sum order depends on nothing else
int loss_grid(int64_t n, bool vec, int W) { return ew_grid(vec ? ceil_div(n, 2 * W) : ceil_div(n, 2), kThreads); }

template <typename T, int KIND>
int fwd_impl(const void* p, const void* t, int64_t n, double m, double delta, void* loss, void* dp) {
  constexpr int W = Pack<T>::W;
  const bool vec = n >= W && aligned16(p) && aligned16(t) && (!dp || aligned16(dp));
  const int grid = loss_grid(n, vec, W);
  double* partials = nullptr;
  unsigned int* counters = nullptr;
  if (grid > 1) {
    void* scratch;
    if (get_scratch((size_t)grid * sizeof(double), &scratch)) return 1;
    partials = (double*)scratch;
    if (col_fold_counters(&counters)) return 1;
  }
  cudaStream_t st = ctx().stream;
  if (vec)
    pointwise_loss_fwd_kernel<T, KIND, true><<<grid, kThreads, 0, st>>>((const T*)p, (const T*)t, n, m, delta,
                                                                       (T*)loss, (T*)dp, partials, counters);
  else
    pointwise_loss_fwd_kernel<T, KIND, false><<<grid, kThreads, 0, st>>>((const T*)p, (const T*)t, n, m, delta,
                                                                        (T*)loss, (T*)dp, partials, counters);
  TNN_POST_LAUNCH();
  return 0;
}

template <typename T, int KIND>
int bwd_impl(void* dp, const void* p, const void* t, int64_t n, double m, double delta, const void* g) {
  constexpr int W = Pack<T>::W;
  const bool vec = n >= W && aligned16(p) && aligned16(t) && aligned16(dp);
  const int grid = loss_grid(n, vec, W);
  cudaStream_t st = ctx().stream;
  if (vec)
    pointwise_loss_bwd_kernel<T, KIND, true><<<grid, kThreads, 0, st>>>((T*)dp, (const T*)p, (const T*)t, n, m,
                                                                       delta, (const T*)g);
  else
    pointwise_loss_bwd_kernel<T, KIND, false><<<grid, kThreads, 0, st>>>((T*)dp, (const T*)p, (const T*)t, n, m,
                                                                        delta, (const T*)g);
  TNN_POST_LAUNCH();
  return 0;
}

int check_args(const char* name, int dtype, int kind, int64_t n, double m, double delta) {
  if (dtype != TNN_F32 && dtype != TNN_F64) TNN_FAIL(std::string(name) + ": bad dtype");
  if (kind < TNN_LOSS_MSE || kind > TNN_LOSS_SIGMOID_CE) TNN_FAIL(std::string(name) + ": bad loss kind");
  if (n < 0) TNN_FAIL(std::string(name) + ": negative element count");
  if (!(m >= 1.0)) TNN_FAIL(std::string(name) + ": m_global must be at least 1");
  if (kind == TNN_LOSS_HUBER && !(delta > 0.0 && delta < INFINITY))
    TNN_FAIL(std::string(name) + ": delta must be finite and > 0");
  return 0;
}

}  // namespace
}  // namespace tnn

using namespace tnn;

#define TNN_LOSS_DISPATCH(impl, ...)                                                       \
  do {                                                                                     \
    if (dtype == TNN_F32) {                                                                \
      switch (kind) {                                                                      \
        case TNN_LOSS_MSE: return impl<float, TNN_LOSS_MSE>(__VA_ARGS__);                  \
        case TNN_LOSS_MAE: return impl<float, TNN_LOSS_MAE>(__VA_ARGS__);                  \
        case TNN_LOSS_HUBER: return impl<float, TNN_LOSS_HUBER>(__VA_ARGS__);              \
        default: return impl<float, TNN_LOSS_SIGMOID_CE>(__VA_ARGS__);                     \
      }                                                                                    \
    }                                                                                      \
    switch (kind) {                                                                        \
      case TNN_LOSS_MSE: return impl<double, TNN_LOSS_MSE>(__VA_ARGS__);                   \
      case TNN_LOSS_MAE: return impl<double, TNN_LOSS_MAE>(__VA_ARGS__);                   \
      case TNN_LOSS_HUBER: return impl<double, TNN_LOSS_HUBER>(__VA_ARGS__);               \
      default: return impl<double, TNN_LOSS_SIGMOID_CE>(__VA_ARGS__);                      \
    }                                                                                      \
  } while (0)

extern "C" {

int tnn_pointwise_loss(int dtype, int kind, const void* p, const void* t, int64_t n, double m_global,
                       double delta, void* loss_dev, void* dp) {
  TNN_REQUIRE_INIT();
  if (check_args("tnn_pointwise_loss", dtype, kind, n, m_global, delta)) return 1;
  TNN_LOSS_DISPATCH(fwd_impl, p, t, n, m_global, delta, loss_dev, dp);
}

int tnn_pointwise_loss_bwd(int dtype, int kind, void* dp, const void* p, const void* t, int64_t n,
                           double m_global, double delta, const void* g_dev) {
  TNN_REQUIRE_INIT();
  if (check_args("tnn_pointwise_loss_bwd", dtype, kind, n, m_global, delta)) return 1;
  if (n == 0) return 0;
  TNN_LOSS_DISPATCH(bwd_impl, dp, p, t, n, m_global, delta, g_dev);
}

}  // extern "C"

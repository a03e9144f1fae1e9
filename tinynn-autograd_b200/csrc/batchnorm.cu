// Batch normalisation over the rows of an (M, C) matrix (new: no reference counterpart).  A 2-D
// (N, C) Dense output and a 4-D (N, H, W, C) NHWC Conv2D output are the same problem with M = N or
// M = N*H*W (core/layers.py BatchNormalization).
//
//   tnn_bn_stats       TRAIN column statistics; its fold writes mr = (mean, 1/sqrt(var + eps), M) and
//                      updates the running statistics, or writes the local (count, mean, M2) that a
//                      data-parallel run all-gathers and hands to
//   tnn_bn_merge       Chan's merge of the ranks' (count, mean, M2) in rank order -> mr + running update
//   tnn_bn_apply       y = (x - mean) * r * gamma + beta  (TEST: mean and r from the running statistics)
//   tnn_bn_bwd_reduce  sum(dy) and sum(dy * xhat) per column, xhat recomputed from x and mr; the fold
//                      writes (or accumulates) dbeta and dgamma
//   tnn_bn_dx          dx = gamma * r * (dy - sum(dy)/M - xhat * sum(dy*xhat)/M)  (TEST: gamma * r * dy)
//
// Layout of every pass: a CTA is TX x TY threads, TX column slots (EL consecutive channels each, one
// 16-byte access when C and the pointers allow it) times TY row lanes, so a warp reads whole rows of
// a narrow matrix.  The two reductions split the rows across CTAs and fold the partials in the last
// CTA to arrive for a column block, in split order (the scheme of reduce.cu's column sum, sharing
// its counters).  All statistics are float64 for both dtypes: the TRAIN sums are taken about each
// column's first row, which keeps sum((x - K)^2) - sum(x - K)^2 / M free of the cancellation a
// one-pass sum of x^2 suffers on offset data.  No floating-point atomics anywhere: results are
// bit-identical run to run and under graph replay.
#include <algorithm>

#include "common.cuh"

namespace tnn {
namespace {

template <typename T, int EL>
struct alignas(sizeof(T) * EL) BnPack {
  T v[EL];
};

constexpr int kThreads = 256;

// sum the per-thread (a, b) over the TY row lanes of the CTA, in lane order; valid where ty == 0
template <int EL>
__device__ __forceinline__ void fold_lanes(double (&a)[EL], double (&b)[EL], double* sm) {
  const int TX = blockDim.x, TY = blockDim.y, tx = threadIdx.x, ty = threadIdx.y;
#pragma unroll
  for (int k = 0; k < EL; ++k) {
    sm[(ty * TX + tx) * EL + k] = a[k];
    sm[kThreads * EL + (ty * TX + tx) * EL + k] = b[k];
  }
  __syncthreads();
  if (ty == 0) {
    for (int j = 1; j < TY; ++j)
#pragma unroll
      for (int k = 0; k < EL; ++k) {
        a[k] += sm[(j * TX + tx) * EL + k];
        b[k] += sm[kThreads * EL + (j * TX + tx) * EL + k];
      }
  }
  __syncthreads();
}

// rows [lo, hi) of the column slot, lane ty taking rows lo+ty, lo+ty+TY, ... with four loads in flight
template <typename T, int EL, typename F>
__device__ __forceinline__ void walk_rows(const T* __restrict__ p, const T* __restrict__ q, int64_t lo, int64_t hi,
                                          int64_t ncol, int64_t col, F&& f) {
  using P = BnPack<T, EL>;
  const int64_t TY = blockDim.y;
  const P* __restrict__ pp = reinterpret_cast<const P*>(p);
  const P* __restrict__ qq = reinterpret_cast<const P*>(q);
  int64_t r = lo + threadIdx.y;
  for (; r + 3 * TY < hi; r += 4 * TY) {
    P u[4], w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      u[i] = pp[(r + i * TY) * ncol + col];
      if (q) w[i] = qq[(r + i * TY) * ncol + col];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) f(u[i], w[i]);
  }
  for (; r < hi; r += TY) {
    P u = pp[r * ncol + col], w{};
    if (q) w = qq[r * ncol + col];
    f(u, w);
  }
}

// mean and 1/sqrt(var + eps) of column c from (n, mean, M2); the running statistics take the unbiased
// variance M2 / (n - 1)
template <typename T>
__device__ __forceinline__ void finalize(int64_t c, int64_t C, double n, double mean, double m2, double* mr,
                                         T* run_mean, T* run_var, double momentum, double eps) {
  const double r = 1.0 / sqrt(m2 / n + eps);
  mr[c] = mean;
  mr[C + c] = r;
  if (c == 0) mr[2 * C] = n;
  run_mean[c] = (T)((1.0 - momentum) * (double)run_mean[c] + momentum * mean);
  run_var[c] = (T)((1.0 - momentum) * (double)run_var[c] + momentum * (m2 / (n - 1.0)));
}

// the two split reductions share everything but what they accumulate and what the fold writes
struct SplitArgs {
  int64_t M, C;
  int nsplit;
  double* stage;           // (nsplit, 2, C) partials
  unsigned int* counters;  // one per column block
};

// partial (a, b) of this CTA's row chunk -> the column block's totals, in the last CTA to arrive
// (returns false in the others, which are done)
template <int EL>
__device__ __forceinline__ bool split_fold(double (&a)[EL], double (&b)[EL], double* sm, const SplitArgs& s,
                                           int64_t c0, bool active) {
  fold_lanes<EL>(a, b, sm);
  if (s.nsplit == 1) return true;
  if (threadIdx.y == 0 && active)
#pragma unroll
    for (int k = 0; k < EL; ++k) {
      s.stage[((int64_t)blockIdx.y * 2) * s.C + c0 + k] = a[k];
      s.stage[((int64_t)blockIdx.y * 2 + 1) * s.C + c0 + k] = b[k];
    }
  if (!col_fold_last_arrival(s.counters + blockIdx.x, (unsigned)s.nsplit)) return false;
#pragma unroll
  for (int k = 0; k < EL; ++k) a[k] = b[k] = 0.0;
  if (active)
    for (int64_t j = threadIdx.y; j < s.nsplit; j += blockDim.y)
#pragma unroll
      for (int k = 0; k < EL; ++k) {
        a[k] += __ldcg(s.stage + (j * 2) * s.C + c0 + k);
        b[k] += __ldcg(s.stage + (j * 2 + 1) * s.C + c0 + k);
      }
  fold_lanes<EL>(a, b, sm);
  return true;
}

template <typename T, int EL>
__global__ void __launch_bounds__(kThreads)
bn_stats_kernel(const T* __restrict__ x, SplitArgs s, double momentum, double eps, T* run_mean, T* run_var,
                double* mr, double* part) {
  __shared__ double sm[2 * kThreads * EL];
  const int64_t ncol = s.C / EL;
  const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = col < ncol;
  const int64_t c0 = col * EL;
  const int64_t chunk = ceil_div(s.M, s.nsplit);
  const int64_t lo = (int64_t)blockIdx.y * chunk, hi = min(lo + chunk, s.M);
  double K[EL], s1[EL], s2[EL];
#pragma unroll
  for (int k = 0; k < EL; ++k) {
    K[k] = (active && s.M > 0) ? (double)x[c0 + k] : 0.0;   // every CTA shifts by the same row 0
    s1[k] = s2[k] = 0.0;
  }
  if (active)
    walk_rows<T, EL>(x, nullptr, lo, hi, ncol, col, [&](const BnPack<T, EL>& u, const BnPack<T, EL>&) {
#pragma unroll
      for (int k = 0; k < EL; ++k) {
        const double d = (double)u.v[k] - K[k];
        s1[k] += d;
        s2[k] = fma(d, d, s2[k]);
      }
    });
  if (!split_fold<EL>(s1, s2, sm, s, c0, active)) return;
  if (threadIdx.y != 0 || !active) return;
  const double n = (double)s.M;
#pragma unroll
  for (int k = 0; k < EL; ++k) {
    const double mean = s.M > 0 ? K[k] + s1[k] / n : 0.0;
    const double m2 = s.M > 0 ? fmax(s2[k] - s1[k] * (s1[k] / n), 0.0) : 0.0;
    if (part) {
      if (c0 + k == 0) part[0] = n;
      part[1 + c0 + k] = mean;
      part[1 + s.C + c0 + k] = m2;
    } else {
      finalize<T>(c0 + k, s.C, n, mean, m2, mr, run_mean, run_var, momentum, eps);
    }
  }
}

// one thread per column; ranks merged in rank order (Chan et al.), so every rank gets the same bits
template <typename T>
__global__ void __launch_bounds__(kThreads)
bn_merge_kernel(const double* __restrict__ gathered, int world, int64_t C, double momentum, double eps,
                T* run_mean, T* run_var, double* mr) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  double n = 0.0, mean = 0.0, m2 = 0.0;
  for (int q = 0; q < world; ++q) {
    const double* p = gathered + (int64_t)q * (1 + 2 * C);
    const double nb = p[0];
    if (nb == 0.0) continue;
    const double tot = n + nb, delta = p[1 + c] - mean;
    mean += delta * (nb / tot);
    m2 += p[1 + C + c] + delta * delta * (n * nb / tot);
    n = tot;
  }
  finalize<T>(c, C, n, mean, m2, mr, run_mean, run_var, momentum, eps);
}

// TEST (run_mean != nullptr): mean and r from the running statistics, also written to mr for backward
template <typename T, int EL>
__device__ __forceinline__ void column_stats(int64_t c0, int64_t C, const double* mr, const T* run_mean,
                                             const T* run_var, double eps, double* mean, double* r) {
#pragma unroll
  for (int k = 0; k < EL; ++k) {
    if (run_mean) {
      mean[k] = (double)run_mean[c0 + k];
      r[k] = 1.0 / sqrt((double)run_var[c0 + k] + eps);
    } else {
      mean[k] = mr[c0 + k];
      r[k] = mr[C + c0 + k];
    }
  }
}

template <typename T, int EL>
__global__ void __launch_bounds__(kThreads)
bn_apply_kernel(T* __restrict__ y, const T* __restrict__ x, int64_t M, int64_t C, const T* gamma, const T* beta,
                double* mr, const T* run_mean, const T* run_var, double eps) {
  using P = BnPack<T, EL>;
  const int64_t ncol = C / EL;
  const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncol) return;
  const int64_t c0 = col * EL;
  double mean[EL], r[EL], scale[EL], shift[EL];
  column_stats<T, EL>(c0, C, mr, run_mean, run_var, eps, mean, r);
#pragma unroll
  for (int k = 0; k < EL; ++k) {
    scale[k] = r[k] * (double)gamma[c0 + k];
    shift[k] = (double)beta[c0 + k];
  }
  if (run_mean && blockIdx.y == 0 && threadIdx.y == 0) {
#pragma unroll
    for (int k = 0; k < EL; ++k) {
      mr[c0 + k] = mean[k];
      mr[C + c0 + k] = r[k];
    }
    if (c0 == 0) mr[2 * C] = (double)M;
  }
  const P* __restrict__ in = reinterpret_cast<const P*>(x);
  P* __restrict__ out = reinterpret_cast<P*>(y);
  const int64_t step = (int64_t)gridDim.y * blockDim.y;
#pragma unroll 4
  for (int64_t row = (int64_t)blockIdx.y * blockDim.y + threadIdx.y; row < M; row += step) {
    const P u = in[row * ncol + col];
    P v;
#pragma unroll
    for (int k = 0; k < EL; ++k) v.v[k] = (T)fma((double)u.v[k] - mean[k], scale[k], shift[k]);
    out[row * ncol + col] = v;
  }
}

template <typename T, int EL>
__global__ void __launch_bounds__(kThreads)
bn_bwd_reduce_kernel(const T* __restrict__ dy, const T* __restrict__ x, SplitArgs s, const double* mr,
                     double* sums, T* dgamma, int acc_gamma, T* dbeta, int acc_beta) {
  __shared__ double sm[2 * kThreads * EL];
  const int64_t ncol = s.C / EL;
  const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = col < ncol;
  const int64_t c0 = active ? col * EL : 0;
  const int64_t chunk = ceil_div(s.M, s.nsplit);
  const int64_t lo = (int64_t)blockIdx.y * chunk, hi = min(lo + chunk, s.M);
  double mean[EL], r[EL], a[EL], b[EL];
#pragma unroll
  for (int k = 0; k < EL; ++k) a[k] = b[k] = mean[k] = r[k] = 0.0;
  if (active) {
    column_stats<T, EL>(c0, s.C, mr, (const T*)nullptr, (const T*)nullptr, 0.0, mean, r);
    walk_rows<T, EL>(dy, x, lo, hi, ncol, col, [&](const BnPack<T, EL>& g, const BnPack<T, EL>& u) {
#pragma unroll
      for (int k = 0; k < EL; ++k) {
        const double gd = (double)g.v[k];
        a[k] += gd;
        b[k] = fma(gd, ((double)u.v[k] - mean[k]) * r[k], b[k]);
      }
    });
  }
  if (!split_fold<EL>(a, b, sm, s, c0, active)) return;
  if (threadIdx.y != 0 || !active) return;
#pragma unroll
  for (int k = 0; k < EL; ++k) {
    const int64_t c = c0 + k;
    sums[c] = a[k];
    sums[s.C + c] = b[k];
    if (dbeta) dbeta[c] = acc_beta ? (T)((double)dbeta[c] + a[k]) : (T)a[k];
    if (dgamma) dgamma[c] = acc_gamma ? (T)((double)dgamma[c] + b[k]) : (T)b[k];
  }
}

template <typename T, int EL, bool TRAIN>
__global__ void __launch_bounds__(kThreads)
bn_dx_kernel(T* __restrict__ dx, const T* __restrict__ dy, const T* __restrict__ x, int64_t M, int64_t C,
             const double* mr, const T* gamma, const double* sums) {
  using P = BnPack<T, EL>;
  const int64_t ncol = C / EL;
  const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncol) return;
  const int64_t c0 = col * EL;
  double mean[EL], r[EL], a[EL], mdy[EL], mdyx[EL];
  column_stats<T, EL>(c0, C, mr, (const T*)nullptr, (const T*)nullptr, 0.0, mean, r);
#pragma unroll
  for (int k = 0; k < EL; ++k) {
    a[k] = (double)gamma[c0 + k] * r[k];
    if (TRAIN) {
      const double n = mr[2 * C];
      mdy[k] = sums[c0 + k] / n;
      mdyx[k] = sums[C + c0 + k] / n;
    }
  }
  const P* __restrict__ gin = reinterpret_cast<const P*>(dy);
  const P* __restrict__ xin = reinterpret_cast<const P*>(x);
  P* __restrict__ out = reinterpret_cast<P*>(dx);
  const int64_t step = (int64_t)gridDim.y * blockDim.y;
#pragma unroll 4
  for (int64_t row = (int64_t)blockIdx.y * blockDim.y + threadIdx.y; row < M; row += step) {
    const P g = gin[row * ncol + col];
    P v;
    if (TRAIN) {
      const P u = xin[row * ncol + col];
#pragma unroll
      for (int k = 0; k < EL; ++k) {
        const double xhat = ((double)u.v[k] - mean[k]) * r[k];
        v.v[k] = (T)(a[k] * ((double)g.v[k] - mdy[k] - xhat * mdyx[k]));
      }
    } else {
#pragma unroll
      for (int k = 0; k < EL; ++k) v.v[k] = (T)(a[k] * (double)g.v[k]);
    }
    out[row * ncol + col] = v;
  }
}

// ---- host side --------------------------------------------------------------------------------
bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

struct Plan {
  int el;       // channels per access
  int tx, ty;   // CTA shape
  int64_t gx;   // column blocks
};

template <typename T>
Plan make_plan(int64_t C, bool ptrs_aligned) {
  Plan p;
  constexpr int V = 16 / sizeof(T);
  p.el = (ptrs_aligned && C % V == 0) ? V : 1;
  const int64_t ncol = C / p.el;
  p.tx = 1;
  while (p.tx < 32 && p.tx < ncol) p.tx *= 2;
  p.ty = kThreads / p.tx;
  p.gx = ceil_div(ncol, p.tx);
  return p;
}

// row chunks of the split reductions: about three CTAs per SM (the column sum's measured optimum),
// at least eight rows per lane in each
int split_count(const Plan& p, int64_t M) {
  const int64_t want = (int64_t)ctx().sm_count * 3;
  int64_t n = std::min<int64_t>(ceil_div(want, p.gx), ceil_div(M, (int64_t)p.ty * 8));
  n = std::max<int64_t>(1, std::min<int64_t>(n, 65535));
  if (p.gx > MAX_COL_COUNTERS) n = 1;
  return (int)n;
}

// rows of the elementwise passes: about eight CTAs per SM in all
int row_blocks(const Plan& p, int64_t M) {
  const int64_t want = ceil_div((int64_t)ctx().sm_count * 8, p.gx);
  return (int)std::max<int64_t>(1, std::min<int64_t>({want, ceil_div(M, (int64_t)p.ty), 65535}));
}

int prepare_split(const char* name, const Plan& p, int64_t M, int64_t C, SplitArgs* s) {
  if (p.gx > 2147483647LL) TNN_FAIL(std::string(name) + ": too many channels");
  s->M = M;
  s->C = C;
  s->nsplit = split_count(p, M);
  s->stage = nullptr;
  s->counters = nullptr;
  if (s->nsplit > 1) {
    void* scratch;
    if (get_scratch((size_t)s->nsplit * 2 * C * sizeof(double), &scratch)) return 1;
    s->stage = (double*)scratch;
    if (col_fold_counters(&s->counters)) return 1;
  }
  return 0;
}

template <typename T>
int stats_impl(const void* x, int64_t M, int64_t C, double momentum, double eps, void* rm, void* rv, double* mr,
               double* part) {
  const Plan p = make_plan<T>(C, aligned16(x));
  SplitArgs s;
  if (prepare_split("tnn_bn_stats", p, M, C, &s)) return 1;
  const dim3 grid((unsigned)p.gx, (unsigned)s.nsplit), block(p.tx, p.ty);
  cudaStream_t st = ctx().stream;
  if (p.el == 1)
    bn_stats_kernel<T, 1><<<grid, block, 0, st>>>((const T*)x, s, momentum, eps, (T*)rm, (T*)rv, mr, part);
  else
    bn_stats_kernel<T, 16 / sizeof(T)><<<grid, block, 0, st>>>((const T*)x, s, momentum, eps, (T*)rm, (T*)rv, mr, part);
  TNN_POST_LAUNCH();
  return 0;
}

template <typename T>
int merge_impl(const double* gathered, int world, int64_t C, double momentum, double eps, void* rm, void* rv,
               double* mr) {
  const int grid = (int)ceil_div(C, kThreads);
  bn_merge_kernel<T><<<grid, kThreads, 0, ctx().stream>>>(gathered, world, C, momentum, eps, (T*)rm, (T*)rv, mr);
  TNN_POST_LAUNCH();
  return 0;
}

template <typename T>
int apply_impl(void* y, const void* x, int64_t M, int64_t C, const void* gamma, const void* beta, double* mr,
               const void* rm, const void* rv, double eps) {
  const Plan p = make_plan<T>(C, aligned16(x) && aligned16(y));
  const dim3 grid((unsigned)p.gx, (unsigned)row_blocks(p, M)), block(p.tx, p.ty);
  cudaStream_t st = ctx().stream;
  if (p.el == 1)
    bn_apply_kernel<T, 1><<<grid, block, 0, st>>>((T*)y, (const T*)x, M, C, (const T*)gamma, (const T*)beta, mr,
                                                  (const T*)rm, (const T*)rv, eps);
  else
    bn_apply_kernel<T, 16 / sizeof(T)><<<grid, block, 0, st>>>((T*)y, (const T*)x, M, C, (const T*)gamma,
                                                               (const T*)beta, mr, (const T*)rm, (const T*)rv, eps);
  TNN_POST_LAUNCH();
  return 0;
}

template <typename T>
int bwd_reduce_impl(const void* dy, const void* x, int64_t M, int64_t C, const double* mr, double* sums,
                    void* dgamma, int acc_gamma, void* dbeta, int acc_beta) {
  const Plan p = make_plan<T>(C, aligned16(dy) && aligned16(x));
  SplitArgs s;
  if (prepare_split("tnn_bn_bwd_reduce", p, M, C, &s)) return 1;
  const dim3 grid((unsigned)p.gx, (unsigned)s.nsplit), block(p.tx, p.ty);
  cudaStream_t st = ctx().stream;
  if (p.el == 1)
    bn_bwd_reduce_kernel<T, 1><<<grid, block, 0, st>>>((const T*)dy, (const T*)x, s, mr, sums, (T*)dgamma,
                                                       acc_gamma, (T*)dbeta, acc_beta);
  else
    bn_bwd_reduce_kernel<T, 16 / sizeof(T)><<<grid, block, 0, st>>>((const T*)dy, (const T*)x, s, mr, sums,
                                                                    (T*)dgamma, acc_gamma, (T*)dbeta, acc_beta);
  TNN_POST_LAUNCH();
  return 0;
}

template <typename T, int EL>
void launch_dx(dim3 grid, dim3 block, void* dx, const void* dy, const void* x, int64_t M, int64_t C,
               const double* mr, const void* gamma, const double* sums) {
  cudaStream_t st = ctx().stream;
  if (sums)
    bn_dx_kernel<T, EL, true><<<grid, block, 0, st>>>((T*)dx, (const T*)dy, (const T*)x, M, C, mr, (const T*)gamma,
                                                      sums);
  else
    bn_dx_kernel<T, EL, false><<<grid, block, 0, st>>>((T*)dx, (const T*)dy, (const T*)x, M, C, mr,
                                                       (const T*)gamma, sums);
}

template <typename T>
int dx_impl(void* dx, const void* dy, const void* x, int64_t M, int64_t C, const double* mr, const void* gamma,
            const double* sums) {
  const Plan p = make_plan<T>(C, aligned16(dx) && aligned16(dy) && (!sums || aligned16(x)));
  const dim3 grid((unsigned)p.gx, (unsigned)row_blocks(p, M)), block(p.tx, p.ty);
  if (p.el == 1) launch_dx<T, 1>(grid, block, dx, dy, x, M, C, mr, gamma, sums);
  else launch_dx<T, 16 / sizeof(T)>(grid, block, dx, dy, x, M, C, mr, gamma, sums);
  TNN_POST_LAUNCH();
  return 0;
}

int check_shape(const char* name, int64_t M, int64_t C) {
  if (M < 0 || C <= 0) TNN_FAIL(std::string(name) + ": bad shape");
  return 0;
}

}  // namespace
}  // namespace tnn

using namespace tnn;

#define TNN_BN_DISPATCH(name, call)                                  \
  do {                                                               \
    if (dtype == TNN_F32) return call(float);                        \
    if (dtype == TNN_F64) return call(double);                       \
    TNN_FAIL(name ": bad dtype");                                    \
  } while (0)

extern "C" {

int tnn_bn_stats(int dtype, const void* x, int64_t M, int64_t C, double momentum, double eps, void* running_mean,
                 void* running_var, double* mr, double* part) {
  TNN_REQUIRE_INIT();
  if (check_shape("tnn_bn_stats", M, C)) return 1;
  if (!part && M < 2) TNN_FAIL("tnn_bn_stats: the unbiased running variance needs at least two rows");
#define TNN_BN_CALL(T) stats_impl<T>(x, M, C, momentum, eps, running_mean, running_var, mr, part)
  TNN_BN_DISPATCH("tnn_bn_stats", TNN_BN_CALL);
#undef TNN_BN_CALL
}

int tnn_bn_merge(int dtype, const double* gathered, int world, int64_t C, double momentum, double eps,
                 void* running_mean, void* running_var, double* mr) {
  TNN_REQUIRE_INIT();
  if (check_shape("tnn_bn_merge", 0, C)) return 1;
  if (world < 1) TNN_FAIL("tnn_bn_merge: bad world size");
#define TNN_BN_CALL(T) merge_impl<T>(gathered, world, C, momentum, eps, running_mean, running_var, mr)
  TNN_BN_DISPATCH("tnn_bn_merge", TNN_BN_CALL);
#undef TNN_BN_CALL
}

int tnn_bn_apply(int dtype, void* y, const void* x, int64_t M, int64_t C, const void* gamma, const void* beta,
                 double* mr, const void* running_mean, const void* running_var, double eps) {
  TNN_REQUIRE_INIT();
  if (check_shape("tnn_bn_apply", M, C)) return 1;
  if (M == 0) return 0;
#define TNN_BN_CALL(T) apply_impl<T>(y, x, M, C, gamma, beta, mr, running_mean, running_var, eps)
  TNN_BN_DISPATCH("tnn_bn_apply", TNN_BN_CALL);
#undef TNN_BN_CALL
}

int tnn_bn_bwd_reduce(int dtype, const void* dy, const void* x, int64_t M, int64_t C, const double* mr,
                      double* sums, void* dgamma, int acc_gamma, void* dbeta, int acc_beta) {
  TNN_REQUIRE_INIT();
  if (check_shape("tnn_bn_bwd_reduce", M, C)) return 1;
#define TNN_BN_CALL(T) bwd_reduce_impl<T>(dy, x, M, C, mr, sums, dgamma, acc_gamma, dbeta, acc_beta)
  TNN_BN_DISPATCH("tnn_bn_bwd_reduce", TNN_BN_CALL);
#undef TNN_BN_CALL
}

int tnn_bn_dx(int dtype, void* dx, const void* dy, const void* x, int64_t M, int64_t C, const double* mr,
              const void* gamma, const double* sums) {
  TNN_REQUIRE_INIT();
  if (check_shape("tnn_bn_dx", M, C)) return 1;
  if (M == 0) return 0;
#define TNN_BN_CALL(T) dx_impl<T>(dx, dy, x, M, C, mr, gamma, sums)
  TNN_BN_DISPATCH("tnn_bn_dx", TNN_BN_CALL);
#undef TNN_BN_CALL
}

}  // extern "C"

// Reductions: ops.py:225-265 (max_, min_, sum_) and the un-broadcast sum that the reference
// inlines into every binary op's grad fn (ops.py:41-46, 50-54, 73-77, ... 205-209):
//     for _ in range(grad.ndim - ts.ndim): grad = grad.sum(axis=0)
//     for i, dim in enumerate(ts.shape):   if dim == 1: grad = grad.sum(axis=i, keepdims=True)
//
// Every reduction is expressed on a contiguous (outer, red, inner) view and is deterministic:
// the red axis is cut into a fixed number of chunks (a function of the shape and the SM count
// only), each chunk is reduced by one CTA with a sequential per-thread walk + warp shuffles +
// a shared-memory tree, the per-chunk partials are written to scratch and a second launch of the
// same kernel folds them in index order.  No floating-point atomics anywhere.
#include <algorithm>
#include <cstdlib>
#include <type_traits>

#include "common.cuh"
#include "math.cuh"

namespace tnn {

template <int RED, typename T>
__device__ __forceinline__ T red_identity() {
  if constexpr (RED == TNN_RED_SUM) return T(0);
  else if constexpr (RED == TNN_RED_MAX) return -INFINITY;
  else return INFINITY;
}

template <int RED, typename T>
__device__ __forceinline__ T red_op(T a, T b) {
  if constexpr (RED == TNN_RED_SUM) return a + b;
  else if constexpr (RED == TNN_RED_MAX) return m_max(a, b);
  else return m_min(a, b);
}

template <int RED, typename T>
__device__ __forceinline__ T warp_reduce(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = red_op<RED, T>(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

template <int RED, typename T>
__device__ __forceinline__ T block_reduce_256(T v) {
  __shared__ T sm[8];
  v = warp_reduce<RED, T>(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  if (lane == 0) sm[w] = v;
  __syncthreads();
  T r = red_identity<RED, T>();
  if (w == 0) {
    r = lane < 8 ? sm[lane] : red_identity<RED, T>();
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) r = red_op<RED, T>(r, __shfl_xor_sync(0xffffffffu, r, o));
  }
  __syncthreads();
  return r;  // valid in warp 0
}

// ---- inner == 1, long rows: one CTA per (row, chunk) -----------------------------------------
template <int RED, typename T>
__global__ void __launch_bounds__(256)
reduce_row_block_kernel(T* out, const T* x, int64_t red, int nsplit) {
  const int64_t o = blockIdx.x;
  const int s = blockIdx.y;
  const int64_t chunk = ceil_div(red, nsplit);
  const int64_t lo = (int64_t)s * chunk;
  int64_t hi = lo + chunk;
  if (hi > red) hi = red;
  const T* row = x + o * red;
  T acc = red_identity<RED, T>();
  // four independent accumulators keep several loads in flight per thread
  T a0 = acc, a1 = acc, a2 = acc, a3 = acc;
  int64_t i = lo + threadIdx.x;
  for (; i + 768 < hi; i += 1024) {
    T v0 = row[i], v1 = row[i + 256], v2 = row[i + 512], v3 = row[i + 768];
    a0 = red_op<RED, T>(a0, v0);
    a1 = red_op<RED, T>(a1, v1);
    a2 = red_op<RED, T>(a2, v2);
    a3 = red_op<RED, T>(a3, v3);
  }
  for (; i < hi; i += 256) a0 = red_op<RED, T>(a0, row[i]);
  acc = red_op<RED, T>(red_op<RED, T>(a0, a1), red_op<RED, T>(a2, a3));
  acc = block_reduce_256<RED, T>(acc);
  if (threadIdx.x == 0) out[o * nsplit + s] = acc;
}

// ---- inner == 1, short rows: one warp per row --------------------------------------------------
template <int RED, typename T>
__global__ void __launch_bounds__(256)
reduce_row_warp_kernel(T* out, const T* x, int64_t outer, int64_t red) {
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (int64_t)gridDim.x * 8;
  for (int64_t o = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); o < outer; o += warps_total) {
    const T* row = x + o * red;
    T acc = red_identity<RED, T>();
    for (int64_t i = lane; i < red; i += 32) acc = red_op<RED, T>(acc, row[i]);
    acc = warp_reduce<RED, T>(acc);
    if (lane == 0) out[o] = acc;
  }
}

// ---- inner > 1: a CTA owns 32 column slots (128-bit each when vectorised) x a chunk of rows ------
// thread (tx, ty) of the 32 x 8 block walks rows lo+ty, lo+ty+8, ... of its column slot (coalesced
// across tx), the 8 row lanes are folded through shared memory in fixed order.
// rows lo+ty, lo+ty+8, ... < hi of one column slot, 8 independent loads in flight per thread (small
// reductions are a handful of DRAM round trips: the fewer, the better), combined in row order
template <int RED, typename T, int VEC>
__device__ __forceinline__ void col_accumulate(const T* __restrict__ base, int64_t lo, int64_t hi,
                                               int64_t inner, int ty, T (&acc)[VEC]) {
  using V = Pack<T, VEC>;
  int64_t r = lo + ty;
  for (; r + 56 < hi; r += 64) {
    V u[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) u[i] = *reinterpret_cast<const V*>(base + (r + 8 * i) * inner);
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[k] = red_op<RED, T>(acc[k], u[i].v[k]);
  }
  if (r < hi) {
    // the tail as ONE more batch of predicated loads (a serial tail would be up to seven exposed DRAM
    // round trips -- most of the time of a 64 MB reduction)
    V u[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (r + 8 * i < hi) u[i] = *reinterpret_cast<const V*>(base + (r + 8 * i) * inner);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (r + 8 * i < hi) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[k] = red_op<RED, T>(acc[k], u[i].v[k]);
      }
  }
}

// One launch also when the rows are split across CTAs: every CTA parks its partial in `stage`, and
// the LAST one to arrive for a column block (a counter per block, reset by that CTA) folds the
// nsplit partials -- always in split order, so the result does not depend on which CTA folds.
template <int RED, typename T, int VEC>
__global__ void __launch_bounds__(256)
reduce_col_kernel(T* out, T* stage, const T* x, int64_t red, int64_t inner, int nsplit,
                  unsigned int* counters) {
  __shared__ T sm[8][32 * VEC + 1];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t ncol = inner / VEC;
  const int64_t col = (int64_t)blockIdx.x * 32 + tx;
  const int64_t o = blockIdx.y / nsplit;
  const int s = blockIdx.y % nsplit;
  const int64_t chunk = ceil_div(red, nsplit);
  const int64_t lo = (int64_t)s * chunk;
  int64_t hi = lo + chunk;
  if (hi > red) hi = red;
  T acc[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) acc[k] = red_identity<RED, T>();
  if (col < ncol) col_accumulate<RED, T, VEC>(x + (o * red) * inner + col * VEC, lo, hi, inner, ty, acc);
#pragma unroll
  for (int k = 0; k < VEC; ++k) sm[ty][tx * VEC + k] = acc[k];
  __syncthreads();
  T* dst1 = nsplit > 1 ? stage + ((o * nsplit + s) * inner) : out + o * inner;
  if (ty == 0 && col < ncol) {
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      T r = sm[0][tx * VEC + k];
#pragma unroll
      for (int j = 1; j < 8; ++j) r = red_op<RED, T>(r, sm[j][tx * VEC + k]);
      dst1[col * VEC + k] = r;
    }
  }
  if (nsplit == 1) return;
  // ---- last CTA of this column block folds the partials ----
  if (!col_fold_last_arrival(counters + o * gridDim.x + blockIdx.x, (unsigned int)nsplit)) return;
#pragma unroll
  for (int k = 0; k < VEC; ++k) acc[k] = red_identity<RED, T>();
  if (col < ncol)
    col_accumulate<RED, T, VEC>(stage + (o * nsplit) * inner + col * VEC, 0, nsplit, inner, ty, acc);
  __syncthreads();
#pragma unroll
  for (int k = 0; k < VEC; ++k) sm[ty][tx * VEC + k] = acc[k];
  __syncthreads();
  if (ty == 0 && col < ncol) {
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      T r = sm[0][tx * VEC + k];
#pragma unroll
      for (int j = 1; j < 8; ++j) r = red_op<RED, T>(r, sm[j][tx * VEC + k]);
      out[o * inner + col * VEC + k] = r;
    }
  }
}

static unsigned int* g_col_counters = nullptr;     // one per (outer, column block), zero between launches

int col_fold_counters(unsigned int** out) {
  if (!g_col_counters) {
    TNN_CUDA(cudaMalloc(&g_col_counters, MAX_COL_COUNTERS * sizeof(unsigned int)));
    TNN_CUDA(cudaMemsetAsync(g_col_counters, 0, MAX_COL_COUNTERS * sizeof(unsigned int), ctx().stream));
  }
  *out = g_col_counters;
  return 0;
}

// dtype: T's code, which the fill of an empty reduction takes
template <int RED, typename T>
static int reduce_impl(int dtype, T* out, const T* x, int64_t outer, int64_t red, int64_t inner) {
  Context& c = ctx();
  cudaStream_t st = c.stream;
  if (outer * inner == 0) return 0;
  if (red == 0) {
    // numpy: sum over an empty axis is 0; max/min raise -- mirror that
    if (RED != TNN_RED_SUM) TNN_FAIL("tnn_reduce: zero-size reduction has no identity");
    return tnn_fill(dtype, out, 0.0, outer * inner);
  }
  const int64_t target_ctas = (int64_t)c.sm_count * 4;
  if (inner == 1) {
    if (red <= 2048 && outer >= 64) {
      int grid = (int)std::min<int64_t>(ceil_div(outer, 8), (int64_t)c.sm_count * 8);
      reduce_row_warp_kernel<RED, T><<<grid, 256, 0, st>>>(out, x, outer, red);
      TNN_POST_LAUNCH();
      return 0;
    }
    // CTA per (row, chunk); chunks of at least 4096 elements
    int64_t nsplit = 1;
    if (outer < target_ctas) {
      nsplit = std::min<int64_t>(ceil_div(target_ctas, outer), ceil_div(red, 4096));
      if (nsplit < 1) nsplit = 1;
      if (nsplit > 65535) nsplit = 65535;
    }
    if (outer > 2147483647LL) TNN_FAIL("tnn_reduce: too many rows");
    if (nsplit == 1) {
      reduce_row_block_kernel<RED, T><<<dim3((unsigned)outer, 1), 256, 0, st>>>(out, x, red, 1);
      TNN_POST_LAUNCH();
      return 0;
    }
    void* scratch;
    if (get_scratch((size_t)(outer * nsplit) * sizeof(T), &scratch)) return 1;
    reduce_row_block_kernel<RED, T>
        <<<dim3((unsigned)outer, (unsigned)nsplit), 256, 0, st>>>((T*)scratch, x, red, (int)nsplit);
    TNN_POST_LAUNCH();
    // fold the partials: (outer, nsplit) -> (outer)
    if (outer >= 64) {
      int grid = (int)std::min<int64_t>(ceil_div(outer, 8), (int64_t)c.sm_count * 8);
      reduce_row_warp_kernel<RED, T><<<grid, 256, 0, st>>>(out, (const T*)scratch, outer, nsplit);
    } else {
      reduce_row_block_kernel<RED, T>
          <<<dim3((unsigned)outer, 1), 256, 0, st>>>(out, (const T*)scratch, nsplit, 1);
    }
    TNN_POST_LAUNCH();
    return 0;
  }
  // inner > 1
  constexpr int VW = 16 / sizeof(T);
  bool vec = (inner % VW == 0) && aligned16(x);
  int64_t ncol = vec ? inner / VW : inner;
  int64_t gx = ceil_div(ncol, 32);
  int64_t nsplit = 1;
  // small inputs (the bias gradients of the MNIST-sized layers: 128 x 200 and below) are bound by
  // launch latency, not bandwidth: one stage, one launch
  if (gx * outer < target_ctas && outer * red * inner > (int64_t(1) << 18)) {
    // CTAs per SM for the split (each at least 64 rows).  Measured on (2^24 / 1024, 1024) -> (1, 1024),
    // graph-replayed over rotating buffers: 1 -> 17.8 us, 2 -> 15.3, 3 -> 14.9, 4 -> 15.7, 8 -> 18.2,
    // 16 -> 18.5 (more partials make the last-block fold longer; fewer starve the load pipeline)
    static int col_ctas_per_sm = -1;
    if (col_ctas_per_sm < 0) {
      const char* e = getenv("TNN_COLSUM_CTAS_PER_SM");
      col_ctas_per_sm = e ? atoi(e) : 3;
      if (col_ctas_per_sm < 1) col_ctas_per_sm = 1;
    }
    const int64_t want = (int64_t)c.sm_count * col_ctas_per_sm;
    nsplit = std::min<int64_t>(ceil_div(want, gx * outer), ceil_div(red, 64));
    if (nsplit < 1) nsplit = 1;
  }
  if (outer * nsplit > 65535) {
    nsplit = std::max<int64_t>(1, 65535 / outer);
    if (outer > 65535) TNN_FAIL("tnn_reduce: outer extent above 65535 with inner > 1 is not supported");
  }
  void* scratch = nullptr;
  if (nsplit > 1) {
    if (gx * outer > MAX_COL_COUNTERS) nsplit = 1;
    else if (get_scratch((size_t)(outer * nsplit * inner) * sizeof(T), &scratch)) return 1;
  }
  unsigned int* counters = nullptr;
  if (nsplit > 1 && col_fold_counters(&counters)) return 1;
  dim3 grid((unsigned)gx, (unsigned)(outer * nsplit));
  with_bool(vec, [&](auto V) {
    reduce_col_kernel<RED, T, V ? VW : 1><<<grid, 256, 0, st>>>(out, (T*)scratch, x, red, inner, (int)nsplit,
                                                                counters);
  });
  TNN_POST_LAUNCH();
  return 0;
}

}  // namespace tnn

using namespace tnn;

extern "C" {

int tnn_reduce(int red_op_code, int dtype, void* out, const void* x, int64_t outer, int64_t red,
               int64_t inner) {
  TNN_REQUIRE_INIT();
  if (outer < 0 || red < 0 || inner < 0) TNN_FAIL("tnn_reduce: negative extent");
  return with_float_type(dtype, "tnn_reduce", [&](auto tag) {
    using T = decltype(tag);
    switch (red_op_code) {
      case TNN_RED_SUM: return reduce_impl<TNN_RED_SUM>(dtype, (T*)out, (const T*)x, outer, red, inner);
      case TNN_RED_MAX: return reduce_impl<TNN_RED_MAX>(dtype, (T*)out, (const T*)x, outer, red, inner);
      case TNN_RED_MIN: return reduce_impl<TNN_RED_MIN>(dtype, (T*)out, (const T*)x, outer, red, inner);
    }
    TNN_FAIL("tnn_reduce: unknown reduction code");
  });
}

int tnn_colsum(int dtype, void* out, const void* g, int64_t R, int64_t C) {
  return tnn_reduce(TNN_RED_SUM, dtype, out, g, 1, R, C);
}

int tnn_unbroadcast(int dtype, void* out, const void* grad, int ndim, const int64_t* gshape,
                    const int32_t* keep) {
  TNN_REQUIRE_INIT();
  if (ndim < 0 || ndim > TNN_MAX_DIMS) TNN_FAIL("tnn_unbroadcast: rank above TNN_MAX_DIMS");
  size_t esz = 0;
  if (with_float_type(dtype, "tnn_unbroadcast", [&](auto tag) { esz = sizeof(tag); return 0; })) return 1;
  // collapse into alternating groups; size-1 axes vanish (summing them is the identity)
  int64_t dims[TNN_MAX_DIMS];
  int kp[TNN_MAX_DIMS];
  int n = 0;
  for (int d = 0; d < ndim; ++d) {
    if (gshape[d] == 1) continue;
    int k = keep[d] ? 1 : 0;
    if (n > 0 && kp[n - 1] == k) dims[n - 1] *= gshape[d];
    else {
      dims[n] = gshape[d];
      kp[n] = k;
      ++n;
    }
  }
  int64_t total = 1;
  for (int i = 0; i < n; ++i) total *= dims[i];
  // repeatedly fold the first reduced group
  const void* cur = grad;
  void* tmp_prev = nullptr;
  while (true) {
    int g = -1;
    for (int i = 0; i < n; ++i)
      if (!kp[i]) {
        g = i;
        break;
      }
    if (g < 0) {
      int rc = 0;
      if (cur != out) rc = tnn_d2d(out, cur, (size_t)total * esz);
      if (tmp_prev) tnn_free(tmp_prev);
      return rc;
    }
    int64_t outer = 1, inner = 1;
    for (int i = 0; i < g; ++i) outer *= dims[i];
    for (int i = g + 1; i < n; ++i) inner *= dims[i];
    bool last = true;
    for (int i = g + 1; i < n; ++i)
      if (!kp[i]) last = false;
    void* dst = out;
    void* tmp = nullptr;
    if (!last) {
      if (tnn_alloc((size_t)(outer * inner) * esz, &tmp)) return 1;
      dst = tmp;
    }
    int rc = tnn_reduce(TNN_RED_SUM, dtype, dst, cur, outer, dims[g], inner);
    if (tmp_prev) tnn_free(tmp_prev);
    if (rc) {
      if (tmp) tnn_free(tmp);
      return rc;
    }
    if (last) return 0;
    tmp_prev = tmp;
    cur = tmp;
    total /= dims[g];
    // drop group g and merge its neighbours (both kept)
    for (int i = g; i + 1 < n; ++i) {
      dims[i] = dims[i + 1];
      kp[i] = kp[i + 1];
    }
    --n;
    if (g > 0 && g < n && kp[g - 1] == kp[g]) {
      dims[g - 1] *= dims[g];
      for (int i = g; i + 1 < n; ++i) {
        dims[i] = dims[i + 1];
        kp[i] = kp[i + 1];
      }
      --n;
    }
  }
}

}  // extern "C"

// Elementwise kernels with numpy broadcasting: the forward values and gradient products of
// core/ops.py:32-249, 293-299, 333-344 of the reference (add_, mul_, div_, pow_, maximum_,
// minimum_, exp_, log_, neg_, clip_ and the comparison operators of core/tensor.py:48-58), and the
// forward and backward passes of the LeakyReLU, ELU, GELU, Softplus and SiLU layers.
//
// HBM-bound.  Three launch shapes, chosen on the host after collapsing adjacent axes:
//   flat  : every operand contiguous (or one element)  -> 128-bit vector loads, grid-stride
//   rows  : (R, C) output, operands full / row-vector / column-vector / scalar (bias add,
//           CE scalar broadcast) -> a thread owns a 128-bit column slot and walks down rows
//   nd    : anything else, up to 8 collapsed axes, index arithmetic per element
// Grids are multiples of the SM count (common.cuh: ew_grid).
#include "common.cuh"
#include "math.cuh"

namespace tnn {

template <typename T>
struct EwParams {
  T p0, p1;
  int flags;
};

template <int OP, typename T>
__device__ __forceinline__ T ew_apply(T x, T y, T z, const EwParams<T>& p) {
  if constexpr (OP == TNN_OP_ADD) return x + y;
  else if constexpr (OP == TNN_OP_SUB) return x - y;
  else if constexpr (OP == TNN_OP_MUL) return x * y;
  else if constexpr (OP == TNN_OP_DIV || OP == TNN_OP_RECIP_MUL) return x / y;
  else if constexpr (OP == TNN_OP_POW) return m_pow(x, y);
  else if constexpr (OP == TNN_OP_MAXIMUM) return m_max(x, y);
  else if constexpr (OP == TNN_OP_MINIMUM) return m_min(x, y);
  else if constexpr (OP == TNN_OP_GE) return x >= y ? T(1) : T(0);
  else if constexpr (OP == TNN_OP_GT) return x > y ? T(1) : T(0);
  else if constexpr (OP == TNN_OP_LE) return x <= y ? T(1) : T(0);
  else if constexpr (OP == TNN_OP_LT) return x < y ? T(1) : T(0);
  else if constexpr (OP == TNN_OP_EQ) return x == y ? T(1) : T(0);
  else if constexpr (OP == TNN_OP_MUL_GE) return y >= z ? x : x * T(0);
  else if constexpr (OP == TNN_OP_MUL_GT) return y > z ? x : x * T(0);
  else if constexpr (OP == TNN_OP_MUL_LE) return y <= z ? x : x * T(0);
  else if constexpr (OP == TNN_OP_MUL_LT) return y < z ? x : x * T(0);
  else if constexpr (OP == TNN_OP_MUL_EQ) return y == z ? x : x * T(0);
  else if constexpr (OP == TNN_OP_DIV_BWD_B) return ((-x) * y) / (z * z);
  else if constexpr (OP == TNN_OP_POW_BWD_A) return (x * z) * m_pow(y, z - T(1));
  else if constexpr (OP == TNN_OP_POW_BWD_B) return x * (m_log(y) * z);
  else if constexpr (OP == TNN_OP_NEG) return -x;
  else if constexpr (OP == TNN_OP_EXP) return m_exp(x);
  else if constexpr (OP == TNN_OP_LOG) return m_log(x);
  else if constexpr (OP == TNN_OP_COPY) return x;
  else if constexpr (OP == TNN_OP_CLIP) {
    T r = x;
    if (p.flags & 1) r = m_max(r, p.p0);
    if (p.flags & 2) r = m_min(r, p.p1);
    return r;
  } else if constexpr (OP == TNN_OP_SCALE) return x * p.p0 + p.p1;
  else if constexpr (OP == TNN_OP_CLIP_BWD) {
    bool m = true;
    if (p.flags & 1) m = m && (y >= p.p0);
    if (p.flags & 2) m = m && (y <= p.p1);
    return m ? x : x * T(0);
  }
  // activations (math.cuh): forward f(x); backward x = upstream gradient, y = the activation's input
  else if constexpr (OP == TNN_OP_LEAKY_RELU) return act_leaky_relu(x, p.p0);
  else if constexpr (OP == TNN_OP_ELU) return act_elu(x, p.p0);
  else if constexpr (OP == TNN_OP_GELU) return act_gelu(x);
  else if constexpr (OP == TNN_OP_GELU_TANH) return act_gelu_tanh(x);
  else if constexpr (OP == TNN_OP_SOFTPLUS) return act_softplus(x);
  else if constexpr (OP == TNN_OP_SILU) return act_silu(x);
  else if constexpr (OP == TNN_OP_LEAKY_RELU_BWD) return act_leaky_relu_bwd(x, y, p.p0);
  else if constexpr (OP == TNN_OP_ELU_BWD) return act_elu_bwd(x, y, p.p0);
  else if constexpr (OP == TNN_OP_GELU_BWD) return act_gelu_bwd(x, y);
  else if constexpr (OP == TNN_OP_GELU_TANH_BWD) return act_gelu_tanh_bwd(x, y);
  else if constexpr (OP == TNN_OP_SOFTPLUS_BWD) return act_softplus_bwd(x, y);
  else if constexpr (OP == TNN_OP_SILU_BWD) return act_silu_bwd(x, y);
  else return x;
}

// codes below 20 and from TNN_OP_LEAKY_RELU_BWD up are binary, 20..39 ternary, 40..59 unary
// except the two binary codes among them
__host__ __device__ constexpr int op_arity(int op) {
  if (op >= 20 && op < 40) return 3;
  if (op < 20 || op >= TNN_OP_LEAKY_RELU_BWD || op == TNN_OP_CLIP_BWD || op == TNN_OP_RECIP_MUL) return 2;
  return 1;
}

// ---- flat ------------------------------------------------------------------------------------
template <int OP, typename T>
__global__ void __launch_bounds__(256)
ew_flat_vec_kernel(T* out, const T* x, const T* y, const T* z, int64_t n, int scalar_mask,
                   EwParams<T> p) {
  constexpr int VEC = 16 / sizeof(T);
  constexpr int AR = op_arity(OP);
  using V = Pack<T, VEC>;
  const int64_t nv = n / VEC;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const bool xs = scalar_mask & 1, ys = scalar_mask & 2, zs = scalar_mask & 4;
  T x0 = xs ? x[0] : T(0);
  T y0 = (AR >= 2 && ys) ? y[0] : T(0);
  T z0 = (AR >= 3 && zs) ? z[0] : T(0);
  constexpr int U = AR == 1 ? 4 : 2;   // independent vector loads in flight per operand and thread
  for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < nv; i0 += U * stride) {
    V a[U], b[U], c[U], r;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < nv) {
        if (!xs) a[u] = reinterpret_cast<const V*>(x)[i];
        if (AR >= 2 && !ys) b[u] = reinterpret_cast<const V*>(y)[i];
        if (AR >= 3 && !zs) c[u] = reinterpret_cast<const V*>(z)[i];
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < nv) {
#pragma unroll
        for (int k = 0; k < VEC; ++k)
          r.v[k] = ew_apply<OP, T>(xs ? x0 : a[u].v[k], (AR >= 2) ? (ys ? y0 : b[u].v[k]) : T(0),
                                   (AR >= 3) ? (zs ? z0 : c[u].v[k]) : T(0), p);
        reinterpret_cast<V*>(out)[i] = r;
      }
    }
  }
  // tail (n not a multiple of VEC)
  int64_t t = nv * VEC + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n)
    out[t] = ew_apply<OP, T>(xs ? x0 : x[t], (AR >= 2) ? (ys ? y0 : y[t]) : T(0),
                             (AR >= 3) ? (zs ? z0 : z[t]) : T(0), p);
}

template <int OP, typename T>
__global__ void __launch_bounds__(256)
ew_flat_scalar_kernel(T* out, const T* x, const T* y, const T* z, int64_t n, int scalar_mask,
                      EwParams<T> p) {
  constexpr int AR = op_arity(OP);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const bool xs = scalar_mask & 1, ys = scalar_mask & 2, zs = scalar_mask & 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = ew_apply<OP, T>(x[xs ? 0 : i], (AR >= 2) ? y[ys ? 0 : i] : T(0),
                             (AR >= 3) ? z[zs ? 0 : i] : T(0), p);
}

// ---- rows: out (R, C); operand strides (rs, cs) with cs in {0,1} --------------------------------
struct RowsArgs {
  int64_t R, C;
  int64_t rs[3], cs[3];
};

template <int OP, typename T, bool VECTOR>
__global__ void __launch_bounds__(256)
ew_rows_kernel(T* out, const T* x, const T* y, const T* z, RowsArgs a, EwParams<T> p) {
  constexpr int VEC = VECTOR ? 16 / sizeof(T) : 1;
  constexpr int AR = op_arity(OP);
  const int64_t ncol = a.C / VEC;  // VECTOR path requires C % VEC == 0
  const int64_t col = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncol) return;
  const int64_t c0 = col * VEC;
  const T* ptr[3] = {x, y, z};
  T keep[3][VEC];  // operands that do not vary down the rows are loaded once
#pragma unroll
  for (int o = 0; o < AR; ++o)
    if (a.rs[o] == 0) {
#pragma unroll
      for (int k = 0; k < VEC; ++k) keep[o][k] = ptr[o][(c0 + k) * a.cs[o]];
    }
  for (int64_t r = blockIdx.y; r < a.R; r += gridDim.y) {
    T v[3][VEC];
#pragma unroll
    for (int o = 0; o < 3; ++o) {
      if (o >= AR) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[o][k] = T(0);
      } else if (a.rs[o] == 0) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[o][k] = keep[o][k];
      } else if (a.cs[o] == 0) {
        T s = ptr[o][r * a.rs[o]];
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[o][k] = s;
      } else if (VECTOR) {
        const Pack<T, VEC> u = *reinterpret_cast<const Pack<T, VEC>*>(ptr[o] + r * a.rs[o] + c0);
#pragma unroll
        for (int k = 0; k < VEC; ++k) v[o][k] = u.v[k];
      } else {
        v[o][0] = ptr[o][r * a.rs[o] + c0];
      }
    }
    if (VECTOR) {
      Pack<T, VEC> u;
#pragma unroll
      for (int k = 0; k < VEC; ++k) u.v[k] = ew_apply<OP, T>(v[0][k], v[1][k], v[2][k], p);
      *reinterpret_cast<Pack<T, VEC>*>(out + r * a.C + c0) = u;
    } else {
      out[r * a.C + c0] = ew_apply<OP, T>(v[0][0], v[1][0], v[2][0], p);
    }
  }
}

// ---- nd ----------------------------------------------------------------------------------------
struct NdArgs {
  int ndim;
  int64_t shape[TNN_MAX_DIMS];
  int64_t st[3][TNN_MAX_DIMS];
};

template <int OP, typename T>
__global__ void __launch_bounds__(256)
ew_nd_kernel(T* out, const T* x, const T* y, const T* z, int64_t n, NdArgs a, EwParams<T> p) {
  constexpr int AR = op_arity(OP);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    int64_t rem = i, off[3] = {0, 0, 0};
#pragma unroll 1
    for (int d = a.ndim - 1; d >= 0; --d) {
      int64_t q = rem / a.shape[d];
      int64_t c = rem - q * a.shape[d];
      rem = q;
      off[0] += c * a.st[0][d];
      if (AR >= 2) off[1] += c * a.st[1][d];
      if (AR >= 3) off[2] += c * a.st[2][d];
    }
    out[i] = ew_apply<OP, T>(x[off[0]], (AR >= 2) ? y[off[1]] : T(0), (AR >= 3) ? z[off[2]] : T(0), p);
  }
}

// ---- host dispatch -------------------------------------------------------------------------
template <int OP, typename T>
static int launch_flat(T* out, const T* x, const T* y, const T* z, int64_t n, int scalar_mask,
                       EwParams<T> p) {
  if (n <= 0) return 0;
  constexpr int AR = op_arity(OP);
  constexpr int VEC = 16 / sizeof(T);
  bool vec_ok = aligned16(out) && n >= VEC;
  if (!(scalar_mask & 1)) vec_ok = vec_ok && aligned16(x);
  if (AR >= 2 && !(scalar_mask & 2)) vec_ok = vec_ok && aligned16(y);
  if (AR >= 3 && !(scalar_mask & 4)) vec_ok = vec_ok && aligned16(z);
  cudaStream_t s = ctx().stream;
  if (vec_ok) {
    int grid = ew_grid(ceil_div(n, VEC), 256);
    ew_flat_vec_kernel<OP, T><<<grid, 256, 0, s>>>(out, x, y, z, n, scalar_mask, p);
  } else {
    int grid = ew_grid(n, 256);
    ew_flat_scalar_kernel<OP, T><<<grid, 256, 0, s>>>(out, x, y, z, n, scalar_mask, p);
  }
  TNN_POST_LAUNCH();
  return 0;
}

template <int OP, typename T>
static int launch_rows(T* out, const T* x, const T* y, const T* z, const RowsArgs& a,
                       EwParams<T> p) {
  constexpr int AR = op_arity(OP);
  constexpr int VEC = 16 / sizeof(T);
  const T* ptr[3] = {x, y, z};
  bool vec_ok = (a.C % VEC == 0) && aligned16(out);
  for (int o = 0; o < AR; ++o)
    if (a.cs[o] == 1) vec_ok = vec_ok && aligned16(ptr[o]) && (a.rs[o] % VEC == 0);
  int64_t ncol = vec_ok ? a.C / VEC : a.C;
  int gx = (int)ceil_div(ncol, 256);
  int64_t want_y = ceil_div((int64_t)ctx().sm_count * 8, gx);
  int gy = (int)(want_y < 1 ? 1 : (want_y > a.R ? a.R : want_y));
  if (gy > 65535) gy = 65535;
  dim3 grid(gx, gy);
  with_bool(vec_ok, [&](auto vec) { ew_rows_kernel<OP, T, vec><<<grid, 256, 0, ctx().stream>>>(out, x, y, z, a, p); });
  TNN_POST_LAUNCH();
  return 0;
}

template <int OP, typename T>
static int launch_nd(T* out, const T* x, const T* y, const T* z, int64_t n, const NdArgs& a,
                     EwParams<T> p) {
  int grid = ew_grid(n, 256);
  ew_nd_kernel<OP, T><<<grid, 256, 0, ctx().stream>>>(out, x, y, z, n, a, p);
  TNN_POST_LAUNCH();
  return 0;
}

template <int OP, typename T>
static int ew_dispatch(void* out, const void* x, const void* y, const void* z, int ndim,
                       const int64_t* shape, const int64_t* xs, const int64_t* ys,
                       const int64_t* zs, double p0, double p1, int flags) {
  constexpr int AR = op_arity(OP);
  EwParams<T> p{(T)p0, (T)p1, flags};
  const int64_t* st_in[3] = {xs, ys, zs};
  // collapse: drop size-1 axes, merge neighbours whose strides nest for every operand
  int64_t cs[TNN_MAX_DIMS];
  int64_t cst[3][TNN_MAX_DIMS];
  int nd = 0;
  int64_t total = 1;
  for (int d = 0; d < ndim; ++d) {
    if (shape[d] < 0) TNN_FAIL("tnn_ew: negative dimension");
    total *= shape[d];
  }
  if (total == 0) return 0;
  for (int d = 0; d < ndim; ++d) {
    if (shape[d] == 1) continue;
    bool merged = false;
    if (nd > 0) {
      bool ok = true;
      for (int o = 0; o < AR; ++o)
        if (cst[o][nd - 1] != st_in[o][d] * shape[d]) ok = false;
      if (ok) {
        cs[nd - 1] *= shape[d];
        for (int o = 0; o < AR; ++o) cst[o][nd - 1] = st_in[o][d];
        merged = true;
      }
    }
    if (!merged) {
      cs[nd] = shape[d];
      for (int o = 0; o < 3; ++o) cst[o][nd] = (o < AR) ? st_in[o][d] : 0;
      ++nd;
    }
  }
  if (nd == 0) {  // single element
    nd = 1;
    cs[0] = 1;
    for (int o = 0; o < 3; ++o) cst[o][0] = 0;
  }
  const T* X = (const T*)x;
  const T* Y = (const T*)y;
  const T* Z = (const T*)z;
  if (nd == 1) {
    bool ok = true;
    int mask = 0;
    for (int o = 0; o < AR; ++o) {
      if (cst[o][0] == 0) mask |= (1 << o);
      else if (cst[o][0] != 1) ok = false;
    }
    if (cs[0] == 1) mask = 7;
    if (ok) return launch_flat<OP, T>((T*)out, X, Y, Z, cs[0], mask, p);
  }
  if (nd == 2) {
    bool ok = true;
    RowsArgs a;
    a.R = cs[0];
    a.C = cs[1];
    for (int o = 0; o < 3; ++o) {
      a.rs[o] = cst[o][0];
      a.cs[o] = cst[o][1];
      if (o < AR && !(a.cs[o] == 0 || a.cs[o] == 1)) ok = false;
    }
    if (ok) return launch_rows<OP, T>((T*)out, X, Y, Z, a, p);
  }
  NdArgs a;
  a.ndim = nd;
  for (int d = 0; d < TNN_MAX_DIMS; ++d) {
    a.shape[d] = d < nd ? cs[d] : 1;
    for (int o = 0; o < 3; ++o) a.st[o][d] = d < nd ? cst[o][d] : 0;
  }
  return launch_nd<OP, T>((T*)out, X, Y, Z, total, a, p);
}

template <int OP, typename T>
static int ew_flat_dispatch(void* out, const void* x, const void* y, const void* z, int64_t n,
                            int scalar_mask, double p0, double p1, int flags) {
  EwParams<T> p{(T)p0, (T)p1, flags};
  return launch_flat<OP, T>((T*)out, (const T*)x, (const T*)y, (const T*)z, n, scalar_mask, p);
}

// cast / fill
template <typename D, typename S>
__global__ void __launch_bounds__(256) cast_kernel(D* dst, const S* src, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dst[i] = (D)src[i];
}

template <typename T>
__global__ void __launch_bounds__(256) fill_kernel(T* dst, T v, int64_t n) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) dst[i] = v;
}

// f(std::integral_constant<int, OP>{}) for an op code; any other code fails, naming the entry point
#define TNN_EW_CASE(OPC) \
  case OPC:              \
    return f(std::integral_constant<int, OPC>{});

template <typename F>
static int with_op(int op, const char* name, F&& f) {
  switch (op) {
    TNN_EW_CASE(TNN_OP_ADD)
    TNN_EW_CASE(TNN_OP_SUB)
    TNN_EW_CASE(TNN_OP_MUL)
    TNN_EW_CASE(TNN_OP_DIV)
    TNN_EW_CASE(TNN_OP_POW)
    TNN_EW_CASE(TNN_OP_MAXIMUM)
    TNN_EW_CASE(TNN_OP_MINIMUM)
    TNN_EW_CASE(TNN_OP_GE)
    TNN_EW_CASE(TNN_OP_GT)
    TNN_EW_CASE(TNN_OP_LE)
    TNN_EW_CASE(TNN_OP_LT)
    TNN_EW_CASE(TNN_OP_EQ)
    TNN_EW_CASE(TNN_OP_MUL_GE)
    TNN_EW_CASE(TNN_OP_MUL_GT)
    TNN_EW_CASE(TNN_OP_MUL_LE)
    TNN_EW_CASE(TNN_OP_MUL_LT)
    TNN_EW_CASE(TNN_OP_MUL_EQ)
    TNN_EW_CASE(TNN_OP_DIV_BWD_B)
    TNN_EW_CASE(TNN_OP_POW_BWD_A)
    TNN_EW_CASE(TNN_OP_POW_BWD_B)
    TNN_EW_CASE(TNN_OP_NEG)
    TNN_EW_CASE(TNN_OP_EXP)
    TNN_EW_CASE(TNN_OP_LOG)
    TNN_EW_CASE(TNN_OP_COPY)
    TNN_EW_CASE(TNN_OP_CLIP)
    TNN_EW_CASE(TNN_OP_SCALE)
    TNN_EW_CASE(TNN_OP_CLIP_BWD)
    TNN_EW_CASE(TNN_OP_RECIP_MUL)
    TNN_EW_CASE(TNN_OP_LEAKY_RELU)
    TNN_EW_CASE(TNN_OP_ELU)
    TNN_EW_CASE(TNN_OP_GELU)
    TNN_EW_CASE(TNN_OP_GELU_TANH)
    TNN_EW_CASE(TNN_OP_SOFTPLUS)
    TNN_EW_CASE(TNN_OP_SILU)
    TNN_EW_CASE(TNN_OP_LEAKY_RELU_BWD)
    TNN_EW_CASE(TNN_OP_ELU_BWD)
    TNN_EW_CASE(TNN_OP_GELU_BWD)
    TNN_EW_CASE(TNN_OP_GELU_TANH_BWD)
    TNN_EW_CASE(TNN_OP_SOFTPLUS_BWD)
    TNN_EW_CASE(TNN_OP_SILU_BWD)
    default:
      TNN_FAIL(std::string(name) + ": unknown op code " + std::to_string(op));
  }
}
#undef TNN_EW_CASE

}  // namespace tnn

using namespace tnn;

extern "C" {

int tnn_ew(int op, int dtype, void* out, const void* x, const void* y, const void* z, int ndim,
           const int64_t* shape, const int64_t* xs, const int64_t* ys, const int64_t* zs,
           double p0, double p1, int flags) {
  TNN_REQUIRE_INIT();
  if (ndim < 0 || ndim > TNN_MAX_DIMS) TNN_FAIL("tnn_ew: rank above TNN_MAX_DIMS");
  return with_op(op, "tnn_ew", [&](auto OP) {
    return with_float_type(dtype, "tnn_ew", [&](auto tag) {
      return ew_dispatch<OP, decltype(tag)>(out, x, y, z, ndim, shape, xs, ys, zs, p0, p1, flags);
    });
  });
}

int tnn_ew_flat(int op, int dtype, void* out, const void* x, const void* y, const void* z,
                int64_t n, int scalar_mask, double p0, double p1, int flags) {
  TNN_REQUIRE_INIT();
  return with_op(op, "tnn_ew_flat", [&](auto OP) {
    return with_float_type(dtype, "tnn_ew_flat", [&](auto tag) {
      return ew_flat_dispatch<OP, decltype(tag)>(out, x, y, z, n, scalar_mask, p0, p1, flags);
    });
  });
}

int tnn_cast(int dst_dtype, void* dst, int src_dtype, const void* src, int64_t n) {
  TNN_REQUIRE_INIT();
  if (n <= 0) return 0;
  int grid = ew_grid(n, 256);
  cudaStream_t s = ctx().stream;
  if (dst_dtype == TNN_F32 && src_dtype == TNN_F64)
    cast_kernel<float, double><<<grid, 256, 0, s>>>((float*)dst, (const double*)src, n);
  else if (dst_dtype == TNN_F64 && src_dtype == TNN_F32)
    cast_kernel<double, float><<<grid, 256, 0, s>>>((double*)dst, (const float*)src, n);
  else if (dst_dtype == src_dtype && (dst_dtype == TNN_F32 || dst_dtype == TNN_F64))
    return tnn_d2d(dst, src, (size_t)n * (dst_dtype == TNN_F32 ? 4 : 8));
  else
    TNN_FAIL("tnn_cast: unsupported dtype pair");
  TNN_POST_LAUNCH();
  return 0;
}

int tnn_fill(int dtype, void* dst, double value, int64_t n) {
  TNN_REQUIRE_INIT();
  if (n <= 0) return 0;
  return with_float_type(dtype, "tnn_fill", [&](auto tag) {
    using T = decltype(tag);
    fill_kernel<T><<<ew_grid(n, 256), 256, 0, ctx().stream>>>((T*)dst, (T)value, n);
    TNN_POST_LAUNCH();
    return 0;
  });
}

}  // extern "C"

// Fused layer / loss / optimizer kernels.
//
//  * ReLU forward + its `x >= 0` backward mask           layers.py:97-98, ops.py:333-344
//  * SoftmaxCrossEntropyLoss with the reference's batch-GLOBAL max and normaliser
//                                                        losses.py:24-32
//  * SGD / Adam / RMSProp / Momentum / Adagrad / Adadelta on the flat parameter arena
//                                                        optimizer.py:41-164, model.py:45-61
//  * AdamW / RAdam / Adamax, which share Adam's per-element code and 128-bit kernel
// All HBM-bound streaming kernels: 128-bit accesses, grid-stride, grids in multiples of the SM
// count.  Reductions inside the loss are two-stage and deterministic (see reduce.cu).
#include <algorithm>

#include "common.cuh"
#include "math.cuh"

namespace tnn {

// ---- ReLU ------------------------------------------------------------------------------------
// forward: np.clip(x, 0.0, None) = maximum(x, 0) (NaN propagates); backward: g * (x >= 0)
template <typename T, bool BWD, bool VEC>
__global__ void __launch_bounds__(256) relu_kernel(T* out, const T* g, const T* x, int64_t n) {
  constexpr int W = VEC ? 16 / sizeof(T) : 1;
  constexpr int U = 4;   // independent 128-bit loads in flight per thread (a 1-read stream needs them)
  const int64_t nv = n / W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < nv; i0 += U * stride) {
    if constexpr (VEC) {
      using V = Pack<T, W>;
      V a[U], b[U], r;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < nv) {
          a[u] = reinterpret_cast<const V*>(x)[i];
          if (BWD) b[u] = reinterpret_cast<const V*>(g)[i];
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < nv) {
#pragma unroll
          for (int k = 0; k < W; ++k)
            r.v[k] = BWD ? (a[u].v[k] >= T(0) ? b[u].v[k] : b[u].v[k] * T(0)) : m_max(a[u].v[k], T(0));
          reinterpret_cast<V*>(out)[i] = r;
        }
      }
    } else {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < nv) {
          T a = x[i];
          out[i] = BWD ? (a >= T(0) ? g[i] : g[i] * T(0)) : m_max(a, T(0));
        }
      }
    }
  }
  if (VEC) {
    int64_t t = nv * W + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) {
      T a = x[t];
      out[t] = BWD ? (a >= T(0) ? g[t] : g[t] * T(0)) : m_max(a, T(0));
    }
  }
}

template <typename T, bool BWD>
static int relu_launch(T* out, const T* g, const T* x, int64_t n) {
  if (n <= 0) return 0;
  constexpr int W = 16 / sizeof(T);
  const bool vec = aligned16(out) && aligned16(x) && (!BWD || aligned16(g)) && n >= W;
  with_bool(vec, [&](auto V) {
    relu_kernel<T, BWD, V><<<ew_grid(V ? ceil_div(n, W) : n, 256), 256, 0, ctx().stream>>>(out, g, x, n);
  });
  TNN_POST_LAUNCH();
  return 0;
}

// ---- block reduction helpers -------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = m_max(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// all threads of a 256-thread block receive the result
template <typename T, bool IS_MAX>
__device__ __forceinline__ T block_all_reduce(T v, T* sm /* >= 8 */) {
  v = IS_MAX ? warp_max(v) : warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sm[w] = v;
  __syncthreads();
  T r = sm[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) r = IS_MAX ? m_max(r, sm[i]) : r + sm[i];
  return r;
}

// ---- cross entropy: stage 1 (max, sum exp) ----------------------------------------------------
// single-CTA version for small logits matrices (the examples/mnist shape: 128 x 10)
template <typename T>
__global__ void __launch_bounds__(256) ce_stats_small_kernel(const T* z, int64_t n, T* stats) {
  __shared__ T sm[8];
  T mx = -INFINITY;
  for (int64_t i = threadIdx.x; i < n; i += 256) mx = m_max(mx, z[i]);
  mx = block_all_reduce<T, true>(mx, sm);
  T s = T(0);
  for (int64_t i = threadIdx.x; i < n; i += 256) s += m_exp(z[i] - mx);
  s = block_all_reduce<T, false>(s, sm);
  if (threadIdx.x == 0) {
    stats[0] = mx;
    stats[1] = s;
  }
}

template <typename T, bool VEC>
__global__ void __launch_bounds__(256)
ce_partial_max_kernel(const T* z, int64_t n, T* partial) {
  __shared__ T sm[8];
  constexpr int W = VEC ? 16 / sizeof(T) : 1;
  const int64_t nv = n / W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  T mx = -INFINITY;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
    if constexpr (VEC) {
      const Pack<T, W> a = reinterpret_cast<const Pack<T, W>*>(z)[i];
#pragma unroll
      for (int k = 0; k < W; ++k) mx = m_max(mx, a.v[k]);
    } else {
      mx = m_max(mx, z[i]);
    }
  }
  if (VEC && blockIdx.x == 0) {
    int64_t t = nv * W + threadIdx.x;
    if (t < n) mx = m_max(mx, z[t]);
  }
  mx = block_all_reduce<T, true>(mx, sm);
  if (threadIdx.x == 0) partial[blockIdx.x] = mx;
}

// every CTA first folds the per-CTA maxima (identical order everywhere), then sums its share
template <typename T, bool VEC>
__global__ void __launch_bounds__(256)
ce_partial_sumexp_kernel(const T* z, int64_t n, const T* pmax, int n_pmax, T* psum, T* stats) {
  __shared__ T sm[8];
  T mx = -INFINITY;
  for (int i = threadIdx.x; i < n_pmax; i += 256) mx = m_max(mx, pmax[i]);
  mx = block_all_reduce<T, true>(mx, sm);
  constexpr int W = VEC ? 16 / sizeof(T) : 1;
  const int64_t nv = n / W;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  T s = T(0);
  if constexpr (VEC) {
    // four independent 128-bit loads in flight per thread: a one-read stream needs them to reach
    // HBM bandwidth (measured 3.5 TB/s with one)
    constexpr int U = 4;
    for (int64_t i0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i0 < nv; i0 += U * stride) {
      Pack<T, W> a[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t i = i0 + u * stride;
        if (i < nv) a[u] = reinterpret_cast<const Pack<T, W>*>(z)[i];
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (i0 + u * stride < nv) {
#pragma unroll
          for (int k = 0; k < W; ++k) s += m_exp(a[u].v[k] - mx);
        }
      }
    }
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride)
      s += m_exp(z[i] - mx);
  }
  if (VEC && blockIdx.x == 0) {
    int64_t t = nv * W + threadIdx.x;
    if (t < n) s += m_exp(z[t] - mx);
  }
  s = block_all_reduce<T, false>(s, sm);
  if (threadIdx.x == 0) {
    psum[blockIdx.x] = s;
    if (blockIdx.x == 0) stats[0] = mx;
  }
}

template <typename T>
__global__ void __launch_bounds__(256) ce_fold_sum_kernel(const T* psum, int n_psum, T* dst) {
  __shared__ T sm[8];
  T s = T(0);
  for (int i = threadIdx.x; i < n_psum; i += 256) s += psum[i];
  s = block_all_reduce<T, false>(s, sm);
  if (threadIdx.x == 0) dst[0] = s;
}

// merge per-rank (max, sumexp) pairs: M = max M_r, S = sum S_r * exp(M_r - M)
template <typename T>
__global__ void ce_merge_stats_kernel(T* out, const T* all, int n_ranks) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    T mx = -INFINITY;
    for (int r = 0; r < n_ranks; ++r) mx = m_max(mx, all[2 * r]);
    T s = T(0);
    for (int r = 0; r < n_ranks; ++r) s += all[2 * r + 1] * m_exp(all[2 * r] - mx);
    out[0] = mx;
    out[1] = s;
  }
}

// ---- cross entropy: stage 2 (per-row q_i, -ln q_i) ---------------------------------------------
// one warp per row; q_i = sum_j (exp(z_ij - M) / S) * y_ij   (losses.py:27-28)
template <typename T, typename TY>
__global__ void __launch_bounds__(256)
ce_rows_kernel(const T* z, const TY* y, int64_t B, int64_t C, const T* stats, T* q, T* nll) {
  const T mx = stats[0], S = stats[1];
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (int64_t)gridDim.x * 8;
  for (int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); r < B; r += warps_total) {
    const T* zr = z + r * C;
    const TY* yr = y + r * C;
    T acc = T(0);
    for (int64_t j = lane; j < C; j += 32) {
      TY yy = yr[j];
      if (yy != TY(0)) acc += (m_exp(zr[j] - mx) / S) * (T)yy;
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      q[r] = acc;
      nll[r] = -m_log(acc);
    }
  }
}

// wide float32 rows (C a multiple of 4, 16-byte aligned): a lane takes 4 consecutive columns per
// 128-bit load, two row chunks (z and y each) in flight; 8 B/element read at HBM speed
__global__ void __launch_bounds__(256)
ce_rows_vec_kernel(const float* z, const float* y, int64_t B, int64_t C, const float* stats, float* q,
                   float* nll) {
  const float mx = stats[0], S = stats[1];
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (int64_t)gridDim.x * 8;
  const int64_t nv = C / 4;
  for (int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); r < B; r += warps_total) {
    const float4* zr = reinterpret_cast<const float4*>(z + r * C);
    const float4* yr = reinterpret_cast<const float4*>(y + r * C);
    float acc = 0.f;
    for (int64_t j0 = lane; j0 < nv; j0 += 64) {
      const int64_t j1 = j0 + 32;
      const float4 ya = yr[j0], za = zr[j0];
      float4 yb = make_float4(0.f, 0.f, 0.f, 0.f), zb = yb;
      if (j1 < nv) {
        yb = yr[j1];
        zb = zr[j1];
      }
      if (ya.x != 0.f) acc += (m_exp(za.x - mx) / S) * ya.x;
      if (ya.y != 0.f) acc += (m_exp(za.y - mx) / S) * ya.y;
      if (ya.z != 0.f) acc += (m_exp(za.z - mx) / S) * ya.z;
      if (ya.w != 0.f) acc += (m_exp(za.w - mx) / S) * ya.w;
      if (yb.x != 0.f) acc += (m_exp(zb.x - mx) / S) * yb.x;
      if (yb.y != 0.f) acc += (m_exp(zb.y - mx) / S) * yb.y;
      if (yb.z != 0.f) acc += (m_exp(zb.z - mx) / S) * yb.z;
      if (yb.w != 0.f) acc += (m_exp(zb.w - mx) / S) * yb.w;
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      q[r] = acc;
      nll[r] = -m_log(acc);
    }
  }
}

// labels given as class indices (a one-hot y that was never materialised: utils/data_iterator.py ships
// int32 labels and core/_backend.LazyOneHot names the dense rows): q_i = p_{i, label_i} -- the one
// non-zero term of the sums above, so bit-identical to them -- without reading B x C labels
template <typename T>
__global__ void __launch_bounds__(256)
ce_rows_label_kernel(const T* z, const int32_t* labels, int64_t B, int64_t C, const T* stats, T* q, T* nll) {
  const T mx = stats[0], S = stats[1];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < B; r += stride) {
    const int64_t l = labels[r];
    T acc = T(0);
    if (l >= 0 && l < C) acc += (m_exp(z[r * C + l] - mx) / S) * T(1);
    q[r] = acc;
    nll[r] = -m_log(acc);
  }
}

template <typename T>
__global__ void __launch_bounds__(256)
ce_fold_loss_kernel(const T* nll, int64_t B, T m, T* loss) {
  __shared__ T sm[8];
  T s = T(0);
  for (int64_t i = threadIdx.x; i < B; i += 256) s += nll[i];
  s = block_all_reduce<T, false>(s, sm);
  if (threadIdx.x == 0) loss[0] = s / m;
}

// ---- cross entropy forward, whole thing in one CTA (the examples/mnist shape: 128 x 10) ----------
// Same arithmetic, in the same order, as ce_stats_small_kernel -> ce_rows_kernel -> ce_fold_loss_kernel
// (so the value is bit-identical to the three-launch path); 2 launches fewer on a launch-bound step.
constexpr int CE_SMALL_MAX_ROWS = 2048;
// 1024 threads.  The two block-wide sums are taken over the first 256 threads only, in the order
// block_all_reduce uses, so they match the 256-thread staged kernels bit for bit; the per-row pass
// uses all 32 warps, four rows per warp in flight at once (a row per warp at a time would be a
// chain of 16 exposed load latencies for the 128-row MNIST batch).
template <typename T, bool IS_MAX>
__device__ __forceinline__ T block1024_reduce_first8(T v, T* sm /* >= 32 */) {
  v = IS_MAX ? warp_max(v) : warp_sum(v);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) sm[w] = v;
  __syncthreads();
  T r = sm[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) r = IS_MAX ? m_max(r, sm[i]) : r + sm[i];
  return r;
}

constexpr int CE_SMALL_STAGE_BYTES = 16384;   // logits staged in shared memory when they fit (MNIST: 1280 values)
template <typename T, typename TY>
__global__ void __launch_bounds__(1024)
ce_fwd_small_kernel(const T* z, const TY* y, int64_t B, int64_t C, T m, T* stats, T* q, T* loss, T* dz_out) {
  __shared__ T sm[32];
  __shared__ T nll[CE_SMALL_MAX_ROWS];
  constexpr int CE_SMALL_STAGE = CE_SMALL_STAGE_BYTES / (int)sizeof(T);
  __shared__ T zs[CE_SMALL_STAGE];
  const int64_t n = B * C;
  const bool first = threadIdx.x < 256;
  pdl_sync();
  // one trip to global memory for the logits when they fit in shared memory: the max pass, the
  // sum-exp pass and the per-row pass then read the staged copy (three dependent round trips
  // were most of this kernel's 9 us)
  const bool staged = n <= CE_SMALL_STAGE;
  if (staged) {
    for (int64_t i = threadIdx.x; i < n; i += 1024) zs[i] = z[i];
    __syncthreads();
  }
  const T* zz = staged ? zs : z;
  T mx = -INFINITY;
  if (first)
    for (int64_t i = threadIdx.x; i < n; i += 256) mx = m_max(mx, zz[i]);
  mx = block1024_reduce_first8<T, true>(mx, sm);
  T S = T(0);
  if (first)
    for (int64_t i = threadIdx.x; i < n; i += 256) S += m_exp(zz[i] - mx);
  S = block1024_reduce_first8<T, false>(S, sm);
  if (threadIdx.x == 0) {
    stats[0] = mx;
    stats[1] = S;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int RU = 4;
  for (int64_t r0 = warp; r0 < B; r0 += 32 * RU) {
    T acc[RU];
#pragma unroll
    for (int u = 0; u < RU; ++u) {
      const int64_t r = r0 + 32 * u;
      acc[u] = T(0);
      if (r < B) {
        const T* zr = zz + r * C;
        const TY* yr = y + r * C;
        for (int64_t j = lane; j < C; j += 32) {
          TY yy = yr[j];
          if (yy != TY(0)) acc[u] += (m_exp(zr[j] - mx) / S) * (T)yy;
        }
      }
    }
#pragma unroll
    for (int u = 0; u < RU; ++u) {
      const int64_t r = r0 + 32 * u;
      const T a = warp_sum(acc[u]);
      if (lane == 0 && r < B) {
        q[r] = a;
        nll[r] = -m_log(a);
      }
    }
  }
  __syncthreads();
  T s = T(0);
  if (first)
    for (int64_t i = threadIdx.x; i < B; i += 256) s += nll[i];
  s = block1024_reduce_first8<T, false>(s, sm);
  if (threadIdx.x == 0) loss[0] = s / m;
  if (dz_out == nullptr) return;
  // dL/dz for the upstream gradient 1 (what loss.backward() seeds): ce_bwd_kernel's expressions,
  // operand for operand, so the bits are the ones that kernel would write with g = 1 -- the backward
  // pass of a step then needs no cross-entropy launch at all (q of this CTA is visible after the
  // barrier above)
  for (int64_t i = threadIdx.x; i < n; i += 1024) {
    const int64_t r = i / C;
    const T qm = q[r] * m;
    const T yv = (T)y[i];
    const T p = m_exp(zz[i] - mx) / S;
    T v = p;
    if (yv != T(0)) v = p - (yv * p) / qm;
    dz_out[i] = v;
  }
}

// ---- cross entropy backward ---------------------------------------------------------------------
// dz_kl = g * ( e_kl/S - (1/m) * y_kl * e_kl / (S * q_k) ),  e = exp(z - M)
template <typename T, typename TY, bool VEC>
__global__ void __launch_bounds__(256)
ce_bwd_kernel(T* dz, const T* z, const TY* y, int64_t B, int64_t C, const T* stats, const T* q,
              T m, const T* gptr, unsigned int* absmax_out, const int32_t* labels) {
  // rows over blockIdx.y, column slots over blockIdx.x * 256 + threadIdx.x: no per-element division.
  // VEC: a slot is 4 consecutive columns moved with 128-bit (z, dz) / 128- or 256-bit (y) accesses.
  constexpr int W = VEC ? 4 : 1;
  pdl_sync();
  const T mx = stats[0], S = stats[1], g = gptr[0];
  const int64_t nslot = C / W;
  unsigned int amax = 0u;   // bits of max |dz| (float32 only): the operand statistics of the next split
  for (int64_t r = blockIdx.y; r < B; r += gridDim.y) {
    const T qm = q[r] * m;
    const T* zr = z + r * C;
    const TY* yr = y + r * C;          // (not dereferenced when labels are given)
    const int64_t lab = labels ? (int64_t)labels[r] : -1;
    T* dr = dz + r * C;
    for (int64_t c = (int64_t)blockIdx.x * 256 + threadIdx.x; c < nslot; c += (int64_t)gridDim.x * 256) {
      T zv[W], yv[W], out[W];
      if constexpr (VEC) {
        const float4 t = *reinterpret_cast<const float4*>(zr + c * 4);
        zv[0] = t.x; zv[1] = t.y; zv[2] = t.z; zv[3] = t.w;
        if (labels) {
#pragma unroll
          for (int k = 0; k < 4; ++k) yv[k] = (c * 4 + k == lab) ? T(1) : T(0);
        } else if constexpr (sizeof(TY) == 4) {
          const float4 u = *reinterpret_cast<const float4*>(yr + c * 4);
          yv[0] = u.x; yv[1] = u.y; yv[2] = u.z; yv[3] = u.w;
        } else {
          const double2 u0 = *reinterpret_cast<const double2*>(yr + c * 4);
          const double2 u1 = *reinterpret_cast<const double2*>(yr + c * 4 + 2);
          yv[0] = (T)u0.x; yv[1] = (T)u0.y; yv[2] = (T)u1.x; yv[3] = (T)u1.y;
        }
      } else {
        zv[0] = zr[c];
        yv[0] = labels ? ((c == lab) ? T(1) : T(0)) : (T)yr[c];
      }
#pragma unroll
      for (int k = 0; k < W; ++k) {
        T p = m_exp(zv[k] - mx) / S;
        T v = p;
        if (yv[k] != T(0)) v = p - (yv[k] * p) / qm;
        out[k] = g * v;
        if constexpr (sizeof(T) == 4) amax = max(amax, __float_as_uint((float)out[k]) & 0x7FFFFFFFu);
      }
      if constexpr (VEC) *reinterpret_cast<float4*>(dr + c * 4) = make_float4(out[0], out[1], out[2], out[3]);
      else dr[c] = out[0];
    }
  }
  if constexpr (sizeof(T) == 4) {
    if (absmax_out != nullptr) {      // integer max: exact and order-independent
      amax = __reduce_max_sync(0xFFFFFFFFu, amax);
      if ((threadIdx.x & 31) == 0 && amax) atomicMax(absmax_out, amax);
    }
  }
}

// ---- optimizers ------------------------------------------------------------------------------
struct OptH {
  double h[8];
};

template <int OPT>
constexpr bool adam_family = OPT == TNN_OPT_ADAM || OPT == TNN_OPT_ADAMW || OPT == TNN_OPT_RADAM ||
                             OPT == TNN_OPT_ADAMAX;

// The Adam family's per-element update, shared by opt_kernel and adam_vec_kernel so that the scalar
// and the 128-bit path give the same bits.  The coefficients are narrowed once from the host's doubles
// (include/tnn_b200.h lists each rule's h[] layout).
template <int OPT, typename T>
struct AdamRule {
  T lr, omb1, b2, eps, c4, c5, c6, wd;
  __device__ __forceinline__ explicit AdamRule(const OptH& hh)
      // 1-b1 and 1-b2 are formed in double like the reference's Python floats, then narrowed
      : lr((T)hh.h[0]), omb1((T)(1.0 - hh.h[1])), b2(OPT == TNN_OPT_ADAMAX ? (T)hh.h[2] : (T)(1.0 - hh.h[2])),
        eps((T)hh.h[3]), c4((T)hh.h[4]), c5((T)hh.h[5]), c6((T)hh.h[6]), wd((T)hh.h[7]) {}

  // moments m (state 0) and v (state 1; Adamax: the infinity norm u) updated in place; returns the
  // step before any weight decay
  __device__ __forceinline__ T step(T g, T& m, T& v) const {
    m += omb1 * (g - m);
    if constexpr (OPT == TNN_OPT_ADAMAX) {
      v = m_max(b2 * v, fabs(g) + eps);   // NaN in either operand propagates
      return -c4 * m / v;
    } else {
      v += b2 * (g * g - v);              // b2 holds 1-b2 here
      if constexpr (OPT == TNN_OPT_RADAM) {
        // r_t (c6) is read here rather than chosen on the host: a recorded step reads it from
        // device memory at every replay and switches to the rectified form when t reaches it
        const T mh = m / c4;
        if (c6 > T(0)) return -lr * c6 * mh * c5 / (m_sqrt(v) + eps);
        return -lr * mh;
      } else {
        T mh = m / c4, vh = v / c5;
        return -lr * mh / (m_sqrt(vh) + eps);
      }
    }
  }

  // the new parameter; `step` takes the opt-in weight decay (h[7], optimizer.py:28-29)
  __device__ __forceinline__ T apply(T p, T& step) const {
    if (wd != T(0)) step -= wd * p;
    if constexpr (OPT == TNN_OPT_ADAMW) return p * c6 + step;   // decoupled decay: p * (1 - lr*wd)
    return p + step;
  }
};

template <int OPT, typename T>
__global__ void __launch_bounds__(256)
opt_kernel(T* param, T* step_out, const T* grad, T* s0, T* s1, int64_t n, OptH hh,
           const OptH* hdev) {
  pdl_sync();
  if (hdev) hh = *hdev;   // captured step: the coefficients are refreshed in device memory per replay
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const T g = grad[i];
    T step;
    if constexpr (adam_family<OPT>) {
      const AdamRule<OPT, T> rule(hh);
      T m = s0[i], v = s1[i];
      step = rule.step(g, m, v);
      s0[i] = m;
      s1[i] = v;
      if (param) param[i] = rule.apply(param[i], step);
    } else {
      if constexpr (OPT == TNN_OPT_SGD) {
        step = -(T)hh.h[0] * g;
      } else if constexpr (OPT == TNN_OPT_RMSPROP) {
        const T lr = (T)hh.h[0], omd = (T)(1.0 - hh.h[1]), mom_c = (T)hh.h[2], eps = (T)hh.h[3];
        T ms = s0[i], mom = s1[i];
        ms += omd * (g * g - ms);
        mom = mom_c * mom + lr * g / m_sqrt(ms + eps);
        s0[i] = ms;
        s1[i] = mom;
        step = -mom;
      } else if constexpr (OPT == TNN_OPT_MOMENTUM) {
        const T lr = (T)hh.h[0], mom_c = (T)hh.h[1];
        T acc = mom_c * s0[i] + g;
        s0[i] = acc;
        step = -lr * acc;
      } else if constexpr (OPT == TNN_OPT_ADAGRAD) {
        const T lr = (T)hh.h[0], eps = (T)hh.h[1];
        T G = s0[i] + g * g;
        s0[i] = G;
        step = -(lr / m_sqrt(G + eps)) * g;
      } else {  // ADADELTA
        const T lr = (T)hh.h[0], omd = (T)(1.0 - hh.h[1]), eps = (T)hh.h[2];
        T Eg = s0[i], delta = s1[i];
        Eg += omd * (g * g - Eg);
        T sd = m_sqrt(delta + eps);
        T d = g * (sd / m_sqrt(Eg + eps));
        step = -lr * d;
        delta += omd * (d * d - delta);
        s0[i] = Eg;
        s1[i] = delta;
      }
      if (param) {
        // optimizer.py:28-29 (`_step -= self.weight_decay * v`, commented out upstream): applied only
        // when the host passes a non-zero coefficient in h[7] (BaseOptimizer.apply_weight_decay)
        const T wd = (T)hh.h[7];
        const T p = param[i];
        if (wd != T(0)) step -= wd * p;
        param[i] = p + step;
      }
    }
    if (step_out) step_out[i] = step;
  }
}

// The Adam family is the hot one (28 B/param): 128-bit variant
template <int OPT, typename T>
__global__ void __launch_bounds__(256)
adam_vec_kernel(T* param, const T* grad, T* s0, T* s1, int64_t nv, OptH hh, const OptH* hdev) {
  pdl_sync();
  if (hdev) hh = *hdev;
  constexpr int W = 16 / sizeof(T);
  using V = Pack<T, W>;
  const AdamRule<OPT, T> rule(hh);
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += stride) {
    const V g = reinterpret_cast<const V*>(grad)[i];
    V m = reinterpret_cast<const V*>(s0)[i];
    V v = reinterpret_cast<const V*>(s1)[i];
    V p = reinterpret_cast<const V*>(param)[i];
#pragma unroll
    for (int k = 0; k < W; ++k) {
      T step = rule.step(g.v[k], m.v[k], v.v[k]);
      p.v[k] = rule.apply(p.v[k], step);
    }
    reinterpret_cast<V*>(s0)[i] = m;
    reinterpret_cast<V*>(s1)[i] = v;
    reinterpret_cast<V*>(param)[i] = p;
  }
}

// calls f(std::integral_constant<int, OPT>) for a known optimizer code
template <typename F>
static int with_opt(int opt, F&& f) {
  switch (opt) {
    case TNN_OPT_SGD: return f(std::integral_constant<int, TNN_OPT_SGD>{});
    case TNN_OPT_ADAM: return f(std::integral_constant<int, TNN_OPT_ADAM>{});
    case TNN_OPT_RMSPROP: return f(std::integral_constant<int, TNN_OPT_RMSPROP>{});
    case TNN_OPT_MOMENTUM: return f(std::integral_constant<int, TNN_OPT_MOMENTUM>{});
    case TNN_OPT_ADAGRAD: return f(std::integral_constant<int, TNN_OPT_ADAGRAD>{});
    case TNN_OPT_ADADELTA: return f(std::integral_constant<int, TNN_OPT_ADADELTA>{});
    case TNN_OPT_ADAMW: return f(std::integral_constant<int, TNN_OPT_ADAMW>{});
    case TNN_OPT_RADAM: return f(std::integral_constant<int, TNN_OPT_RADAM>{});
    case TNN_OPT_ADAMAX: return f(std::integral_constant<int, TNN_OPT_ADAMAX>{});
  }
  TNN_FAIL("tnn_opt_step: unknown optimizer code");
}

template <typename T>
static int opt_dispatch(int opt, T* param, T* step_out, const T* grad, T* s0, T* s1, int64_t n,
                        const OptH& hh, const OptH* hdev) {
  cudaStream_t st = ctx().stream;
  int grid = ew_grid(n, 256);
  // a small arena is the tail of a launch-bound chain (the MNIST-sized step): programmatic dependency
  const bool pdl = grid <= 2 * ctx().sm_count;
  constexpr int W = 16 / sizeof(T);
  const bool vec = param && !step_out && aligned16(param) && aligned16(grad) && aligned16(s0) &&
                   aligned16(s1) && n >= W;
  return with_opt(opt, [&](auto OPT) {
    if constexpr (adam_family<OPT>) {
      if (vec) {
        const int64_t nv = n / W, done = nv * W;
        TNN_CUDA(launch_small(adam_vec_kernel<OPT, T>, dim3(ew_grid(nv, 256)), dim3(256), st, pdl, 1u, param, grad,
                              s0, s1, nv, hh, hdev));
        ctx().launches++;
        if (done == n) return 0;
        TNN_CUDA(launch_small(opt_kernel<OPT, T>, dim3(1), dim3(256), st, pdl, 1u, param + done, (T*)nullptr,
                              grad + done, s0 + done, s1 + done, n - done, hh, hdev));
        TNN_POST_LAUNCH();
        return 0;
      }
    }
    TNN_CUDA(launch_small(opt_kernel<OPT, T>, dim3(grid), dim3(256), st, pdl, 1u, param, step_out, grad, s0, s1, n, hh, hdev));
    TNN_POST_LAUNCH();
    return 0;
  });
}

// ---- CE host drivers ---------------------------------------------------------------------------
template <typename T>
static int ce_stats_impl(const T* z, int64_t B, int64_t C, T* stats) {
  const int64_t n = B * C;
  if (n <= 0) TNN_FAIL("tnn_ce_stats: empty logits");
  cudaStream_t st = ctx().stream;
  if (n <= 16384) {
    ce_stats_small_kernel<T><<<1, 256, 0, st>>>(z, n, stats);
    TNN_POST_LAUNCH();
    return 0;
  }
  const bool vec = aligned16(z);
  const int W = vec ? 16 / sizeof(T) : 1;
  int grid = ew_grid(ceil_div(n, W), 256, 4);
  void* scratch;
  if (get_scratch((size_t)grid * 2 * sizeof(T), &scratch)) return 1;
  T* pmax = (T*)scratch;
  T* psum = pmax + grid;
  with_bool(vec, [&](auto V) { ce_partial_max_kernel<T, V><<<grid, 256, 0, st>>>(z, n, pmax); });
  TNN_POST_LAUNCH();
  with_bool(vec, [&](auto V) { ce_partial_sumexp_kernel<T, V><<<grid, 256, 0, st>>>(z, n, pmax, grid, psum, stats); });
  TNN_POST_LAUNCH();
  ce_fold_sum_kernel<T><<<1, 256, 0, st>>>(psum, grid, stats + 1);
  TNN_POST_LAUNCH();
  return 0;
}

template <typename T, typename TY>
static int ce_loss_impl(const T* z, const TY* y, int64_t B, int64_t C, const T* stats, double m,
                        T* q, T* loss, const int32_t* labels) {
  cudaStream_t st = ctx().stream;
  void* scratch;
  if (get_scratch((size_t)B * sizeof(T), &scratch)) return 1;
  T* nll = (T*)scratch;
  if (labels) {
    ce_rows_label_kernel<T><<<ew_grid(B, 256), 256, 0, st>>>(z, labels, B, C, stats, q, nll);
    TNN_POST_LAUNCH();
    ce_fold_loss_kernel<T><<<1, 256, 0, st>>>(nll, B, (T)m, loss);
    TNN_POST_LAUNCH();
    return 0;
  }
  int grid = (int)std::min<int64_t>(ceil_div(B, 8), (int64_t)ctx().sm_count * 8);
  // the 128-bit path is float32 logits and labels in wide 16-byte-aligned rows
  constexpr bool f32 = sizeof(T) == 4 && sizeof(TY) == 4;
  const bool vec = f32 && C >= 512 && C % 4 == 0 && aligned16(z) && aligned16(y);
  with_bool(vec, [&](auto V) {
    if constexpr (V && f32)
      ce_rows_vec_kernel<<<grid, 256, 0, st>>>((const float*)z, (const float*)y, B, C, (const float*)stats,
                                               (float*)q, (float*)nll);
    else
      ce_rows_kernel<T, TY><<<grid, 256, 0, st>>>(z, y, B, C, stats, q, nll);
  });
  TNN_POST_LAUNCH();
  ce_fold_loss_kernel<T><<<1, 256, 0, st>>>(nll, B, (T)m, loss);
  TNN_POST_LAUNCH();
  return 0;
}

template <typename T, typename TY>
static int ce_bwd_impl(T* dz, const T* z, const TY* y, int64_t B, int64_t C, const T* stats,
                       const T* q, double m, const T* g, unsigned int* absmax_out, const int32_t* labels) {
  // the 128-bit path is float32 logits with 4-column-aligned rows
  constexpr bool f32 = sizeof(T) == 4;
  const bool vec = f32 && (C % 4 == 0) && aligned16(dz) && aligned16(z) && (labels || aligned16(y));
  const int64_t nslot = vec ? C / 4 : C;
  int gx = (int)std::min<int64_t>(ceil_div(nslot, 256), 64);
  int64_t gy = std::min<int64_t>(B, std::max<int64_t>(1, (int64_t)ctx().sm_count * 8 / gx));
  if (gy > 65535) gy = 65535;
  // a small grid is part of a launch-bound chain (the MNIST-sized step): programmatic dependency
  const bool pdl = (int64_t)gx * gy <= 2 * (int64_t)ctx().sm_count;
  return with_bool(vec, [&](auto V) {
    if constexpr (!V || f32) {
      TNN_CUDA(launch_small(ce_bwd_kernel<T, TY, V>, dim3(gx, (unsigned)gy), dim3(256), ctx().stream, pdl, 1u,
                            dz, z, y, B, C, stats, q, (T)m, g, absmax_out, labels));
      ctx().launches++;
    }
    return 0;
  });
}

}  // namespace tnn

using namespace tnn;

extern "C" {

int tnn_relu_fwd(int dtype, void* out, const void* x, int64_t n) {
  TNN_REQUIRE_INIT();
  return with_float_type(dtype, "tnn_relu_fwd", [&](auto tag) {
    using T = decltype(tag);
    return relu_launch<T, false>((T*)out, nullptr, (const T*)x, n);
  });
}

int tnn_relu_bwd(int dtype, void* dx, const void* g, const void* x, int64_t n) {
  TNN_REQUIRE_INIT();
  return with_float_type(dtype, "tnn_relu_bwd", [&](auto tag) {
    using T = decltype(tag);
    return relu_launch<T, true>((T*)dx, (const T*)g, (const T*)x, n);
  });
}

int tnn_ce_stats(int dtype, const void* z, int64_t B, int64_t C, void* stats_dev) {
  TNN_REQUIRE_INIT();
  return with_float_type(dtype, "tnn_ce_stats", [&](auto tag) {
    using T = decltype(tag);
    return ce_stats_impl<T>((const T*)z, B, C, (T*)stats_dev);
  });
}

int tnn_ce_merge_stats(int dtype, void* stats_out_dev, const void* stats_all_dev, int n_ranks) {
  TNN_REQUIRE_INIT();
  return with_float_type(dtype, "tnn_ce_merge_stats", [&](auto tag) {
    using T = decltype(tag);
    ce_merge_stats_kernel<T><<<1, 32, 0, ctx().stream>>>((T*)stats_out_dev, (const T*)stats_all_dev, n_ranks);
    TNN_POST_LAUNCH();
    return 0;
  });
}

int tnn_ce_loss(int dtype, const void* z, int y_dtype, const void* y, int64_t B, int64_t C,
                const void* stats_dev, double m_global, void* q_dev, void* loss_dev,
                const int32_t* labels_dev) {
  TNN_REQUIRE_INIT();
  if (B <= 0 || C <= 0) TNN_FAIL("tnn_ce_loss: empty logits");
  if (!y && !labels_dev) TNN_FAIL("tnn_ce_loss: neither dense labels nor class indices");
  return with_float_type(dtype, "tnn_ce_loss", [&](auto tag) {
    return with_float_type(y_dtype, "tnn_ce_loss", [&](auto ytag) {
      using T = decltype(tag);
      using TY = decltype(ytag);
      return ce_loss_impl<T, TY>((const T*)z, (const TY*)y, B, C, (const T*)stats_dev, m_global, (T*)q_dev,
                                 (T*)loss_dev, labels_dev);
    });
  });
}

int tnn_ce_fwd_small(int dtype, const void* z, int y_dtype, const void* y, int64_t B, int64_t C,
                     double m_global, void* stats_dev, void* q_dev, void* loss_dev, void* dz_dev) {
  TNN_REQUIRE_INIT();
  if (B <= 0 || C <= 0) TNN_FAIL("tnn_ce_fwd_small: empty logits");
  if (B > CE_SMALL_MAX_ROWS || B * C > 16384) TNN_FAIL("tnn_ce_fwd_small: at most 2048 rows and 16384 logits");
  return with_float_type(dtype, "tnn_ce_fwd_small", [&](auto tag) {
    return with_float_type(y_dtype, "tnn_ce_fwd_small", [&](auto ytag) {
      using T = decltype(tag);
      using TY = decltype(ytag);
      TNN_CUDA(launch_small(ce_fwd_small_kernel<T, TY>, dim3(1), dim3(1024), ctx().stream, true, 1u, (const T*)z,
                            (const TY*)y, B, C, (T)m_global, (T*)stats_dev, (T*)q_dev, (T*)loss_dev, (T*)dz_dev));
      TNN_POST_LAUNCH();
      return 0;
    });
  });
}

int tnn_ce_bwd(int dtype, void* dz, const void* z, int y_dtype, const void* y, int64_t B, int64_t C,
               const void* stats_dev, const void* q_dev, double m_global, const void* g_dev,
               void* stat_meta, const int32_t* labels_dev) {
  TNN_REQUIRE_INIT();
  if (B <= 0 || C <= 0) return 0;
  if (!y && !labels_dev) TNN_FAIL("tnn_ce_bwd: neither dense labels nor class indices");
  unsigned int* am = (unsigned int*)stat_meta;   // word 0 of an f16 operand record (gemm_f16.cu)
  return with_float_type(dtype, "tnn_ce_bwd", [&](auto tag) {
    using T = decltype(tag);
    if (am && !std::is_same<T, float>::value) TNN_FAIL("tnn_ce_bwd: operand statistics are float32 only");
    return with_float_type(y_dtype, "tnn_ce_bwd", [&](auto ytag) {
      using TY = decltype(ytag);
      return ce_bwd_impl<T, TY>((T*)dz, (const T*)z, (const TY*)y, B, C, (const T*)stats_dev, (const T*)q_dev,
                                m_global, (const T*)g_dev, am, labels_dev);
    });
  });
}

int tnn_opt_step(int opt, int dtype, void* param, void* step_out, const void* grad, void* s0,
                 void* s1, int64_t n, const double* h, int n_h) {
  TNN_REQUIRE_INIT();
  if (n <= 0) return 0;
  if (n_h < 0 || n_h > 8) TNN_FAIL("tnn_opt_step: at most 8 hyper-parameters");
  OptH hh;
  for (int i = 0; i < 8; ++i) hh.h[i] = i < n_h ? h[i] : 0.0;
  return with_float_type(dtype, "tnn_opt_step", [&](auto tag) {
    using T = decltype(tag);
    return opt_dispatch<T>(opt, (T*)param, (T*)step_out, (const T*)grad, (T*)s0, (T*)s1, n, hh, nullptr);
  });
}

int tnn_opt_step_dev(int opt, int dtype, void* param, void* step_out, const void* grad, void* s0,
                     void* s1, int64_t n, const double* h_dev) {
  TNN_REQUIRE_INIT();
  if (n <= 0) return 0;
  if (!h_dev) TNN_FAIL("tnn_opt_step_dev: h_dev is NULL");
  OptH hh = {};
  const OptH* hd = reinterpret_cast<const OptH*>(h_dev);
  return with_float_type(dtype, "tnn_opt_step_dev", [&](auto tag) {
    using T = decltype(tag);
    return opt_dispatch<T>(opt, (T*)param, (T*)step_out, (const T*)grad, (T*)s0, (T*)s1, n, hh, hd);
  });
}

}  // extern "C"

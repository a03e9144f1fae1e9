// Fused training pass of the SMALL tail of a Dense/ReLU MLP (the examples/mnist network:
// 784-200-100-70-30-10 at batch 128, examples/mnist/run.py:59-84).
//
// At that size a step is bound by launch count and per-kernel latency, not by arithmetic: the r01
// recorded step was 13 kernels of 4-6 us.  Everything after the first (wide-input) layer has all its
// weights (119 KB) in one SM's shared memory, and every batch row is independent of the others
// except for the loss's batch-global softmax normaliser (losses.py:26-27).  So ONE launch does, for
// 4 batch rows per CTA:
//     forward of Dense 2..L with ReLU        layers.py:43-49, 97-98
//     global-softmax cross-entropy           losses.py:24-32   (one grid-wide exchange of (max, sum-exp))
//     dL/dz_L, the dX chain with ReLU masks  ops.py:156-157, 336-343
//     dL/dz_1 for the first layer's own backward launch
// and then, after a second grid-wide rendezvous, the whole grid turns to
//     dW / db of layers 2..L                 ops.py:159-160, 49-55
// as 32x32 output tiles over ALL batch rows (each element summed by one thread in row order:
// deterministic, no floating-point atomics, no partial buffers), written straight into the flat
// gradient arena.
// The first layer (forward 128x784x200, backward 784x200x128) keeps its own two launches: its
// 627 KB of weights have to be tiled across CTAs by columns, not by rows.
#include <algorithm>

#include "common.cuh"

namespace tnn {
namespace mlp {

constexpr int MAX_LAYERS = 6;     // tail Dense layers
constexpr int R = 4;              // batch rows per CTA (one float4 per feature)
constexpr int THREADS = 256;    // (1024 threads measured slower: the phases are issue-bound on per-thread overhead)
constexpr int MAX_WIDTH = 256;    // widest tail layer (input or output)
constexpr int MAX_BATCH = 256;  // rows (phase 2 stages [rows][32] tiles)

struct TailArgs {
  int L;                          // number of tail layers
  int in[MAX_LAYERS], out[MAX_LAYERS];
  const float* w[MAX_LAYERS];     // [in, out] row-major
  const float* b[MAX_LAYERS];     // [out]
  int64_t dw_off[MAX_LAYERS];     // element offsets of dW / db from `grad` (the first tail parameter's
  int64_t db_off[MAX_LAYERS];     // slot in the flat gradient arena)
  int w_s[MAX_LAYERS];            // shared-memory offsets (floats): weights, row pitch = out | 1
  int b_s[MAX_LAYERS];
  int z_s[MAX_LAYERS + 1];        // float4 arrays: pre-activation of layer l (index 0: the input z1)
  int a_s[MAX_LAYERS + 1];        // relu of it
  int g_s[MAX_LAYERS + 1];        // dL/dz of layer l
  int scratch_s;                  // K-split partial sums: up to THREADS float4
  int smem_floats;
  int64_t act_g[MAX_LAYERS];      // global scratch offsets (floats): input of layer l, [B, in_l]
  int64_t dz_g[MAX_LAYERS];       //                                  dL/dz of layer l's output, [B, out_l]
  int tile_first[MAX_LAYERS + 1]; // phase 2: first 32x32 dW tile of layer l (prefix sums)
  int row_ctas;                   // CTAs that own batch rows (the rest of the grid joins for phase 2)
  // thread split of the two small products of layer l, worked out on the host (integer divisions are
  // 100+ dependent cycles each on the device, and this kernel is a chain of short serial phases):
  // warps per K group, K groups, k per group -- [0] forward (N = out), [1] backward (N = in)
  int wpg[MAX_LAYERS][2], ks[MAX_LAYERS][2], per[MAX_LAYERS][2];
};

__device__ __forceinline__ float4 f4(float v) { return make_float4(v, v, v, v); }
__device__ __forceinline__ void fma4(float4& acc, const float4& a, float w) {
  acc.x = fmaf(a.x, w, acc.x);
  acc.y = fmaf(a.y, w, acc.y);
  acc.z = fmaf(a.z, w, acc.z);
  acc.w = fmaf(a.w, w, acc.w);
}
// clip(x, 0): NaN-propagating like numpy's (layers.py:97-98)
__device__ __forceinline__ float4 relu4(const float4& z) {
  return make_float4(z.x < 0.f ? 0.f : z.x, z.y < 0.f ? 0.f : z.y, z.z < 0.f ? 0.f : z.z, z.w < 0.f ? 0.f : z.w);
}
__device__ __forceinline__ float4 add4(const float4& a, const float4& b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

// out[j] (j < N) = init[j] + sum_k in[k] * W(k, j) for the CTA's 4 rows at once.
// The threads are split into KS groups along K (KS * roundup32(N) <= THREADS, at least 8 k per group;
// the split comes from the host); group partials are folded in group order.  TRANSPOSED = false: W(k, j) = ws[k * pitch + j] (forward);
// true: W(k, j) = ws[j * pitch + k] (backward, dA = dZ @ W^T: k runs over the layer's outputs).
template <bool TRANSPOSED>
__device__ __forceinline__ void small_gemm(const float4* __restrict__ in, int K, int N,
                                           const float* __restrict__ ws, int pitch,
                                           float4* __restrict__ scratch, int wpg, int ks, int per,
                                           float4& result, bool& owner) {
  const int npad = wpg * 32;
  int grp = 0, w = threadIdx.x >> 5;
  while (w >= wpg) { w -= wpg; ++grp; }          // (warp id) / (warps per group) without a division
  const int j = w * 32 + (threadIdx.x & 31);
  float4 acc = f4(0.f);
  if (grp < ks && j < N) {
    const int k0 = grp * per, k1 = min(K, k0 + per);
    if constexpr (!TRANSPOSED) {
      const float* wp = ws + j + k0 * pitch;
      const float4* ip = in + k0;
#pragma unroll 8
      for (int k = 0; k < k1 - k0; ++k) fma4(acc, ip[k], wp[k * pitch]);
    } else {
      const float* wp = ws + j * pitch + k0;
      const float4* ip = in + k0;
#pragma unroll 8
      for (int k = 0; k < k1 - k0; ++k) fma4(acc, ip[k], wp[k]);
    }
  }
  owner = grp == 0 && j < N;
  if (ks > 1) {
    __syncthreads();                       // scratch is free (previous users are past their reads)
    if (grp > 0 && grp < ks && j < N) scratch[(grp - 1) * npad + j] = acc;
    __syncthreads();
    if (owner)
      for (int g = 1; g < ks; ++g) acc = add4(acc, scratch[(g - 1) * npad + j]);
  }
  result = acc;
}

// block-wide reductions over 256 threads (8 warps), fixed order
__device__ __forceinline__ float block_max(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
#pragma unroll
  for (int i = 1; i < THREADS / 32; ++i) r = fmaxf(r, red[i]);
  return r;
}
__device__ __forceinline__ float block_sum(float v, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = red[0];
#pragma unroll
  for (int i = 1; i < THREADS / 32; ++i) r += red[i];
  return r;
}

// grid-wide rendezvous on a monotonically increasing counter (all CTAs are co-resident: cooperative launch)
__device__ __forceinline__ void grid_arrive_and_wait(unsigned int* counter, unsigned int target) {
  __threadfence();
  atomicAdd(counter, 1u);
  unsigned int seen;
  const long long t0 = clock64();
  do {
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(counter) : "memory");
    if (clock64() - t0 > 4000000000LL) {
      printf("tnn mlp_tail: grid rendezvous timed out (cta %d saw %u of %u)\n", (int)blockIdx.x, seen, target);
      __trap();
    }
  } while (seen < target);
}

template <typename TY>
__global__ void __launch_bounds__(THREADS, 1)
mlp_tail_kernel(const __grid_constant__ TailArgs a, const float* __restrict__ z1, int B,
                const TY* __restrict__ y, float m_global, float* __restrict__ grad,
                float* __restrict__ gscratch, float* __restrict__ dz1_out, float2* __restrict__ stats,
                float* __restrict__ loss_part, float* __restrict__ loss_out,
                unsigned int* __restrict__ counters, float* __restrict__ logits_out) {
  extern __shared__ float4 smem4[];
  float* sm = reinterpret_cast<float*>(smem4);
  __shared__ float red[THREADS / 32];
  __shared__ float bcast[2 + R];
  const int tid = threadIdx.x;
  const int L = a.L;
  const bool has_rows = (int)blockIdx.x < a.row_ctas;
  const int row0 = blockIdx.x * R;
#ifdef TNN_MLP_TIMING
  long long tprobe[8];
  int nprobe = 0;
#define TNN_PROBE() do { __syncthreads(); if (nprobe < 8) tprobe[nprobe++] = clock64(); } while (0)
#else
#define TNN_PROBE() do { } while (0)
#endif
  TNN_PROBE();

  if (has_rows) {
    // ================= phase 1: this CTA's 4 batch rows through the whole tail =================
    // ---- stage the weights (odd row pitch: conflict-free both by column and by row) and biases ----
    for (int l = 0; l < L; ++l) {
      const int K = a.in[l], N = a.out[l], pitch = N | 1;
      const float* __restrict__ wg = a.w[l];
      float* ws = sm + a.w_s[l];
      const int total = K * N;
      // 4-byte cp.async per element (the odd pitch rules out wider ones): every element of the layer
      // is in flight at once and nothing passes through registers; (row, column) advance
      // incrementally by the constant stride, no division per element.  (r02: batches of eight
      // 128-bit loads followed by scalar stores took 16 k cycles for the 119 KB of the MNIST tail.)
      {
        const int dk = THREADS / N, dj = THREADS - dk * N;
        int k = tid / N, j = tid - k * N;
        for (int q = tid; q < total; q += THREADS) {
          const uint32_t dst = (uint32_t)__cvta_generic_to_shared(ws + k * pitch + j);
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(wg + q) : "memory");
          j += dj;
          k += dk;
          if (j >= N) { j -= N; ++k; }
        }
      }
      for (int j = tid; j < N; j += THREADS) sm[a.b_s[l] + j] = a.b[l][j];
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
#ifdef TNN_MLP_TIMING
    asm volatile("cp.async.wait_group 0;" ::: "memory");
#endif
    TNN_PROBE();   // 1: weights staged
    // ---- the CTA's rows of z1 (pre-activation of the first layer) and a1 = relu(z1) ----
    {
      const int K = a.in[0];
      float4* zs = reinterpret_cast<float4*>(sm + a.z_s[0]);
      float4* as = reinterpret_cast<float4*>(sm + a.a_s[0]);
      for (int k = tid; k < K; k += THREADS) {
        float v[R];
#pragma unroll
        for (int r = 0; r < R; ++r) v[r] = row0 + r < B ? z1[(int64_t)(row0 + r) * K + k] : 0.f;
        zs[k] = make_float4(v[0], v[1], v[2], v[3]);
        as[k] = relu4(zs[k]);
      }
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");   // the weights (in flight since the top) have landed
    __syncthreads();
    float4* scratch = reinterpret_cast<float4*>(sm + a.scratch_s);

    // ---- forward ----
    for (int l = 0; l < L; ++l) {
      const int K = a.in[l], N = a.out[l];
      float4 acc;
      bool owner;
      small_gemm<false>(reinterpret_cast<const float4*>(sm + a.a_s[l]), K, N, sm + a.w_s[l], N | 1, scratch,
                        a.wpg[l][0], a.ks[l][0], a.per[l][0], acc, owner);
      if (owner) {
        const float bj = sm[a.b_s[l] + tid];
        const float4 z = make_float4(acc.x + bj, acc.y + bj, acc.z + bj, acc.w + bj);
        reinterpret_cast<float4*>(sm + a.z_s[l + 1])[tid] = z;
        reinterpret_cast<float4*>(sm + a.a_s[l + 1])[tid] = relu4(z);
      }
      __syncthreads();
    }

    TNN_PROBE();   // 2: forward done
    // ---- cross-entropy with the batch-global normaliser (losses.py:24-32) ----
    const int C = a.out[L - 1];
    const bool has_col = tid < C;            // C <= 256: one logit column per thread, 4 rows each
    float zv[R];
    {
      const float4 z = has_col ? reinterpret_cast<const float4*>(sm + a.z_s[L])[tid] : f4(0.f);
      zv[0] = z.x; zv[1] = z.y; zv[2] = z.z; zv[3] = z.w;
    }
    if (logits_out != nullptr && has_col) {
      // the network's output rows (Model.forward's return value), for a caller that reads them
      // after the step
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (row0 + r < B) logits_out[(int64_t)(row0 + r) * C + tid] = zv[r];
    }
    float lmax = -INFINITY;
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (has_col && row0 + r < B) lmax = fmaxf(lmax, zv[r]);
    lmax = block_max(lmax, red);
    float lsum = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (has_col && row0 + r < B) lsum += expf(zv[r] - lmax);
    lsum = block_sum(lsum, red);
    // one exchange across the row CTAs: every one publishes its (max, sum-exp), waits for the others,
    // then merges all pairs in CTA order (same arithmetic everywhere -> identical M and S)
    float2* pairs = reinterpret_cast<float2*>(sm + a.scratch_s);      // K-split scratch is idle here
    if (tid == 0) {
      stats[blockIdx.x] = make_float2(lmax, lsum);
      grid_arrive_and_wait(counters + 0, (unsigned int)a.row_ctas);
    }
    __syncthreads();
    if (tid < a.row_ctas) pairs[tid] = __ldcg(&stats[tid]);           // one L2 round trip for all pairs
    __syncthreads();
    if (tid == 0) {
      float M = -INFINITY;
      for (int c = 0; c < a.row_ctas; ++c) M = fmaxf(M, pairs[c].x);
      float S = 0.f;
      for (int c = 0; c < a.row_ctas; ++c) S += pairs[c].y * expf(pairs[c].x - M);
      bcast[0] = M;
      bcast[1] = S;
    }
    __syncthreads();
    const float M = bcast[0], S = bcast[1];
    float pv[R], yv[R], py[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const bool ok = has_col && row0 + r < B;
      pv[r] = ok ? expf(zv[r] - M) / S : 0.f;
      yv[r] = ok ? (float)y[(int64_t)(row0 + r) * C + tid] : 0.f;
      py[r] = pv[r] * yv[r];
    }
    float q[R];
#pragma unroll
    for (int r = 0; r < R; ++r) q[r] = block_sum(py[r], red);
    if (tid == 0) {
      float nll = 0.f;
#pragma unroll
      for (int r = 0; r < R; ++r)
        if (row0 + r < B) nll += -logf(q[r]);
      loss_part[blockIdx.x] = nll;
    }
    if (has_col) {
      float g[R];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        float v = pv[r];
        if (yv[r] != 0.f) v = pv[r] - (yv[r] * pv[r]) / (q[r] * m_global);
        g[r] = row0 + r < B ? v : 0.f;
      }
      reinterpret_cast<float4*>(sm + a.g_s[L])[tid] = make_float4(g[0], g[1], g[2], g[3]);
    }
    __syncthreads();

    TNN_PROBE();   // 3: cross-entropy (and its exchange) done
    // ---- backward chain: dA = dZ @ W^T, ReLU mask of the layer below; every layer's input and dL/dz
    // rows go to global scratch for phase 2 ----
    for (int l = L - 1; l >= 0; --l) {
      const int K = a.in[l], N = a.out[l];
      const float4* gz = reinterpret_cast<const float4*>(sm + a.g_s[l + 1]);   // dL/dz of this layer
      const float4* ain = reinterpret_cast<const float4*>(sm + a.a_s[l]);      // its input
      float* ag = gscratch + a.act_g[l];
      float* dg = gscratch + a.dz_g[l];
      for (int k = tid; k < K; k += THREADS) {
        const float4 v = ain[k];
        const float e[R] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int r = 0; r < R; ++r)
          if (row0 + r < B) ag[(int64_t)(row0 + r) * K + k] = e[r];
      }
      for (int j = tid; j < N; j += THREADS) {
        const float4 v = gz[j];
        const float e[R] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int r = 0; r < R; ++r)
          if (row0 + r < B) dg[(int64_t)(row0 + r) * N + j] = e[r];
      }
      float4 acc;
      bool owner;
      small_gemm<true>(gz, N, K, sm + a.w_s[l], N | 1, scratch, a.wpg[l][1], a.ks[l][1], a.per[l][1], acc, owner);
      if (owner) {
        const float4 z = reinterpret_cast<const float4*>(sm + a.z_s[l])[tid];
        const float4 m = make_float4(z.x >= 0.f ? acc.x : acc.x * 0.f, z.y >= 0.f ? acc.y : acc.y * 0.f,
                                     z.z >= 0.f ? acc.z : acc.z * 0.f, z.w >= 0.f ? acc.w : acc.w * 0.f);
        if (l > 0) {
          reinterpret_cast<float4*>(sm + a.g_s[l])[tid] = m;
        } else {
          const float e[R] = {m.x, m.y, m.z, m.w};
#pragma unroll
          for (int r = 0; r < R; ++r)
            if (row0 + r < B) dz1_out[(int64_t)(row0 + r) * K + tid] = e[r];
        }
      }
      __syncthreads();
    }
  }

  TNN_PROBE();     // 4: backward chain done
  // ================= rendezvous of the whole grid, then phase 2: dW / db tiles =================
  __syncthreads();
  if (tid == 0) grid_arrive_and_wait(counters + 1, gridDim.x);
  __syncthreads();
  if (blockIdx.x == 0) {
    float* lp = sm + a.scratch_s;
    if (tid < a.row_ctas) lp[tid] = __ldcg(&loss_part[tid]);
    __syncthreads();
    if (tid == 0) {
      float s = 0.f;
      for (int c = 0; c < a.row_ctas; ++c) s += lp[c];
      *loss_out = s / m_global;
    }
    __syncthreads();
  }
  TNN_PROBE();     // 5: rendezvous passed
  // shared memory is free again: [rows][32] tiles of the layer input and of dL/dz, all batch rows
  float (*As)[32] = reinterpret_cast<float (*)[32]>(sm);
  float (*Gs)[32] = reinterpret_cast<float (*)[32]>(sm + 32 * MAX_BATCH);
  const int n_tiles = a.tile_first[L];
  const int tx = tid & 15, ty = tid >> 4;        // 16 x 16 threads, 2 x 2 outputs each
  for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    int l = 0;
    while (t >= a.tile_first[l + 1]) ++l;
    const int K = a.in[l], N = a.out[l];
    const int tiles_n = (N + 31) >> 5;
    int lt = t - a.tile_first[l], ib = 0;
    while (lt >= tiles_n) { lt -= tiles_n; ++ib; }
    const int i0 = ib * 32, j0 = lt * 32;
    const float* __restrict__ ag = gscratch + a.act_g[l];
    const float* __restrict__ dg = gscratch + a.dz_g[l];
    __syncthreads();                               // previous tile's readers are done
    {
      // thread -> column c of rows r0, r0 + 8, ...: all loads of a thread are issued before its stores
      const int c = tid & 31, r0 = tid >> 5;
      const bool ca = i0 + c < K, cg = j0 + c < N;
      for (int rb = r0; rb < B; rb += 64) {
        float va[8], vg[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int r = rb + 8 * u;
          va[u] = (ca && r < B) ? __ldcg(&ag[(int64_t)r * K + i0 + c]) : 0.f;
          vg[u] = (cg && r < B) ? __ldcg(&dg[(int64_t)r * N + j0 + c]) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int r = rb + 8 * u;
          if (r < B) {
            As[r][c] = va[u];
            Gs[r][c] = vg[u];
          }
        }
      }
    }
    __syncthreads();
    float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
#pragma unroll 8
    for (int r = 0; r < B; ++r) {
      const float2 x = *reinterpret_cast<const float2*>(&As[r][ty * 2]);
      const float2 g = *reinterpret_cast<const float2*>(&Gs[r][tx * 2]);
      acc[0][0] = fmaf(x.x, g.x, acc[0][0]);
      acc[0][1] = fmaf(x.x, g.y, acc[0][1]);
      acc[1][0] = fmaf(x.y, g.x, acc[1][0]);
      acc[1][1] = fmaf(x.y, g.y, acc[1][1]);
    }
    float* dw = grad + a.dw_off[l];
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int v = 0; v < 2; ++v) {
        const int i = i0 + ty * 2 + u, j = j0 + tx * 2 + v;
        if (i < K && j < N) dw[(int64_t)i * N + j] = acc[u][v];
      }
    if (i0 == 0 && tid < 32 && j0 + tid < N) {     // the bias gradient rides on the first tile row
      float sacc = 0.f;
      for (int r = 0; r < B; ++r) sacc += Gs[r][tid];
      grad[a.db_off[l] + j0 + tid] = sacc;
    }
  }
  TNN_PROBE();     // 6: dW / db tiles done
#ifdef TNN_MLP_TIMING
  if (blockIdx.x == 0 && tid == 0)
    for (int i = 1; i < nprobe; ++i) counters[4 + i] = (unsigned int)(tprobe[i] - tprobe[i - 1]);
#endif
  // last CTA out rearms the counters for the next step
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const unsigned int done = atomicAdd(counters + 2, 1u);
    if (done == gridDim.x - 1) {
      counters[0] = 0u;
      counters[1] = 0u;
      counters[2] = 0u;
      __threadfence();
    }
  }
}

}  // namespace mlp
}  // namespace tnn

using namespace tnn;

extern "C" {

int tnn_mlp_tail_workspace(int n_layers, const int64_t* in_dims, const int64_t* out_dims, int64_t batch,
                           int64_t* smem_bytes, int64_t* n_ctas, int64_t* scratch_floats) {
  if (n_layers < 1 || n_layers > mlp::MAX_LAYERS) TNN_FAIL("tnn_mlp_tail: 1..6 tail layers");
  if (batch < 1 || batch > mlp::MAX_BATCH) TNN_FAIL("tnn_mlp_tail: batch must be 1..256 rows");
  int64_t floats = 0, tiles = 0, per_row = 0;
  for (int l = 0; l < n_layers; ++l) {
    if (in_dims[l] < 1 || out_dims[l] < 1 || in_dims[l] > mlp::MAX_WIDTH || out_dims[l] > mlp::MAX_WIDTH)
      TNN_FAIL("tnn_mlp_tail: layer widths must be 1..256");
    if (l > 0 && in_dims[l] != out_dims[l - 1]) TNN_FAIL("tnn_mlp_tail: layer widths do not chain");
    floats += in_dims[l] * (out_dims[l] | 1) + ((out_dims[l] + 3) & ~int64_t(3));
    tiles += ((in_dims[l] + 31) / 32) * ((out_dims[l] + 31) / 32);
    per_row += in_dims[l] + out_dims[l];
  }
  int64_t feats = in_dims[0];
  for (int l = 0; l < n_layers; ++l) feats += out_dims[l];
  floats = ((floats + 3) & ~int64_t(3)) + 3 * 4 * feats + 4 * mlp::THREADS;
  floats = std::max<int64_t>(floats, 2 * 32 * mlp::MAX_BATCH);      // phase 2 tiles reuse the space
  const int64_t row_ctas = (batch + mlp::R - 1) / mlp::R;
  if (smem_bytes) *smem_bytes = floats * 4;
  if (n_ctas) *n_ctas = std::max<int64_t>(row_ctas, std::min<int64_t>(tiles, 96));
  if (scratch_floats) *scratch_floats = batch * per_row;
  return 0;
}

// One fused pass over the tail of the MLP (see the file header and include/tnn_b200.h).
int tnn_mlp_tail_step(int n_layers, const int64_t* in_dims, const int64_t* out_dims, const void* const* w,
                      const void* const* b, const int64_t* grad_off, void* grad, int64_t n_grad,
                      const void* z1, const void* y, int y_dtype, int64_t B, double m_global, void* dz1,
                      void* loss_out, void* scratch, void* stats, void* loss_part, void* counters,
                      void* logits_out) {
  TNN_REQUIRE_INIT();
  int64_t smem_bytes = 0, n_ctas = 0, scratch_floats = 0;
  if (tnn_mlp_tail_workspace(n_layers, in_dims, out_dims, B, &smem_bytes, &n_ctas, &scratch_floats)) return 1;
  if (smem_bytes > 220 * 1024) TNN_FAIL("tnn_mlp_tail_step: the tail's weights do not fit in shared memory");
  if (n_ctas > ctx().sm_count) TNN_FAIL("tnn_mlp_tail_step: more CTAs than SMs (the grid rendezvous needs co-residency)");
  mlp::TailArgs a = {};
  a.L = n_layers;
  a.row_ctas = (int)((B + mlp::R - 1) / mlp::R);
  int off = 0;
  int64_t goff = 0;
  for (int l = 0; l < n_layers; ++l) {
    a.in[l] = (int)in_dims[l];
    a.out[l] = (int)out_dims[l];
    a.w[l] = (const float*)w[l];
    a.b[l] = (const float*)b[l];
    a.dw_off[l] = grad_off[2 * l];
    a.db_off[l] = grad_off[2 * l + 1];
    if (a.dw_off[l] < 0 || a.dw_off[l] + in_dims[l] * out_dims[l] > n_grad || a.db_off[l] < 0 ||
        a.db_off[l] + out_dims[l] > n_grad)
      TNN_FAIL("tnn_mlp_tail_step: gradient offsets outside the tail's stretch of the arena");
    a.w_s[l] = off;
    off += a.in[l] * (a.out[l] | 1);
    a.b_s[l] = off;
    off += (a.out[l] + 3) & ~3;
    a.act_g[l] = goff;
    goff += B * in_dims[l];
    a.dz_g[l] = goff;
    goff += B * out_dims[l];
    a.tile_first[l + 1] = a.tile_first[l] + ((a.in[l] + 31) / 32) * ((a.out[l] + 31) / 32);
    for (int d = 0; d < 2; ++d) {
      const int K = d == 0 ? a.in[l] : a.out[l], N = d == 0 ? a.out[l] : a.in[l];
      const int npad = (N + 31) & ~31;
      int ks = mlp::THREADS / npad;
      if (ks > 8) ks = 8;
      while (ks > 1 && K / ks < 8) --ks;
      a.wpg[l][d] = npad / 32;
      a.ks[l][d] = ks;
      a.per[l][d] = (K + ks - 1) / ks;
    }
  }
  off = (off + 3) & ~3;
  for (int l = 0; l <= n_layers; ++l) {
    const int f = l == 0 ? a.in[0] : a.out[l - 1];
    a.z_s[l] = off; off += 4 * f;
    a.a_s[l] = off; off += 4 * f;
    a.g_s[l] = off; off += 4 * f;
  }
  a.scratch_s = off;
  off += 4 * mlp::THREADS;
  a.smem_floats = off;
  if ((int64_t)std::max(off, 2 * 32 * mlp::MAX_BATCH) * 4 != smem_bytes || goff != scratch_floats)
    TNN_FAIL("tnn_mlp_tail_step: internal workspace layout mismatch");

  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)n_ctas);
  cfg.blockDim = dim3(mlp::THREADS);
  cfg.dynamicSmemBytes = (size_t)smem_bytes;
  cfg.stream = ctx().stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;     // all CTAs resident: the rendezvous cannot deadlock
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return with_float_type(y_dtype, "tnn_mlp_tail_step", [&](auto tag) {
    using TY = decltype(tag);
    auto kern = mlp::mlp_tail_kernel<TY>;
    static bool attr_set = false;   // one per label type
    if (!attr_set) {
      TNN_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
      attr_set = true;
    }
    TNN_CUDA(cudaLaunchKernelEx(&cfg, kern, a, (const float*)z1, (int)B, (const TY*)y, (float)m_global,
                                (float*)grad, (float*)scratch, (float*)dz1, (float2*)stats, (float*)loss_part,
                                (float*)loss_out, (unsigned int*)counters, (float*)logits_out));
    ctx().launches++;
    return 0;
  });
}

}  // extern "C"

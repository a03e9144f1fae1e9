// SIMT GEMM for ops.py:150-163 (dot_: A@B, grad@B.T, A.T@grad) on shapes the tensor-core path
// cannot or should not take: float64 (the reference's test path), and the small / odd-sized
// layers of the examples/mnist MLP (70-, 30-, 10-wide: row pitches of 280/120/40 bytes break
// TMA's 16-byte stride rule).  Operands are addressed through (row, col) element strides so the
// transposed products of the backward pass read the original buffers in place.
//
// C[M,N] = A[M,K] * B[K,N] (+ bias[N]) (+ C), shared-memory tiled, register-blocked, the next
// K-slab prefetched into registers while the current one is multiplied.  Deterministic: each
// output element is accumulated by one thread in k order.
//
// Few tiles and a deep K (the 128x200x784 first layer of the MNIST MLP: 28 tiles, 13 slabs, each a
// round trip to L2/HBM -> 30 us on 28 of 148 SMs) run as a thread-block CLUSTER along K: the S CTAs
// of a cluster each multiply one K slice of the same output tile, park their 32x32 partial in
// their own shared memory, and CTA 0 adds the partials in rank order over distributed shared
// memory -- one launch, no scratch buffer, no atomics, a fixed summation order.
#include <cooperative_groups.h>

#include <cstdlib>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace tnn {

// shared-memory row pitch: even for the 2x2 micro-tile so a thread's two A (or B) values of one k are
// ONE 64/128-bit load (2-way store conflict in the k-fast layout, 16 stores per slab: cheap), odd
// (conflict-free) otherwise
template <int B, int TT>
struct Pitch {
  static constexpr int value = B + (TT == 2 ? 2 : 1);
};

// One output tile.  SPLITK: gridDim.z CTAs (one cluster) share the tile, CTA z covers k in
// [z*kslice, ...).
template <typename T, int BM, int BN, int BK, int TM, int TN, bool SPLITK>
__device__ __forceinline__ void
gemm_tile(T (*As)[Pitch<BM, TM>::value], T (*Bs)[Pitch<BN, TN>::value], int tile_x, int tile_y, T* __restrict__ C, int64_t ldc,
          const T* __restrict__ A, int64_t a_rs, int64_t a_cs, const T* __restrict__ B, int64_t b_rs,
          int64_t b_cs, int64_t M, int64_t N, int64_t K, const T* __restrict__ bias, int flags,
          T* __restrict__ act_out, const T* __restrict__ mask_src, int64_t kslice) {
  constexpr int NT = (BM / TM) * (BN / TN);
  constexpr int A_PER = (BM * BK) / NT;
  constexpr int B_PER = (BK * BN) / NT;
  static_assert((BM * BK) % NT == 0 && (BK * BN) % NT == 0, "tile/threads mismatch");

  const int tid = threadIdx.x;
  const int tx = tid % (BN / TN), ty = tid / (BN / TN);
  const int64_t m0 = (int64_t)tile_y * BM, n0 = (int64_t)tile_x * BN;
  const bool a_kfast = (a_cs == 1);   // k contiguous in memory
  const bool b_nfast = (b_cs == 1);   // n contiguous in memory

  T acc[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) acc[i][j] = T(0);

  T ra[A_PER], rb[B_PER];

  // Element e of this thread's share of a slab is element `tid + e*NT` of the tile.  With NT a
  // multiple of BK, BM and BN the (row, k) of element e is (row0 + e*drow, k0 + e*dk): one of the
  // two advances is zero, so every load is `base + e*step` behind two compares.  (Written out by
  // hand: left to the compiler, the div/mod per element and the runtime layout select were 2,000
  // integer instructions around 44 loads, and the MNIST-sized products are issue-bound.)
  static_assert(NT % BK == 0 && NT % BM == 0 && NT % BN == 0, "strength-reduced tile loads");
  const int a_m = a_kfast ? tid / BK : tid % BM, a_k = a_kfast ? tid % BK : tid / BM;
  const int a_dm = a_kfast ? NT / BK : 0, a_dk = a_kfast ? 0 : NT / BM;
  const int b_k = b_nfast ? tid / BN : tid % BK, b_n = b_nfast ? tid % BN : tid / BK;
  const int b_dk = b_nfast ? NT / BN : 0, b_dn = b_nfast ? 0 : NT / BK;
  const T* a_base = A + (m0 + a_m) * a_rs + (int64_t)a_k * a_cs;
  const T* b_base = B + (int64_t)b_k * b_rs + (n0 + b_n) * b_cs;
  const int64_t a_step = (int64_t)a_dm * a_rs + (int64_t)a_dk * a_cs;
  const int64_t b_step = (int64_t)b_dk * b_rs + (int64_t)b_dn * b_cs;
  // bounds as 32-bit counts (clamped): one integer compare per load instead of a 64-bit pair
  auto clamp32 = [](int64_t v) { return (int)(v > (1 << 30) ? (1 << 30) : (v < -1 ? -1 : v)); };
  const int a_rows_left = clamp32(M - m0 - a_m);   // row e*a_dm is valid while e*a_dm < a_rows_left
  const int b_cols_left = clamp32(N - n0 - b_n);

  auto load_tiles = [&](int64_t k0) {
    const T* ap = a_base + k0 * a_cs;
    const T* bp = b_base + k0 * b_rs;
    const int a_k_left = clamp32(K - k0 - a_k), b_k_left = clamp32(K - k0 - b_k);
    int rl = a_rows_left, kl = a_k_left;       // running bounds and pointers: adds, no multiplies
#pragma unroll
    for (int e = 0; e < A_PER; ++e) {
      ra[e] = (rl > 0 && kl > 0) ? *ap : T(0);
      rl -= a_dm;
      kl -= a_dk;
      ap += a_step;
    }
    int cl = b_cols_left;
    kl = b_k_left;
#pragma unroll
    for (int e = 0; e < B_PER; ++e) {
      rb[e] = (cl > 0 && kl > 0) ? *bp : T(0);
      cl -= b_dn;
      kl -= b_dk;
      bp += b_step;
    }
  };
  T* const as_base = &As[a_k][a_m];
  T* const bs_base = &Bs[b_k][b_n];
  const int as_step = a_dk * Pitch<BM, TM>::value + a_dm, bs_step = b_dk * Pitch<BN, TN>::value + b_dn;
  auto store_tiles = [&]() {
#pragma unroll
    for (int e = 0; e < A_PER; ++e) as_base[e * as_step] = ra[e];
#pragma unroll
    for (int e = 0; e < B_PER; ++e) bs_base[e * bs_step] = rb[e];
  };

  int64_t k_begin = 0;
  if constexpr (SPLITK) {
    // this CTA's K slice; operands beyond it read as zero through the `gk < K` guard
    k_begin = (int64_t)blockIdx.z * kslice;
    const int64_t k_end = k_begin + kslice < K ? k_begin + kslice : K;
    K = k_end > k_begin ? k_end : k_begin;
  }
  load_tiles(k_begin);
  for (int64_t k0 = k_begin; k0 < K; k0 += BK) {
    store_tiles();
    __syncthreads();
    if (k0 + BK < K) load_tiles(k0 + BK);
    // only as deep as this slab really is (a 30-deep MNIST product must not multiply 98 zeros)
    const int depth = (K - k0 < BK) ? (int)(K - k0) : BK;
#pragma unroll 8
    for (int kk = 0; kk < depth; ++kk) {
      T a[TM], b[TN];
      if constexpr (TM == 2 && TN == 2) {
        struct alignas(2 * sizeof(T)) Pair { T v[2]; };
        const Pair pa = *reinterpret_cast<const Pair*>(&As[kk][ty * 2]);
        const Pair pb = *reinterpret_cast<const Pair*>(&Bs[kk][tx * 2]);
        a[0] = pa.v[0]; a[1] = pa.v[1]; b[0] = pb.v[0]; b[1] = pb.v[1];
      } else {
#pragma unroll
        for (int i = 0; i < TM; ++i) a[i] = As[kk][ty * TM + i];
#pragma unroll
        for (int j = 0; j < TN; ++j) b[j] = Bs[kk][tx * TN + j];
      }
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] += a[i] * b[j];
    }
    __syncthreads();
  }

  if constexpr (SPLITK) {
    // partial tile -> own shared memory; CTA 0 folds the cluster's partials in rank order
    static_assert(BK >= BN, "the partial tile reuses the As slab");
    cg::cluster_group cluster = cg::this_cluster();
    auto part = As;            // rows 0..BN-1 of the A slab hold the BN x BM partial (BK >= BN)
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TN; ++j) part[tx * TN + j][ty * TM + i] = acc[i][j];
    cluster.sync();
    if (blockIdx.z == 0) {
      // all remote loads are issued before the first add (one DSMEM latency, not S-1 of them);
      // the adds then run in rank order
      const unsigned S = gridDim.z;
      T pv[7][TM][TN];
#pragma unroll
      for (unsigned r = 1; r < 8; ++r) {
        if (r < S) {
          auto peer = reinterpret_cast<T (*)[Pitch<BM, TM>::value]>(cluster.map_shared_rank(&As[0][0], r));
#pragma unroll
          for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j) pv[r - 1][i][j] = peer[tx * TN + j][ty * TM + i];
        }
      }
#pragma unroll
      for (unsigned r = 1; r < 8; ++r) {
        if (r < S) {
#pragma unroll
          for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j) acc[i][j] += pv[r - 1][i][j];
        }
      }
    }
    cluster.sync();            // peers keep their shared memory alive until CTA 0 has read it
    if (blockIdx.z != 0) return;
  }
  const bool accumulate = flags & 1;
#pragma unroll
  for (int i = 0; i < TM; ++i) {
    int64_t gm = m0 + ty * TM + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < TN; ++j) {
      int64_t gn = n0 + tx * TN + j;
      if (gn >= N) continue;
      T v = acc[i][j];
      if (bias) v += bias[gn];
      if (accumulate) v += C[gm * ldc + gn];
      C[gm * ldc + gn] = v;
      if (act_out) {
        // fused ReLU output, or (backward form) the ReLU gradient mask of ops.py:336-343 applied
        // to this dX: act = v * (pre-activation >= 0)
        if (mask_src) act_out[gm * ldc + gn] = mask_src[gm * ldc + gn] >= T(0) ? v : v * T(0);
        else act_out[gm * ldc + gn] = v < T(0) ? T(0) : v;
      }
    }
  }
}

template <typename T, int BM, int BN, int BK, int TM, int TN, bool SPLITK>
__global__ void __launch_bounds__((BM / TM) * (BN / TN), BM == 32 ? 2 : 1)   // small tiles: two CTAs per SM, so an 8-way K cluster of 28 tiles is one wave
gemm_simt_kernel(T* __restrict__ C, int64_t ldc, const T* __restrict__ A, int64_t a_rs, int64_t a_cs,
                 const T* __restrict__ B, int64_t b_rs, int64_t b_cs, int64_t M, int64_t N, int64_t K,
                 const T* __restrict__ bias, int flags, T* __restrict__ act_out,
                 const T* __restrict__ mask_src, int64_t kslice) {
  __shared__ __align__(16) T As[BK][Pitch<BM, TM>::value];
  __shared__ __align__(16) T Bs[BK][Pitch<BN, TN>::value];
  pdl_sync();
  gemm_tile<T, BM, BN, BK, TM, TN, SPLITK>(As, Bs, (int)blockIdx.x, (int)blockIdx.y, C, ldc, A, a_rs, a_cs,
                                           B, b_rs, b_cs, M, N, K, bias, flags, act_out, mask_src, kslice);
}

// ---- grouped launch: the three gradient products of a small Dense layer in one kernel -------------
// dX = g @ w^T (+ the ReLU mask of the layer below), dW = x^T @ g, db = 1^T @ g are independent given
// g; for the MNIST-sized layers each is a handful of 32x32 tiles and a launch costs more than the
// arithmetic, so they share one grid: CTA b works on tile (b - first[p]) of problem p.
template <typename T>
struct SimtProblem {
  T* C;
  int64_t ldc;
  const T* A;
  int64_t a_rs, a_cs;
  const T* B;
  int64_t b_rs, b_cs;
  int64_t M, N, K;
  int flags;
  T* act_out;
  const T* mask_src;
  int tiles_x, first;     // tiles per row of this problem's tile grid, first CTA index
};
template <typename T>
struct SimtGroup {
  SimtProblem<T> p[3];
  int count;
};

template <typename T, int BK>
__global__ void __launch_bounds__(256, 2)
gemm_simt_group_kernel(const SimtGroup<T> grp) {
  __shared__ __align__(16) T As[BK][Pitch<32, 2>::value];
  __shared__ __align__(16) T Bs[BK][Pitch<32, 2>::value];
  pdl_sync();
  int pi = 0;
#pragma unroll
  for (int i = 1; i < 3; ++i)
    if (i < grp.count && (int)blockIdx.x >= grp.p[i].first) pi = i;
  const SimtProblem<T>& q = grp.p[pi];
  const int local = (int)blockIdx.x - q.first;
  if (q.A == nullptr) {
    // bias gradient: column sums of B[K, N] for 32 columns.  8 row lanes per column, folded in a
    // fixed order through shared memory (deterministic)
    const int col = local * 32 + (threadIdx.x & 31), lane = threadIdx.x >> 5;
    T acc = T(0);
    if (col < q.N)
      for (int64_t r = lane; r < q.K; r += 8) acc += q.B[r * q.b_rs + col * q.b_cs];
    As[lane][threadIdx.x & 31] = acc;
    __syncthreads();
    if (lane == 0 && col < q.N) {
      T v = As[0][col & 31];
#pragma unroll
      for (int i = 1; i < 8; ++i) v += As[i][col & 31];
      if (q.flags & 1) v += q.C[col];
      q.C[col] = v;
    }
    return;
  }
  gemm_tile<T, 32, 32, BK, 2, 2, false>(As, Bs, local % q.tiles_x, local / q.tiles_x, q.C, q.ldc, q.A, q.a_rs,
                                        q.a_cs, q.B, q.b_rs, q.b_cs, q.M, q.N, q.K, nullptr, q.flags,
                                        q.act_out, q.mask_src, 0);
}

template <typename T>
static int gemm_simt_impl(T* C, int64_t ldc, const T* A, int64_t a_rs, int64_t a_cs, const T* B,
                          int64_t b_rs, int64_t b_cs, int64_t M, int64_t N, int64_t K,
                          const T* bias, int flags, T* act_out, const T* mask_src) {
  if (M <= 0 || N <= 0) return 0;
  cudaStream_t st = ctx().stream;
  prof_begin(2);
  int64_t tiles64 = ceil_div(M, 64) * ceil_div(N, 64);
  if (tiles64 >= ctx().sm_count) {
    dim3 grid((unsigned)ceil_div(N, 64), (unsigned)ceil_div(M, 64));
    if (grid.y > 65535) TNN_FAIL("tnn_gemm_simt: M too large for the SIMT path");
    gemm_simt_kernel<T, 64, 64, 16, 4, 4, false><<<grid, 256, 0, st>>>(C, ldc, A, a_rs, a_cs, B, b_rs, b_cs, M, N, K, bias, flags, act_out, mask_src, 0);
  } else {
    // few CTAs: the K loop is a chain of exposed global-load latencies (measured 53 us for the
    // 128x200x784 first MNIST layer with 16-wide K slabs), so the small-tile variant takes 64-wide
    // slabs: 4x fewer round trips, 8 loads in flight per thread
    dim3 grid((unsigned)ceil_div(N, 32), (unsigned)ceil_div(M, 32));
    const int64_t tiles = (int64_t)grid.x * grid.y;
    // One slab per CTA is one exposed load latency instead of a chain of them, so the slab is as
    // deep as shared memory allows (128 k for float, 64 for double) and, when the tiles leave most
    // SMs idle, K is cut across a cluster of S CTAs (S <= 4 by default, TNN_SIMT_MAX_SPLIT up to the
    // portable cluster size of 8) until a slice fits one slab.
    constexpr int SBK = sizeof(T) == 4 ? 128 : 64;
    static int max_split = -1;
    if (max_split < 0) {
      const char* e = getenv("TNN_SIMT_MAX_SPLIT");
      // measured on the 128x784x200 first MNIST layer (scripts/simt_bench.py): unsplit 26.6 us,
      // 2-way 18.4, 4-way 12.6, 8-way 16.4 (an 8-CTA cluster is slower to place and to fold)
      max_split = e ? atoi(e) : 4;
      if (max_split < 1) max_split = 1;
      if (max_split > 8) max_split = 8;
    }
    int64_t S = 1;
    while (S < max_split && tiles * (S * 2) <= 2 * (int64_t)ctx().sm_count && ceil_div(K, S) > SBK) S *= 2;
    if (S > 1 && grid.y <= 65535) {
      grid.z = (unsigned)S;
      const int64_t kslice = ceil_div(K, S);
      TNN_CUDA(launch_small(gemm_simt_kernel<T, 32, 32, SBK, 2, 2, true>, grid, dim3(256), st, true, (unsigned)S,
                            C, ldc, A, a_rs, a_cs, B, b_rs, b_cs, M, N, K, bias, flags, act_out, mask_src,
                            kslice));
      ctx().launches++;
      prof_end(2);
      return 0;
    }
    TNN_CUDA(launch_small(gemm_simt_kernel<T, 32, 32, SBK, 2, 2, false>, grid, dim3(256), st, true, 1u,
                          C, ldc, A, a_rs, a_cs, B, b_rs, b_cs, M, N, K, bias, flags, act_out, mask_src,
                          (int64_t)0));
    ctx().launches++;
    prof_end(2);
    return 0;
  }
  TNN_POST_LAUNCH();
  prof_end(2);
  return 0;
}

// dX[B,K] = g[B,N] @ w[K,N]^T (optional; with mask: masked = dX * (mask >= 0)),
// dW[K,N] (+)= x[B,K]^T @ g[B,N],  db[1,N] (+)= column sums of g -- one grouped launch
template <typename T>
static int dense_bwd_impl(const T* g, const T* x, const T* w, const T* mask, T* dx, T* masked, T* dw,
                          int dw_acc, T* db, int db_acc, int64_t Bn, int64_t K, int64_t N) {
  SimtGroup<T> grp;
  grp.count = 0;
  int next = 0;
  auto add = [&](T* C, int64_t ldc, const T* A, int64_t a_rs, int64_t a_cs, const T* Bm, int64_t b_rs,
                 int64_t b_cs, int64_t M, int64_t Nn, int64_t Kk, int flags, T* act, const T* msk) {
    SimtProblem<T>& q = grp.p[grp.count++];
    q.C = C; q.ldc = ldc; q.A = A; q.a_rs = a_rs; q.a_cs = a_cs; q.B = Bm; q.b_rs = b_rs; q.b_cs = b_cs;
    q.M = M; q.N = Nn; q.K = Kk; q.flags = flags; q.act_out = act; q.mask_src = msk;
    q.tiles_x = (int)ceil_div(Nn, 32);
    q.first = next;
    next += q.tiles_x * (int)ceil_div(M, 32);
  };
  // the deepest products first: their CTAs start first and finish last
  add(dw, N, x, 1, K, g, N, 1, K, N, Bn, dw_acc ? 1 : 0, nullptr, nullptr);          // x^T @ g
  if (dx) add(dx, K, g, N, 1, w, 1, N, Bn, K, N, 0, masked, masked ? mask : nullptr);   // g @ w^T
  add(db, N, nullptr, 0, 0, g, N, 1, 1, N, Bn, db_acc ? 1 : 0, nullptr, nullptr);      // 1^T @ g
  constexpr int SBK = sizeof(T) == 4 ? 128 : 64;
  prof_begin(2);
  TNN_CUDA(launch_small(gemm_simt_group_kernel<T, SBK>, dim3((unsigned)next), dim3(256), ctx().stream, true, 1u,
                        grp));
  ctx().launches++;
  prof_end(2);
  return 0;
}

}  // namespace tnn

using namespace tnn;

extern "C" int tnn_dense_bwd_simt(int dtype, const void* g, const void* x, const void* w,
                                  const void* mask_src, void* dx, void* dx_masked, void* dw,
                                  int dw_accumulate, void* db, int db_accumulate, int64_t B, int64_t K,
                                  int64_t N) {
  TNN_REQUIRE_INIT();
  if (B <= 0 || K <= 0 || N <= 0) TNN_FAIL("tnn_dense_bwd_simt: empty operand");
  if (!g || !x || !w || !dw || !db) TNN_FAIL("tnn_dense_bwd_simt: g, x, w, dw, db are required");
  if (dx_masked && (!dx || !mask_src)) TNN_FAIL("tnn_dense_bwd_simt: dx_masked needs dx and mask_src");
  if (ceil_div(K, 32) * ceil_div(N, 32) + ceil_div(B, 32) * ceil_div(K, 32) + ceil_div(N, 32) > 65535)
    TNN_FAIL("tnn_dense_bwd_simt: layer too large for the grouped SIMT launch");
  return with_float_type(dtype, "tnn_dense_bwd_simt", [&](auto tag) {
    using T = decltype(tag);
    return dense_bwd_impl<T>((const T*)g, (const T*)x, (const T*)w, (const T*)mask_src, (T*)dx, (T*)dx_masked,
                             (T*)dw, dw_accumulate, (T*)db, db_accumulate, B, K, N);
  });
}

extern "C" int tnn_gemm_simt(int dtype, void* C, int64_t ldc, const void* A, int64_t a_rs,
                             int64_t a_cs, const void* B, int64_t b_rs, int64_t b_cs, int64_t M,
                             int64_t N, int64_t K, const void* bias, int flags, void* act_out,
                             const void* mask_src) {
  TNN_REQUIRE_INIT();
  if (M < 0 || N < 0 || K < 0) TNN_FAIL("tnn_gemm_simt: negative extent");
  if (mask_src && !act_out) TNN_FAIL("tnn_gemm_simt: mask_src needs act_out");
  return with_float_type(dtype, "tnn_gemm_simt", [&](auto tag) {
    using T = decltype(tag);
    return gemm_simt_impl<T>((T*)C, ldc, (const T*)A, a_rs, a_cs, (const T*)B, b_rs, b_cs, M, N, K, (const T*)bias,
                             flags, (T*)act_out, (const T*)mask_src);
  });
}

// What the two tcgen05 GEMM kernels (gemm_tc.cu: TF32 / mixed split, gemm_f16.cu: fp16 split) share:
// tile order, work units, barrier layout and set-up, the TMEM hand-back, the split-K publish, the
// epilogue's patch writer, and on the host the tensor maps, the tail planner and the persistent
// cluster launch.  sm_100a only.
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>

#include <algorithm>

#include "common.cuh"
#include "tc_ptx.cuh"

namespace tnn {
namespace tc {

// ---- device side -------------------------------------------------------------------------------

// Tile rasterisation.  group_m = 1: row-major (the ~74 concurrent CTA pairs share ~5 A row-blocks
// and sweep all B column-blocks).  group_m = -g: column panels of g tile columns (all tile rows of a
// panel, row-major inside it, before the next panel), so the panel's B operand stays L2-resident
// across waves.  group_m = g > 1: row groups (consecutive tiles walk g tile rows before the next tile
// column).
__device__ __forceinline__ void tile_coords(int t, int tiles_m, int tiles_n, int group_m, int& tm, int& tn) {
  if (group_m == 1) {
    tm = t / tiles_n;
    tn = t - tm * tiles_n;
  } else if (group_m < 0) {
    const int gn = -group_m;
    const int per_panel = tiles_m * gn;
    const int g = t / per_panel;
    const int first_n = g * gn;
    const int cols = min(gn, tiles_n - first_n);
    const int r = t - g * per_panel;
    tm = r / cols;
    tn = first_n + r % cols;
  } else {
    const int per_group = group_m * tiles_n;
    const int g = t / per_group;
    const int first_m = g * group_m;
    const int rows = min(group_m, tiles_m - first_m);
    const int r = t - g * per_group;
    tm = first_m + r % rows;
    tn = r / rows;
  }
}

// Work units of a persistent launch.  Tiles [0, t_full) are whole-K units.  The remaining "tail"
// tiles -- the ones that would form a ragged last wave (4096x4096 dW product: 256 tiles on 74 CTA
// pairs = 3 full waves + 34 tiles) -- are cut into tail_split K ranges each, so the last wave is short
// AND full: unit t_full + j covers tile t_full + j % rem, K range j / rem.  Range s > 0 adds onto what
// range s-1 stored, in that fixed order (a per-tile arrival counter, splitk_publish, gates the
// read-modify-write; never a floating-point atomic), so the result does not depend on
// timing.
struct WorkUnits {
  int t_full, tail_rem, num_units, num_kb, kb_per_split;
  __device__ __forceinline__ WorkUnits(int t_full_, int tail_split, int num_tiles, int num_kb_)
      : t_full(t_full_), tail_rem(num_tiles - t_full_), num_units(t_full_ + (num_tiles - t_full_) * tail_split),
        num_kb(num_kb_), kb_per_split((num_kb_ + tail_split - 1) / tail_split) {}
  __device__ __forceinline__ void decode(int u, int& t, int& sp, int& kb_begin, int& kb_end) const {
    if (u < t_full) {
      t = u; sp = 0; kb_begin = 0; kb_end = num_kb;
    } else {
      const int j = u - t_full;
      t = t_full + j % tail_rem;
      sp = j / tail_rem;
      kb_begin = sp * kb_per_split;
      kb_end = min(num_kb, kb_begin + kb_per_split);
    }
  }
};

// Barriers after the STAGES operand stages: full[STAGES], empty[STAGES], tmem_full[2],
// tmem_empty[2], then the word tcgen05.alloc writes the TMEM base address to.
template <int STAGES>
struct Barriers {
  static constexpr int TMEM_PTR_OFF = 8 * (2 * STAGES + 4);   // bytes from the first barrier
  uint32_t base;
  __device__ __forceinline__ uint32_t full(int s) const { return base + 8u * s; }
  __device__ __forceinline__ uint32_t empty(int s) const { return base + 8u * (STAGES + s); }
  __device__ __forceinline__ uint32_t tfull(int a) const { return base + 8u * (2 * STAGES + a); }
  __device__ __forceinline__ uint32_t tempty(int a) const { return base + 8u * (2 * STAGES + 2 + a); }
  // one thread: empty_count arrivals free a stage, tempty_count arrivals free an accumulator
  __device__ __forceinline__ void init(uint32_t empty_count, uint32_t tempty_count) const {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full(s), 1);
      mbar_init(empty(s), empty_count);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull(a), 1);
      mbar_init(tempty(a), tempty_count);
    }
    fence_barrier_init();
  }
};

// Warp 1 allocates the TMEM accumulators; after the (cluster) barrier every thread reads their base
// address through bar_gen, the generic address of the first barrier.
template <int CG, int STAGES>
__device__ __forceinline__ uint32_t tmem_setup(const Barriers<STAGES>& bar, const uint8_t* bar_gen, int warp,
                                               uint32_t cols) {
  if (warp == 1) {
    tmem_alloc<CG>(bar.base + Barriers<STAGES>::TMEM_PTR_OFF, cols);
    tmem_relinquish<CG>();
  }
  tc_fence_before();
  if constexpr (CG == 1) __syncthreads();
  else cluster_sync_all();
  tc_fence_after();
  return *reinterpret_cast<const volatile uint32_t*>(bar_gen + Barriers<STAGES>::TMEM_PTR_OFF);
}

// Everyone (every CTA of the cluster) must be done before TMEM goes away.  The single-lane roles
// re-converge first: the cluster barrier and tcgen05.dealloc are .aligned instructions.
template <int CG>
__device__ __forceinline__ void tmem_teardown(int warp, uint32_t tmem_base, uint32_t cols) {
  __syncwarp();
  tc_fence_before();
  if constexpr (CG == 1) __syncthreads();
  else cluster_sync_all();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<CG>(tmem_base, cols);
  }
}

// This warp is done reading the accumulator: hand it back to the MMA issuer, whose barrier `bar` is
// in CTA `cta` of the cluster (CLUSTER = false: in this CTA).  The arrive publishes no memory, so it
// is relaxed: the release form compiles to MEMBAR.ALL.CTA + ERRBAR, which would wait for the whole
// tile this warp has just stored.
template <bool CLUSTER>
__device__ __forceinline__ void tmem_hand_back(uint32_t bar, uint32_t cta, int lane) {
  tc_fence_before();
  __syncwarp();
  if (lane == 0) {
    if constexpr (CLUSTER) mbar_arrive_cluster_relaxed(bar, cta);
    else mbar_arrive(bar);
  }
}

// Split-K ordering, after storing a range of a tile that is not its last: this warp's part of the
// tile is in global memory, so count it in the tile's counter flags[idx].  The range after it waits
// (in the kernel) until the counter holds every epilogue warp of the ranges before it.
__device__ __forceinline__ void splitk_publish(unsigned int* flags, int idx, int lane) {
  __threadfence();
  __syncwarp();
  if (lane == 0) atomicAdd(flags + idx, 1u);
}

// registers -> swizzled 32 x 32 patch for the 32-column block CB of a thread's 128 sums (SCALE: times
// f1 * f2), plus the bias, which is per column: it is added while the thread still owns consecutive
// columns
template <int CB, bool SCALE>
__device__ __forceinline__ void patch_write(const float (&sum)[128], float4* patch, int lane, float f1,
                                            float f2, const float* bias_u, int colb, int N) {
#pragma unroll
  for (int c4 = 0; c4 < 8; ++c4) {
    const float* s = sum + CB * 32 + c4 * 4;
    float4 v = SCALE ? make_float4(s[0] * f1 * f2, s[1] * f1 * f2, s[2] * f1 * f2, s[3] * f1 * f2)
                     : make_float4(s[0], s[1], s[2], s[3]);
    if (bias_u) {
      const int c = colb + c4 * 4;
      if (c + 3 < N) {
        const float4 b = *reinterpret_cast<const float4*>(bias_u + c);
        v.x += b.x; v.y += b.y; v.z += b.z; v.w += b.w;
      } else {
        if (c < N) v.x += bias_u[c];
        if (c + 1 < N) v.y += bias_u[c + 1];
        if (c + 2 < N) v.z += bias_u[c + 2];
      }
    }
    patch[lane * 8 + (c4 ^ (lane & 7))] = v;
  }
}

// the same for a run-time block cb (register indices must be compile-time, hence the switch)
template <bool SCALE>
__device__ __forceinline__ void patch_write(int cb, const float (&sum)[128], float4* patch, int lane, float f1,
                                            float f2, const float* bias_u, int colb, int N) {
  switch (cb) {
    case 0: patch_write<0, SCALE>(sum, patch, lane, f1, f2, bias_u, colb, N); break;
    case 1: patch_write<1, SCALE>(sum, patch, lane, f1, f2, bias_u, colb, N); break;
    case 2: patch_write<2, SCALE>(sum, patch, lane, f1, f2, bias_u, colb, N); break;
    default: patch_write<3, SCALE>(sum, patch, lane, f1, f2, bias_u, colb, N); break;
  }
}

// ---- host side ---------------------------------------------------------------------------------

inline PFN_cuTensorMapEncodeTiled_v12000 g_encode = nullptr;

inline int get_encode_fn() {
  if (g_encode) return 0;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  TNN_CUDA(cudaGetDriverEntryPointByVersion("cuTensorMapEncodeTiled", &fn, 12000, cudaEnableDefault, &qres));
  if (qres != cudaDriverEntryPointSuccess || !fn) TNN_FAIL("cuTensorMapEncodeTiled is not available");
  g_encode = (PFN_cuTensorMapEncodeTiled_v12000)fn;
  return 0;
}

// Tensor map of one operand plane with row pitch ld elements: K-major [rows, K] or MN-major [K, rows].
// box = {inner, outer} extents in elements (K-major: {k, rows}, MN-major: {mn, k}).  The error
// messages name the plane (`plane`, `pitch`) and the encoding (`enc`, after the function name).
inline int make_map(CUtensorMap* map, CUtensorMapDataType dtype, const void* ptr, int64_t rows, int64_t K,
                    int64_t ld, bool mn_major, int box_inner, int box_outer, CUtensorMapSwizzle swizzle,
                    const char* plane, const char* pitch, const char* enc) {
  const int64_t esize = dtype == CU_TENSOR_MAP_DATA_TYPE_FLOAT32 ? 4 : 2;
  if ((reinterpret_cast<uintptr_t>(ptr) & 15) != 0) TNN_FAIL(std::string(plane) + " must be 16-byte aligned");
  if (ld * esize % 16 != 0)
    TNN_FAIL(std::string(pitch) + " must be a multiple of " + std::to_string(16 / esize) + " elements");
  cuuint64_t dims[2] = {(cuuint64_t)(mn_major ? rows : K), (cuuint64_t)(mn_major ? K : rows)};
  cuuint64_t strides[1] = {(cuuint64_t)(ld * esize)};
  cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(map, dtype, 2, (void*)ptr, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    TNN_FAIL(std::string("cuTensorMapEncodeTiled") + enc + " failed with code " + std::to_string((int)r));
  return 0;
}

// checks every GEMM entry point makes; `empty` = the output has no elements, nothing to launch
inline int gemm_entry_checks(const char* who, int64_t M, int64_t N, int64_t K, bool& empty) {
  TNN_REQUIRE_INIT();
  empty = M <= 0 || N <= 0;
  if (empty) return 0;
  if (K <= 0) TNN_FAIL(std::string(who) + ": K must be positive");
  if (M > 2147483647LL || N > 2147483647LL || K > 2147483647LL) TNN_FAIL(std::string(who) + ": extent above int32");
  return get_encode_fn();
}

// SMs the persistent grids leave free (tnn_set_gemm_reserved_sms): room for an NCCL kernel running
// beside the backward pass (comm.cu)
inline int g_reserved_sms = 0;

// CTA groups (pairs, or clusters of `cluster` CTAs) a persistent grid may occupy
inline int max_groups(int cluster) { return std::max(1, (ctx().sm_count - g_reserved_sms) / cluster); }

// Split-K arrival counters, one per output tile, for both kernels.  One buffer serves every launch:
// all GEMMs run on the compute stream (ctx().stream), and each launch that splits clears the
// counters it uses on that stream before it runs, so no launch sees another's counts.
constexpr int MAX_FLAG_TILES = 1 << 16;
inline unsigned int* g_tile_flags = nullptr;

struct TailPlan {
  int t_full, tail_split;   // see WorkUnits
};

// Tail split: when the `units` scheduling units leave a ragged last wave on `groups` CTA groups,
// the units of that wave are cut into 2 or 4 K ranges, as long as the last wave still fits and every
// range keeps at least min_kb K blocks.  Measured on the 4096x4096x8192 dW product (256 tiles, 74
// CTA pairs): see profiles/.  The ReLU epilogue (flags & 2) needs the complete sum, so it never
// splits; nor does a launch with more than MAX_FLAG_TILES output tiles (flag_tiles).
inline TailPlan plan_tail(int flags, int64_t units, int64_t flag_tiles, int groups, int64_t num_kb, int min_kb) {
  TailPlan p{(int)units, 1};
  if ((flags & 2) || flag_tiles > MAX_FLAG_TILES) return p;
  const int64_t rem = units % groups;
  if (rem > 0) {
    int s = 1;
    while (s < 4 && rem * (s * 2) <= groups && num_kb / (s * 2) >= min_kb) s *= 2;
    if (s > 1) p = {(int)(units - rem), s};
  }
  return p;
}

// the counters of a split launch's flag_tiles output tiles, cleared on the compute stream
inline int clear_tile_flags(const TailPlan& p, int64_t flag_tiles) {
  if (p.tail_split > 1) {
    if (!g_tile_flags) TNN_CUDA(cudaMalloc(&g_tile_flags, MAX_FLAG_TILES * sizeof(unsigned int)));
    TNN_CUDA(cudaMemsetAsync(g_tile_flags, 0, (size_t)flag_tiles * sizeof(unsigned int), ctx().stream));
  }
  return 0;
}

// Persistent launch of KERN on the compute stream: one cluster of CL CTAs per CTA group, as many
// groups as there are work units, at most `groups`.  cap_coresident: also at most as many clusters as
// can be resident at once -- clusters of 4 do not tile every GPC (B200: 33 of the 37 that 148 SMs
// would hold), and a cluster that cannot start waits for a whole one to finish.  `family` is the
// per-launch profiling family (tnn_prof_enable).
template <auto KERN, typename... Args>
int launch_persistent(int CL, int threads, int smem_bytes, int64_t units, int groups, bool cap_coresident,
                      int family, Args... args) {
  static bool attr_set = false;   // one per kernel instantiation
  if (!attr_set) {
    TNN_CUDA(cudaFuncSetAttribute(KERN, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    attr_set = true;
  }
  groups = (int)std::min<int64_t>(units, groups);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(groups * CL));
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = ctx().stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (cap_coresident) {
    static int max_clusters = 0;
    if (!max_clusters) {
      TNN_CUDA(cudaOccupancyMaxActiveClusters(&max_clusters, KERN, &cfg));
      if (max_clusters < 1) max_clusters = 1;
    }
    if (groups > max_clusters) cfg.gridDim = dim3((unsigned)(max_clusters * CL));
  }
  prof_begin(family);
  TNN_CUDA(cudaLaunchKernelEx(&cfg, KERN, args...));
  ctx().launches++;
  prof_end(family);
  return 0;
}

}  // namespace tc
}  // namespace tnn

// Tensor-core GEMM for ops.py:150-163 (dot_: A@B, grad@B.T, A.T@grad), scaled two-plane fp16 split:
//
//     X = x * 2^e                        e per TENSOR, so that max|X| lies in [2^14, 2^15)
//     hf = fp16(X)                       11 significant bits (the same mantissa tf32(x) keeps)
//     l  = fp16(X - hf)                  the next 11 bits
//     A*B ~= 2^-(ea+eb) * ( l_A*hf_B + hf_A*l_B + hf_A*hf_B )          fp32 accumulation in TMEM
//
// i.e. the 3xTF32 expansion with every factor held in 16 bits: 4 bytes of planes per element instead
// of 8 and three kind::f16 MMAs per K=16 step (the tensor pipe's fastest dense fp32-accumulating
// rate) instead of one kind::tf32 + two kind::f16.  (kind::f16 does not take an f16 and a bf16 operand
// in one instruction -- tried, "illegal instruction" -- so both planes are fp16.)
// Element error: |X - hf - l| <= 2^-22 |X| while the residual is a normal fp16 number (|X| >= 2^-3),
// <= 2^-25 absolute below, i.e.
//     err(a_ik) <= 2^-20 * max(|a_ik|, 2^-19 * max|A|)        (2^-25 <= 2^-39 max|X|)
// -- at least the mixed tf32/bf16 split's accuracy for every element within 19 binades of the
// tensor's largest, an absolute floor of 2^-39 max|A| (five orders below fp32's own rounding of the
// large entries) under that; the dropped l*l term is 2^-22 relative.  That is a tensor-relative
// bound, so the split kernel guards it ON THE DEVICE: it counts the non-zero elements below the
// floor (|X| < 2^-5) and flags the tensor `unsafe` when they are more than 1/256 of the non-zeros
// (rows or columns on wildly different scales, exponents spread over tens of binades) or when the
// tensor holds NaN/Inf.  The f16 GEMM returns at once for an unsafe operand and the conditional
// mixed-split launches that follow it (gemm_tc.cu: tnn_split_tf32_bf16_cond,
// tnn_gemm_tf32_bf16x2_cond) do the product instead -- no host round trip, capturable in a graph.
//
// Kernel: same skeleton as gemm_tc.cu (persistent CTA pairs, cta_group::2, tile 256 x 256, warp 0 TMA
// producer, warp 1 MMA issuer, warps 4-11 drain TMEM chunks into fp32 registers with RN adds), with
// 64-wide K blocks (128-byte rows of 16-bit elements, SWIZZLE_128B both majors), 3 stages x 64 KB.
// Algorithmic work 2*M*N*K flop per call; the tensor pipe executes 3x that at the bf16/fp16 rate;
// operand bytes 4*(M+N)*K.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "tc_gemm.cuh"

namespace tnn {
namespace f16 {

using namespace tnn::tc;

#ifndef TNN_F16_BK
#define TNN_F16_BK 64
#endif
#ifndef TNN_F16_STAGES
#define TNN_F16_STAGES (192 / TNN_F16_BK)
#endif
constexpr int BK = TNN_F16_BK;               // 16-bit elements per K block: 64 (128-byte rows) or 32
constexpr int ROWS = 128;                    // rows of A and rows of B staged per CTA
constexpr int UMMA_N = 256;
constexpr int TILE_M = 256;                  // CTA pair
constexpr int UMMA_K = 16;
constexpr int PLANE_BYTES = ROWS * BK * 2;   // 16 KB
constexpr int STAGE_BYTES = 4 * PLANE_BYTES; // A.hf, A.l, B.hf, B.l
constexpr int STAGES = TNN_F16_STAGES;
constexpr int CHUNK_KB = 256 / BK;           // 256 k per TMEM accumulator chunk (as gemm_tc.cu)
#ifndef TNN_F16_THREADS
#define TNN_F16_THREADS 384
#endif
// 384 threads: warpgroup 0 = TMA producer warp, MMA issuer warp, 2 idle warps (setmaxnreg.dec 40);
// warpgroups 1-2 = epilogue (setmaxnreg.inc 216: 128 tile sums + a 32-column TMEM chunk per thread).
// (TNN_F16_THREADS=320 -- ten warps, no setmaxnreg -- was tried to give ptxas a larger launch-time
// budget: registers are allocated per 4 warps, so the budget stays 168 and the spills grow.)
constexpr int NUM_THREADS = TNN_F16_THREADS;
constexpr int EPI_WARP0 = NUM_THREADS == 320 ? 2 : 4;   // first epilogue warp
constexpr uint32_t TMEM_COLS = 512;
constexpr int EPI_PATCH_BYTES = 8 * 4096;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + 256 + EPI_PATCH_BYTES;
#ifndef TNN_F16_KBOX_ROWS
#define TNN_F16_KBOX_ROWS 128
#endif
constexpr int KBOX_ROWS = TNN_F16_KBOX_ROWS;   // rows per TMA box of a K-major plane (BK = 64: 128-byte rows)
constexpr int MN_BOX_BYTES = 64 * BK * 2;    // one {64 mn, 64 k} box
constexpr float SMALL_LIMIT = 0.03125f;      // 2^-5: below it the residual plane is subnormal
constexpr unsigned int GUARD_FRACTION = 256; // unsafe when small non-zeros * 256 > non-zeros

// per-operand device record (32 bytes).  absmax is filled by stats_kernel or a producer's epilogue;
// the rest by split_f16_kernel.  Word 3 (`safe`) is what the conditional kernels of gemm_tc.cu read.
struct Meta {
  unsigned int absmax;      // bits of max |x| (NaN sorts above Inf)
  unsigned int need_stats;  // set by the fallback product: absmax of its result was not recorded
  int exp;                  // planes hold x * 2^exp
  int safe;                 // 1: planes are valid and inside the guard
  unsigned int n_small;     // non-zero elements with |X| < SMALL_LIMIT
  unsigned int n_nz;        // non-zero elements
  unsigned int ticket;      // CTAs of the split kernel that have finished
  unsigned int pad;
};

// scale exponent from the tensor's largest magnitude; ok = 0 for NaN/Inf or a tensor so small that
// the scale itself would overflow
__device__ __forceinline__ void meta_scale(unsigned int amax_bits, int& e, int& ok) {
  e = 0;
  ok = 1;
  if (amax_bits == 0u) return;                       // all zeros
  if (amax_bits >= 0x7F800000u) { ok = 0; return; }
  const int ex = (int)(amax_bits >> 23) - 127;
  if (ex < -112) { ok = 0; return; }
  e = 14 - ex;
}

__device__ __forceinline__ float pow2f(int e) {      // e in [-126, 127]
  return __int_as_float((e + 127) << 23);
}

// K-major, SWIZZLE_128B: rows of 128 B, 8-row groups 1024 B apart; a K=16 step advances 32 B.
// MN-major, SWIZZLE_128B: {64 mn, 64 k} boxes of 8192 B (k-row j at j*128 B); 8-k groups 1024 B
// apart (SBO), 64-element M/N chunks one box apart (LBO); a K=16 step advances 2048 B.
template <bool MN>
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(MN ? (MN_BOX_BYTES >> 4) : 1) << 16;
  // K-major rows are BK*2 bytes: 128 B -> SWIZZLE_128B, 8-row groups 1024 B apart; 64 B (BK = 32) ->
  // SWIZZLE_64B, groups 512 B apart.  MN-major k-rows are always 128 B (64 elements).
  d |= (uint64_t)(((MN || BK == 64) ? 1024 : 512) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)((MN || BK == 64) ? 2 : 4) << 61;
  return d;
}
// D = F32; a_fmt / b_fmt: 0 = F16, 1 = BF16
__host__ __device__ constexpr uint32_t make_idesc(int a_fmt, int b_fmt, bool a_mn, bool b_mn) {
  return (1u << 4) | ((uint32_t)a_fmt << 7) | ((uint32_t)b_fmt << 10) | ((a_mn ? 1u : 0u) << 15) |
         ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(UMMA_N >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
}

// flags: 1 accumulate into D, 2 ReLU in place, 8 statistics of relu(D) instead of D
// CL = 2: one CTA pair per tile.  CL = 4: a cluster of two pairs on adjacent tile columns (tm, 2j)
// and (tm, 2j+1); they need the same A rows, so each CTA fetches only half of its A tile and TMA
// multicasts it to its counterpart in the other pair (A's L2->SM traffic halves: 48 KB instead of
// 64 KB per CTA per K block).  Both pairs then move through the K blocks in lock-step: a stage is
// refilled when BOTH pairs' MMAs have released it (empty barriers count two commits).
template <bool A_MN, bool B_MN, int CL>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_f16x3_kernel(const __grid_constant__ CUtensorMap map_a_h, const __grid_constant__ CUtensorMap map_a_l,
                  const __grid_constant__ CUtensorMap map_b_h, const __grid_constant__ CUtensorMap map_b_l,
                  float* __restrict__ D, int64_t ldd, int M, int N, int K,
                  const float* __restrict__ bias, int flags, int t_full, int tail_split,
                  unsigned int* __restrict__ tile_flags, float* __restrict__ act_out,
                  const float* __restrict__ mask_src, const Meta* __restrict__ meta_a,
                  const Meta* __restrict__ meta_b, Meta* __restrict__ stat_out, int group_m) {
  // operands outside the guard: the conditional mixed-split launches behind this one take over
  if (!(meta_a->safe && meta_b->safe)) return;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const Barriers<STAGES> bar{smem_base + STAGES * STAGE_BYTES};

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cl_rank = cluster_ctarank();          // 0..CL-1
  const uint32_t pair = cl_rank >> 1;                  // which tile column of the cluster's two
  const uint32_t cta_rank = cl_rank & 1u;              // rank inside the CTA pair
  const bool leader = cta_rank == 0;
  const uint16_t pair_mask = (uint16_t)(3u << (2 * pair));

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_h);
    tma_prefetch_desc(&map_a_l);
    tma_prefetch_desc(&map_b_h);
    tma_prefetch_desc(&map_b_l);
    // empty: one tcgen05.commit per pair that reads (or feeds) a stage; tmem_empty: one arrival per
    // epilogue warp of both CTAs
    bar.init(CL / 2, 16);
  }
  const uint32_t tmem_base = tmem_setup<2>(bar, smem_gen + STAGES * STAGE_BYTES, warp, TMEM_COLS);

  const int tiles_m = (M + TILE_M - 1) / TILE_M;
  const int tiles_n = (N + UMMA_N - 1) / UMMA_N;
  const int tiles_ns = CL == 4 ? (tiles_n + 1) / 2 : tiles_n;   // scheduling units per tile row
  const int num_tiles = tiles_m * tiles_ns;
  const int num_kb = (K + BK - 1) / BK;
  const int group = blockIdx.x / CL;
  const int num_groups = gridDim.x / CL;
  const WorkUnits work(t_full, tail_split, num_tiles, num_kb);

  if (warp == 0) {
    // ================= TMA producer =================
    if constexpr (NUM_THREADS == 384) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = group; u < work.num_units; u += num_groups) {
        int t, sp, kb_begin, kb_end;
        work.decode(u, t, sp, kb_begin, kb_end);
        int tm, tn;
        tile_coords((flags & 32) ? num_tiles - 1 - t : t, tiles_m, tiles_ns, group_m, tm, tn);
        if constexpr (CL == 4) tn = 2 * tn + (int)pair;
        const int row_a = tm * TILE_M + (int)cta_rank * ROWS;
        const int row_b = tn * UMMA_N + (int)cta_rank * ROWS;   // (beyond N for the odd pair of a ragged row: zero fill)
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(bar.empty(stage), phase ^ 1u);
          const uint32_t sa_h = smem_base + stage * STAGE_BYTES;
          const uint32_t sa_l = sa_h + PLANE_BYTES;
          const uint32_t sb_h = sa_h + 2 * PLANE_BYTES;
          const uint32_t sb_l = sa_h + 3 * PLANE_BYTES;
          if (leader) mbar_expect_tx(bar.full(stage), (uint32_t)STAGE_BYTES * 2u);
          const int k0 = kb * BK;
          if (flags & 128) {
            // TIMING EXPERIMENT (TNN_EXP_FLAGS, results are wrong): no operand fetch
            if (leader)
              asm volatile("mbarrier.complete_tx.shared::cta.b64 [%0], %1;" ::"r"(bar.full(stage)), "r"((uint32_t)STAGE_BYTES * 2u) : "memory");
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            continue;
          }
#ifdef TNN_F16_PREFETCH
          if (kb + TNN_F16_PREFETCH < kb_end) {
            // pull the boxes of a later K block into L2 now, so that the load that fills the stage
            // then is an L2 hit rather than a DRAM round trip
            const int kp = (kb + TNN_F16_PREFETCH) * BK;
            if constexpr (A_MN) {
#pragma unroll
              for (int j = 0; j < ROWS / 64; ++j) {
                tma_prefetch_l2_2d(&map_a_l, row_a + 64 * j, kp);
                tma_prefetch_l2_2d(&map_a_h, row_a + 64 * j, kp);
              }
            } else {
              tma_prefetch_l2_2d(&map_a_l, kp, row_a);
              tma_prefetch_l2_2d(&map_a_h, kp, row_a);
            }
            if constexpr (B_MN) {
#pragma unroll
              for (int j = 0; j < ROWS / 64; ++j) {
                tma_prefetch_l2_2d(&map_b_h, row_b + 64 * j, kp);
                tma_prefetch_l2_2d(&map_b_l, row_b + 64 * j, kp);
              }
            } else {
              tma_prefetch_l2_2d(&map_b_h, kp, row_b);
              tma_prefetch_l2_2d(&map_b_l, kp, row_b);
            }
          }
#endif
          if constexpr (CL == 4) {
            // this CTA's half (64 rows: 8 KB per plane) of the A tile, to itself and to the CTA of the
            // same pair rank in the other pair; the other half arrives from there
            const uint16_t mc = (uint16_t)((1u << cta_rank) | (1u << (cta_rank + 2)));
            const uint32_t off = pair * (uint32_t)(PLANE_BYTES / 2);
            const int ra = row_a + 64 * (int)pair;
            if constexpr (A_MN) {
              tma_load_2d_pair_mc(sa_l + off, &map_a_l, bar.full(stage), ra, k0, mc);
              tma_load_2d_pair_mc(sa_h + off, &map_a_h, bar.full(stage), ra, k0, mc);
            } else {
              tma_load_2d_pair_mc(sa_l + off, &map_a_l, bar.full(stage), k0, ra, mc);
              tma_load_2d_pair_mc(sa_h + off, &map_a_h, bar.full(stage), k0, ra, mc);
            }
          } else if constexpr (A_MN) {
#pragma unroll
            for (int j = 0; j < ROWS / 64; ++j) {
              tma_load_2d<2>(sa_l + j * MN_BOX_BYTES, &map_a_l, bar.full(stage), row_a + 64 * j, k0);
              tma_load_2d<2>(sa_h + j * MN_BOX_BYTES, &map_a_h, bar.full(stage), row_a + 64 * j, k0);
            }
          } else {
#pragma unroll
            for (int j = 0; j < ROWS / KBOX_ROWS; ++j) {
              tma_load_2d<2>(sa_l + j * KBOX_ROWS * 128, &map_a_l, bar.full(stage), k0, row_a + j * KBOX_ROWS);
              tma_load_2d<2>(sa_h + j * KBOX_ROWS * 128, &map_a_h, bar.full(stage), k0, row_a + j * KBOX_ROWS);
            }
          }
          if constexpr (B_MN) {
#pragma unroll
            for (int j = 0; j < ROWS / 64; ++j) {
              tma_load_2d<2>(sb_h + j * MN_BOX_BYTES, &map_b_h, bar.full(stage), row_b + 64 * j, k0);
              tma_load_2d<2>(sb_l + j * MN_BOX_BYTES, &map_b_l, bar.full(stage), row_b + 64 * j, k0);
            }
          } else {
#pragma unroll
            for (int j = 0; j < ROWS / KBOX_ROWS; ++j) {
              tma_load_2d<2>(sb_h + j * KBOX_ROWS * 128, &map_b_h, bar.full(stage), k0, row_b + j * KBOX_ROWS);
              tma_load_2d<2>(sb_l + j * KBOX_ROWS * 128, &map_b_l, bar.full(stage), k0, row_b + j * KBOX_ROWS);
            }
          }
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA only) =================
    if constexpr (NUM_THREADS == 384) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc(0, 0, A_MN, B_MN);      // f16 x f16 -> f32
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
#ifdef TNN_F16_PROBE
      long long w_full = 0, w_empty = 0, t_begin = clock64();
#endif
      for (int u = group; u < work.num_units; u += num_groups) {
        int t, sp, kb_begin, kb_end;
        work.decode(u, t, sp, kb_begin, kb_end);
        for (int kb0 = kb_begin; kb0 < kb_end; kb0 += CHUNK_KB) {
#ifdef TNN_F16_PROBE
          long long p0 = clock64();
#endif
          mbar_wait(bar.tempty(acc), acc_phase ^ 1u);
#ifdef TNN_F16_PROBE
          w_empty += clock64() - p0;
#endif
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + (uint32_t)(acc * UMMA_N);
          const int kb1 = min(kb0 + CHUNK_KB, kb_end);
          for (int kb = kb0; kb < kb1; ++kb) {
#ifdef TNN_F16_PROBE
            long long p1 = clock64();
#endif
            mbar_wait(bar.full(stage), phase);
#ifdef TNN_F16_PROBE
            w_full += clock64() - p1;
#endif
            tc_fence_after();
            const uint32_t sa_h = smem_base + stage * STAGE_BYTES;
            const uint32_t sa_l = sa_h + PLANE_BYTES;
            const uint32_t sb_h = sa_h + 2 * PLANE_BYTES;
            const uint32_t sb_l = sa_h + 3 * PLANE_BYTES;
            if (!(flags & 256))   // (256: timing experiment, no MMA issued)
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {
              const uint32_t koff_a = (uint32_t)(k * (A_MN ? 2048 : 32));
              const uint32_t koff_b = (uint32_t)(k * (B_MN ? 2048 : 32));
              const uint64_t da_h = make_desc<A_MN>(sa_h + koff_a);
              const uint64_t da_l = make_desc<A_MN>(sa_l + koff_a);
              const uint64_t db_h = make_desc<B_MN>(sb_h + koff_b);
              const uint64_t db_l = make_desc<B_MN>(sb_l + koff_b);
              // small terms first; the first MMA of a chunk overwrites the accumulator
              umma_bf16<2>(tmem_d, da_l, db_h, idesc, (kb != kb0 || k != 0) ? 1u : 0u);
              umma_bf16<2>(tmem_d, da_h, db_l, idesc, 1u);
              umma_bf16<2>(tmem_d, da_h, db_h, idesc, 1u);
            }
            umma_commit_pair_mask(bar.empty(stage), CL == 4 ? (uint16_t)15 : (uint16_t)3);
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
          umma_commit_pair_mask(bar.tfull(acc), pair_mask);
          if (++acc == 2) {
            acc = 0;
            acc_phase ^= 1u;
          }
        }
      }
#ifdef TNN_F16_PROBE
      if (group == 0 || group == 37)
        printf("probe group %d: loop %lld cycles, wait full %lld, wait tmem-empty %lld\n", group,
               clock64() - t_begin, w_full, w_empty);
#endif
    }
  } else if (warp < EPI_WARP0) {
    if constexpr (NUM_THREADS == 384) asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
  } else {
    // ================= epilogue =================
    if constexpr (NUM_THREADS == 384) asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    const int quad = warp & 3;                       // TMEM lanes [32*quad, 32*quad+32): fixed by warp id % 4
    const int half = (warp - EPI_WARP0) >> 2;        // accumulator columns [128*half, 128*half+128)
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool relu = flags & 2;
    // 2^-(ea+eb) as two factors (each a normal float; the intermediate lies between the scaled
    // sum and the result, so it cannot overflow or underflow unless the result does)
    const int ec = -(meta_a->exp + meta_b->exp);
    const float f1 = pow2f(ec / 2), f2 = pow2f(ec - ec / 2);
    unsigned int st_max = 0u;
#ifdef TNN_F16_PROBE
    long long ep_wait = 0, ep_store = 0;
    const long long ep_begin = clock64();
#endif
    for (int u = group; u < work.num_units; u += num_groups) {
      int t, sp, kb_begin, kb_end;
      work.decode(u, t, sp, kb_begin, kb_end);
      const bool accumulate = (flags & 1) || sp > 0;
      const bool final_unit = (u < t_full || sp + 1 == tail_split);
      const bool emit_act = act_out != nullptr && final_unit;
      const bool want_stats = stat_out != nullptr && final_unit;
      const float* bias_u = sp == 0 ? bias : nullptr;
      int tm, tn;
      tile_coords((flags & 32) ? num_tiles - 1 - t : t, tiles_m, tiles_ns, group_m, tm, tn);
      if constexpr (CL == 4) tn = 2 * tn + (int)pair;
      const bool tile_valid = tn < tiles_n;            // (the odd pair of a ragged tile row computes zeros)
      const int flag_idx = tm * tiles_n + tn;
      const int col0 = tn * UMMA_N + half * 128;
      float sum[128];
#pragma unroll
      for (int j = 0; j < 128; ++j) sum[j] = 0.f;
      for (int kb0 = kb_begin; kb0 < kb_end; kb0 += CHUNK_KB) {
#ifdef TNN_F16_PROBE
        const long long q0 = clock64();
#endif
        mbar_wait(bar.tfull(acc), acc_phase);
#ifdef TNN_F16_PROBE
        ep_wait += clock64() - q0;
#endif
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) +
                               (uint32_t)(acc * UMMA_N + half * 128);
        // The chunk drain here and the split-K ordering wait below are written out in this kernel
        // (gemm_tc.cu has its own copies) rather than taken from tc_gemm.cuh: as shared helpers they
        // change this kernel's register allocation and spill layout, and this is the hot kernel.
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          uint32_t r[32];
          tmem_ld_32x32b_x32(taddr + (uint32_t)(c * 32), r);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) sum[c * 32 + j] += __uint_as_float(r[j]);
        }
        tmem_hand_back<true>(bar.tempty(acc), 2 * pair, lane);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
      if (sp > 0 && tile_valid) {
        if (lane == 0) {
          const unsigned int need = (unsigned int)(sp * 16);
          unsigned int seen;
          long long t0 = clock64();
          do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(tile_flags + flag_idx) : "memory");
            if (clock64() - t0 > 8000000000LL) {
              printf("tnn gemm_f16: split-K ordering wait timed out (tile %d split %d)\n", t, sp);
              __trap();
            }
          } while (seen < need);
        }
        __syncwarp();
        __threadfence();
      }
#ifdef TNN_F16_PROBE
      const long long q1 = clock64();
#endif
      {
        // ---- store the tile.  Each warp bounces its 32 x 32 blocks through a private 4 KB swizzled
        // shared-memory patch and comes back with 8 lanes per row, so every global access is 4 full
        // 128-byte lines.  The MMA issuer can only run two chunks ahead while the epilogue warps are
        // here, so this phase is on the critical path: the code is kept SMALL (one rolled copy of
        // the store loop; a fully unrolled version was 8,000 SASS instructions that every warp
        // walked once per tile, instruction-fetch-bound at ~40 k cycles per tile).
        const int row_base = tm * TILE_M + (int)cta_rank * ROWS + quad * 32;
        float4* patch = reinterpret_cast<float4*>(smem_gen + STAGES * STAGE_BYTES + 256) + (warp - EPI_WARP0) * 256;
        const bool rows_aligned = (ldd % 4 == 0) && ((reinterpret_cast<uintptr_t>(D) & 15) == 0);
        const bool act_aligned = !emit_act || (((reinterpret_cast<uintptr_t>(act_out) |
                                                  reinterpret_cast<uintptr_t>(mask_src)) & 15) == 0);
        const bool want_mask = emit_act && mask_src != nullptr;
        const bool want_relu_side = !want_mask && (emit_act || (flags & 8));
        const float* pre_src = accumulate ? D : (want_mask ? mask_src : nullptr);
        const int rr = lane >> 3, c4l = lane & 7;
#pragma unroll 1
        for (int cb = 0; cb < 4; ++cb) {
          const int colb = col0 + cb * 32;
          if (colb >= N) break;                                 // warp-uniform
          patch_write<true>(cb, sum, patch, lane, f1, f2, bias_u, colb, N);
          __syncwarp();
          const int gcol = colb + c4l * 4;
          if (rows_aligned && act_aligned && colb + 32 <= N) {
            if (pre_src == nullptr) {
              // plain / relu / statistics: nothing to read back.  Unrolled with everything that does
              // not change hoisted: per row group one 128-bit shared-memory load at a constant
              // offset, one 128-bit store through a running pointer (a rolled version that
              // rebuilt its indices every iteration spent ~21 k cycles per tile here).
              const int nrows = min(32, M - row_base);          // rows of this warp's block inside M
              const float4* pp0 = patch + rr * 8 + (c4l ^ rr);              // rows rr, rr+8, ...  (r & 7 = rr)
              const float4* pp1 = patch + (rr + 4) * 8 + (c4l ^ (rr + 4));  // rows rr+4, rr+12, ... (r & 7 = rr+4)
              float* dp = D + (int64_t)(row_base + rr) * ldd + gcol;
              float* ap = emit_act ? act_out + (int64_t)(row_base + rr) * ldd + gcol : nullptr;
              const int64_t step = 4 * ldd;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                if (4 * i + rr < nrows) {
                  float4 v = (i & 1) ? pp1[(i >> 1) * 64] : pp0[(i >> 1) * 64];
                  if (relu) {
                    v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f);
                    v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
                  }
                  *reinterpret_cast<float4*>(dp) = v;
                  if (want_relu_side) {                        // ReLU(D), NaN-propagating like np.clip
                    v.x = v.x < 0.f ? 0.f : v.x; v.y = v.y < 0.f ? 0.f : v.y;
                    v.z = v.z < 0.f ? 0.f : v.z; v.w = v.w < 0.f ? 0.f : v.w;
                    if (emit_act) *reinterpret_cast<float4*>(ap) = v;
                  }
                  if (want_stats)
                    st_max = max(max(st_max, __float_as_uint(v.x) & 0x7FFFFFFFu),
                                 max(max(__float_as_uint(v.y) & 0x7FFFFFFFu, __float_as_uint(v.z) & 0x7FFFFFFFu),
                                     __float_as_uint(v.w) & 0x7FFFFFFFu));
                }
                dp += step;
                if (emit_act) ap += step;
              }
            } else {
              // accumulate-into-D and / or the ReLU-backward mask: whatever has to be READ first is
              // fetched for all 8 row groups up front (8 independent 128-bit loads in flight)
              const int nrows = min(32, M - row_base);
              const float4* pp0 = patch + rr * 8 + (c4l ^ rr);
              const float4* pp1 = patch + (rr + 4) * 8 + (c4l ^ (rr + 4));
              const int64_t off0 = (int64_t)(row_base + rr) * ldd + gcol, step = 4 * ldd;
              float4 pre[8];
              {
                const float* sp_ = pre_src + off0;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                  if (4 * i + rr < nrows) pre[i] = *reinterpret_cast<const float4*>(sp_);
                  sp_ += step;
                }
              }
              float* dp = D + off0;
              float* ap = emit_act ? act_out + off0 : nullptr;
              const float* mp = (want_mask && accumulate) ? mask_src + off0 : nullptr;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                if (4 * i + rr < nrows) {
                  float4 v = (i & 1) ? pp1[(i >> 1) * 64] : pp0[(i >> 1) * 64];
                  if (accumulate) {
                    v.x += pre[i].x; v.y += pre[i].y; v.z += pre[i].z; v.w += pre[i].w;
                  }
                  if (relu) {
                    v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f);
                    v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
                  }
                  *reinterpret_cast<float4*>(dp) = v;
                  if (want_mask) {
                    // act = D * (pre-activation >= 0): the ReLU gradient mask of ops.py:336-343
                    const float4 z = accumulate ? *reinterpret_cast<const float4*>(mp) : pre[i];
                    v.x = z.x >= 0.f ? v.x : v.x * 0.f; v.y = z.y >= 0.f ? v.y : v.y * 0.f;
                    v.z = z.z >= 0.f ? v.z : v.z * 0.f; v.w = z.w >= 0.f ? v.w : v.w * 0.f;
                  } else if (want_relu_side) {
                    v.x = v.x < 0.f ? 0.f : v.x; v.y = v.y < 0.f ? 0.f : v.y;
                    v.z = v.z < 0.f ? 0.f : v.z; v.w = v.w < 0.f ? 0.f : v.w;
                  }
                  if (emit_act) *reinterpret_cast<float4*>(ap) = v;
                  if (want_stats)
                    st_max = max(max(st_max, __float_as_uint(v.x) & 0x7FFFFFFFu),
                                 max(max(__float_as_uint(v.y) & 0x7FFFFFFFu, __float_as_uint(v.z) & 0x7FFFFFFFu),
                                     __float_as_uint(v.w) & 0x7FFFFFFFu));
                }
                dp += step;
                if (emit_act) ap += step;
                if (mp) mp += step;
              }
            }
          } else {
            // ragged right edge or unaligned rows: element by element
#pragma unroll 1
            for (int i = 0; i < 8; ++i) {
              const int r = 4 * i + rr, grow = row_base + r;
              if (grow >= M) break;
              const float4 v4 = patch[r * 8 + (c4l ^ (r & 7))];
              const float s[4] = {v4.x, v4.y, v4.z, v4.w};
#pragma unroll 1
              for (int k = 0; k < 4; ++k) {
                if (gcol + k >= N) break;
                const int64_t off = (int64_t)grow * ldd + gcol + k;
                float x = k == 0 ? s[0] : (k == 1 ? s[1] : (k == 2 ? s[2] : s[3]));
                if (accumulate) x += D[off];
                if (relu) x = fmaxf(x, 0.f);
                D[off] = x;
                float a = x;
                if (want_mask) a = mask_src[off] >= 0.f ? x : x * 0.f;
                else if (want_relu_side) a = x < 0.f ? 0.f : x;
                if (emit_act) act_out[off] = a;
                if (want_stats) st_max = max(st_max, __float_as_uint(a) & 0x7FFFFFFFu);
              }
            }
          }
          __syncwarp();
        }
      }
#ifdef TNN_F16_PROBE
      ep_store += clock64() - q1;
#endif
      if (u >= t_full && sp + 1 < tail_split && tile_valid) splitk_publish(tile_flags, flag_idx, lane);
    }
#ifdef TNN_F16_PROBE
    if ((group == 0 || group == 37) && warp == 4 && lane == 0 && cta_rank == 0)
      printf("probe group %d epilogue warp 4: total %lld cycles, waiting for a chunk %lld, storing tiles %lld\n",
             group, clock64() - ep_begin, ep_wait, ep_store);
#endif
    if (stat_out != nullptr) {
      // integer max is exact and order-independent: the record does not depend on timing
      st_max = __reduce_max_sync(0xFFFFFFFFu, st_max);
      if (lane == 0 && st_max) atomicMax(&stat_out->absmax, st_max);
    }
  }

  tmem_teardown<2>(warp, tmem_base, TMEM_COLS);
}

// ---- statistics + split ---------------------------------------------------------------------------

// max |x| of (relu_mode ? relu(x) : x) over n elements -> meta->absmax (integer atomicMax)
__global__ void __launch_bounds__(256)
stats_kernel(const float* __restrict__ x, int64_t n, Meta* __restrict__ meta, int relu_mode, int vec,
             int only_if_needed) {
  if (only_if_needed && !meta->need_stats) return;
  unsigned int mx = 0u;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  auto take = [&](float v) {
    if (relu_mode && v < 0.f) v = 0.f;
    mx = max(mx, __float_as_uint(v) & 0x7FFFFFFFu);
  };
  if (vec) {
    const int64_t n4 = n / 4;
    const float4* x4 = reinterpret_cast<const float4*>(x);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
      const float4 t = x4[i];
      take(t.x); take(t.y); take(t.z); take(t.w);
    }
    for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) take(x[i]);
  } else {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) take(x[i]);
  }
  mx = __reduce_max_sync(0xFFFFFFFFu, mx);
  __shared__ unsigned int s_mx[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) s_mx[warp] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < 8; ++w) mx = max(mx, s_mx[w]);
    if (mx) atomicMax(&meta->absmax, mx);
  }
}

// x [R, C] (relu_mode: relu(x)) -> hf = fp16(x 2^e), l = fp16(x 2^e - hf), pitch ld (multiple of 8,
// pad columns zeroed); e is derived from meta->absmax by every thread.  While writing, the kernel
// counts non-zero and "small" elements (integer atomics: order-independent); the last CTA to finish
// turns the counts into the `safe` flag.  8 B written per 4 B read.
__global__ void __launch_bounds__(256)
split_f16_kernel(const float* __restrict__ x, int64_t R, int64_t C, __half* __restrict__ hf,
                 __half* __restrict__ l16, int64_t ld, Meta* __restrict__ meta, int relu_mode,
                 int vec_in) {
  int e, ok;
  meta_scale(meta->absmax, e, ok);
  const float sc = ok ? pow2f(e) : 1.f;
  const int64_t gpr = ld / 8;
  const int64_t total = R * gpr;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned int n_small = 0u, n_nz = 0u;
  if (ok) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
      const int64_t r = i / gpr, c = (i - r * gpr) * 8;
      float v[8];
      if (vec_in && c + 7 < C) {
        const float4 t0 = *reinterpret_cast<const float4*>(x + r * C + c);
        const float4 t1 = *reinterpret_cast<const float4*>(x + r * C + c + 4);
        v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w;
        v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
      } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = (c + k < C) ? x[r * C + c + k] : 0.f;
      }
      union { __half2 h[4]; uint4 u; } ph, pl;
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float a = v[2 * k], b = v[2 * k + 1];
        if (relu_mode) { a = a < 0.f ? 0.f : a; b = b < 0.f ? 0.f : b; }
        a *= sc; b *= sc;
        n_nz += (a != 0.f) + (b != 0.f);
        n_small += (a != 0.f && fabsf(a) < SMALL_LIMIT) + (b != 0.f && fabsf(b) < SMALL_LIMIT);
        const __half2 h = __floats2half2_rn(a, b);
        const float2 hb = __half22float2(h);
        ph.h[k] = h;
        pl.h[k] = __floats2half2_rn(a - hb.x, b - hb.y);
      }
      *reinterpret_cast<uint4*>(hf + r * ld + c) = ph.u;
      *reinterpret_cast<uint4*>(l16 + r * ld + c) = pl.u;
    }
  }
  n_small = __reduce_add_sync(0xFFFFFFFFu, n_small);
  n_nz = __reduce_add_sync(0xFFFFFFFFu, n_nz);
  __shared__ unsigned int s_small[8], s_nz[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { s_small[warp] = n_small; s_nz[warp] = n_nz; }
  __syncthreads();
  if (threadIdx.x == 0) {
#pragma unroll
    for (int w = 1; w < 8; ++w) { n_small += s_small[w]; n_nz += s_nz[w]; }
    if (n_small) atomicAdd(&meta->n_small, n_small);
    if (n_nz) atomicAdd(&meta->n_nz, n_nz);
    __threadfence();
    if (atomicAdd(&meta->ticket, 1u) == gridDim.x - 1) {
      __threadfence();
      const unsigned int ts = *reinterpret_cast<volatile unsigned int*>(&meta->n_small);
      const unsigned int tn = *reinterpret_cast<volatile unsigned int*>(&meta->n_nz);
      meta->exp = e;
      meta->safe = (ok && (unsigned long long)ts * GUARD_FRACTION <= (unsigned long long)tn) ? 1 : 0;
    }
  }
}

// ---- host side ---------------------------------------------------------------------------------
// 16-bit plane.  K-major [rows, K]: box {64 k, box_rows}.  MN-major [K, rows]: box {64 mn, 64 k}.
// 128-byte swizzle both ways.
static int make_map(CUtensorMap* map, const void* ptr, int64_t rows, int64_t K, int64_t ld, bool mn_major,
                    int box_rows) {
  return tc::make_map(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, ptr, rows, K, ld, mn_major, mn_major ? 64 : BK,
                      mn_major ? BK : box_rows,
                      (mn_major || BK == 64) ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                      "f16 GEMM: operand plane", "f16 GEMM: operand pitch", " (f16 planes)");
}

static int g_group_m = -8;     // tile rasterisation: panels of 8 tile columns measured 1-2 % ahead of row-major;
                               // (TNN_F16_GROUP_M), see tile_coords
static bool g_reverse = true;  // tiles in descending order (TNN_F16_REVERSE=0: ascending): the product starts on
                               // the rows the split pass wrote last (still in L2) and ends on the rows the next
                               // split pass reads first; measured 8.33 -> 8.20 ms/step (same box, 3 runs each)
static int g_cluster = 2;      // 2: CTA pairs (default).  4: two pairs per cluster sharing A by TMA multicast
                               // (TNN_F16_CLUSTER=4): correct, -6 % time per tile round, but only 33 such
                               // clusters are co-resident on B200's 148 SMs (132 SMs busy, 8 rounds instead of
                               // 7 for 512 tiles), so it measures 3-20 % slower overall

template <bool A_MN, bool B_MN, int CL>
static int launch(float* D, int64_t ldd, const void* a_h, const void* a_l, int64_t lda, const void* b_h,
                  const void* b_l, int64_t ldb, int64_t M, int64_t N, int64_t K, const float* bias,
                  int flags, float* act_out, const float* mask_src, const Meta* meta_a,
                  const Meta* meta_b, Meta* stat_out) {
  CUtensorMap ma_h, ma_l, mb_h, mb_l;
  // (CL = 4: a CTA fetches half of its A tile -- 64 rows -- and receives the other half by multicast)
  if (make_map(&ma_h, a_h, M, K, lda, A_MN, CL == 4 ? 64 : KBOX_ROWS)) return 1;
  if (make_map(&ma_l, a_l, M, K, lda, A_MN, CL == 4 ? 64 : KBOX_ROWS)) return 1;
  if (make_map(&mb_h, b_h, N, K, ldb, B_MN, KBOX_ROWS)) return 1;
  if (make_map(&mb_l, b_l, N, K, ldb, B_MN, KBOX_ROWS)) return 1;
  const int64_t tiles_m = ceil_div(M, TILE_M), tiles_n = ceil_div(N, UMMA_N);
  const int64_t tiles = tiles_m * (CL == 4 ? ceil_div(tiles_n, 2) : tiles_n);   // scheduling units
  const int groups = tc::max_groups(CL);
  const tc::TailPlan plan = tc::plan_tail(flags, tiles, tiles_m * tiles_n, groups, ceil_div(K, BK), 512 / BK);
  if (tc::clear_tile_flags(plan, tiles_m * tiles_n)) return 1;
  // rasterisation knob in scheduling units: a panel of g tile columns = g/2 units when CL = 4
  const int gm = (CL == 4 && g_group_m < 0) ? std::min(-1, g_group_m / 2) : g_group_m;
  return tc::launch_persistent<gemm_f16x3_kernel<A_MN, B_MN, CL>>(
      CL, NUM_THREADS, SMEM_BYTES, plan.t_full + (tiles - plan.t_full) * plan.tail_split, groups, CL == 4, 1, ma_h,
      ma_l, mb_h, mb_l, D, ldd, (int)M, (int)N, (int)K, bias, flags, plan.t_full, plan.tail_split, tc::g_tile_flags,
      act_out, mask_src, meta_a, meta_b, stat_out, gm);
}

template <int CL>
static int launch_layout(int layout, float* D, int64_t ldd, const void* a_h, const void* a_l, int64_t lda,
                         const void* b_h, const void* b_l, int64_t ldb, int64_t M, int64_t N, int64_t K,
                         const float* bias, int flags, float* act_out, const float* mask_src,
                         const Meta* ma, const Meta* mb, Meta* st) {
  switch (layout & 3) {
    case 0: return launch<false, false, CL>(D, ldd, a_h, a_l, lda, b_h, b_l, ldb, M, N, K, bias, flags, act_out, mask_src, ma, mb, st);
    case 1: return launch<true, false, CL>(D, ldd, a_h, a_l, lda, b_h, b_l, ldb, M, N, K, bias, flags, act_out, mask_src, ma, mb, st);
    case 2: return launch<false, true, CL>(D, ldd, a_h, a_l, lda, b_h, b_l, ldb, M, N, K, bias, flags, act_out, mask_src, ma, mb, st);
    default: return launch<true, true, CL>(D, ldd, a_h, a_l, lda, b_h, b_l, ldb, M, N, K, bias, flags, act_out, mask_src, ma, mb, st);
  }
}

}  // namespace f16
}  // namespace tnn

using namespace tnn;

extern "C" {

int tnn_set_gemm_f16_cluster(int cl) {
  if (cl != 2 && cl != 4) TNN_FAIL("tnn_set_gemm_f16_cluster: 2 (CTA pairs) or 4 (two pairs sharing A by TMA multicast)");
  f16::g_cluster = cl;
  return 0;
}

int tnn_f16_stats(const float* x, int64_t n, void* meta, int relu_mode) {
  TNN_REQUIRE_INIT();
  if (!meta) TNN_FAIL("tnn_f16_stats: meta is required");
  TNN_CUDA(cudaMemsetAsync(meta, 0, sizeof(f16::Meta), ctx().stream));
  if (n <= 0) return 0;
  const int vec = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  prof_begin(3);
  f16::stats_kernel<<<ew_grid(ceil_div(n, 16), 256), 256, 0, ctx().stream>>>(x, n, (f16::Meta*)meta, relu_mode, vec, 0);
  TNN_POST_LAUNCH();
  prof_end(3);
  return 0;
}

int tnn_f16_stats_cond(const float* x, int64_t n, void* meta, int relu_mode) {
  TNN_REQUIRE_INIT();
  if (!meta) TNN_FAIL("tnn_f16_stats_cond: meta is required");
  if (n <= 0) return 0;
  const int vec = (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  prof_begin(3);
  f16::stats_kernel<<<ew_grid(ceil_div(n, 16), 256, 4), 256, 0, ctx().stream>>>(x, n, (f16::Meta*)meta, relu_mode, vec, 1);
  TNN_POST_LAUNCH();
  prof_end(3);
  return 0;
}

int tnn_f16_meta_reset(void* meta) {
  TNN_REQUIRE_INIT();
  if (!meta) TNN_FAIL("tnn_f16_meta_reset: meta is required");
  TNN_CUDA(cudaMemsetAsync(meta, 0, sizeof(f16::Meta), ctx().stream));
  return 0;
}

int tnn_split_f16(const float* x, int64_t R, int64_t C, void* hf, void* l16, int64_t ld, void* meta,
                  int relu_mode) {
  TNN_REQUIRE_INIT();
  if (R <= 0 || C <= 0) return 0;
  if (!hf || !l16 || !meta) TNN_FAIL("tnn_split_f16: both planes and the meta record are required");
  if (ld % 8 != 0 || ld < C) TNN_FAIL("tnn_split_f16: ld must be >= C and a multiple of 8");
  const int vec_in = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  prof_begin(3);
  f16::split_f16_kernel<<<ew_grid(R * (ld / 8), 256), 256, 0, ctx().stream>>>(
      x, R, C, (__half*)hf, (__half*)l16, ld, (f16::Meta*)meta, relu_mode, vec_in);
  TNN_POST_LAUNCH();
  prof_end(3);
  return 0;
}

int tnn_gemm_f16x3(float* D, int64_t ldd, const void* a_hf, const void* a_l16, int64_t lda,
                   const void* a_meta, const void* b_hf, const void* b_l16, int64_t ldb,
                   const void* b_meta, int64_t M, int64_t N, int64_t K, const float* bias, int flags,
                   int layout, float* act_out, const float* mask_src, void* stat_meta) {
  bool empty;
  if (tc::gemm_entry_checks("tnn_gemm_f16x3", M, N, K, empty)) return 1;
  if (empty) return 0;
  if (!a_meta || !b_meta) TNN_FAIL("tnn_gemm_f16x3: operand meta records are required");
  if (mask_src && !act_out) TNN_FAIL("tnn_gemm_f16x3: the mask_src form needs act_out");
  if (act_out && (flags & 2)) TNN_FAIL("tnn_gemm_f16x3: act_out and the relu-in-place flag are exclusive");
  if (getenv("TNN_EXP_FLAGS")) flags |= atoi(getenv("TNN_EXP_FLAGS")) & (128 | 256);
  static bool env_read = false;
  if (!env_read) {
    const char* gm = getenv("TNN_F16_GROUP_M");
    if (gm && atoi(gm) != 0 && atoi(gm) >= -64 && atoi(gm) <= 64) f16::g_group_m = atoi(gm);
    const char* rv = getenv("TNN_F16_REVERSE");
    if (rv) f16::g_reverse = atoi(rv) != 0;
    const char* cl = getenv("TNN_F16_CLUSTER");
    if (cl && (atoi(cl) == 2 || atoi(cl) == 4)) f16::g_cluster = atoi(cl);
    env_read = true;
  }
  if (f16::g_reverse) flags |= 32;
  const f16::Meta* ma = (const f16::Meta*)a_meta;
  const f16::Meta* mb = (const f16::Meta*)b_meta;
  f16::Meta* st = (f16::Meta*)stat_meta;
  // two pairs per cluster only pay when there are at least two tile columns to share A over
  if (f16::g_cluster == 4 && N > f16::UMMA_N)
    return f16::launch_layout<4>(layout, D, ldd, a_hf, a_l16, lda, b_hf, b_l16, ldb, M, N, K, bias, flags, act_out, mask_src, ma, mb, st);
  return f16::launch_layout<2>(layout, D, ldd, a_hf, a_l16, lda, b_hf, b_l16, ldb, M, N, K, bias, flags, act_out, mask_src, ma, mb, st);
}

}  // extern "C"

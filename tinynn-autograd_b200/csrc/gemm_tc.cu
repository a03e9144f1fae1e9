// Tensor-core GEMM for ops.py:150-163 (dot_: A@B, grad@B.T, A.T@grad) in fp32-accurate 3xTF32:
//
//     x = hi + lo,  hi = tf32(x), lo = tf32(x - hi)
//     A*B ~= A_lo*B_hi + A_hi*B_lo + A_hi*B_hi        (fp32 accumulation in TMEM)
//
// Pipeline (sm_100a only):
//   tnn_split_tf32   one pass over an fp32 matrix -> hi/lo planes, optionally also transposed,
//                    so every product of the forward/backward pass becomes the one canonical
//                    form below (both operands K-major).
//   tnn_gemm_tf32x3  D[M,N] = A[M,K] * B[N,K]^T.  Persistent, warp-specialised:
//                      warp 0    TMA producer  (cp.async.bulk.tensor, SWIZZLE_128B, mbarrier tx)
//                      warp 1    MMA issuer    (tcgen05.mma.kind::tf32, 3 MMAs per K=8 step)
//                      warps 4-11 epilogue     (tcgen05.ld TMEM -> fp32 regs (+=) -> bias/relu/accumulate)
//                    The tensor core accumulates in fp32 with round-toward-zero, which biases a long
//                    K loop (measured: ~6e-5 relative at K = 4096).  So a TMEM accumulator only
//                    ever holds a short chain (CHUNK_KB K blocks = 128 k): the 8 epilogue warps
//                    drain each chunk with tcgen05.ld and add it, round-to-nearest, into fp32
//                    registers (128 per thread) that carry the tile.  The two TMEM accumulators
//                    (2 x 256 columns) alternate per chunk, so draining chunk c overlaps the MMAs
//                    of chunk c+1 and the store of tile i overlaps the first chunks of tile i+1.
//                    CG = 1: one CTA per SM, tile 128 x 256.
//                    CG = 2: CTA pair (cta_group::2), tile 256 x 256, each CTA stages its own
//                            128 rows of A and half of B -> half the L2->SMEM operand traffic
//                            per flop and room for a third pipeline stage.
// Algorithmic work: 2*M*N*K flop per call; the tensor pipe executes 3x that in TF32.
//
// MIX variant (tnn_gemm_tf32_bf16x2, the default): the two cross terms only need ~9 significant
// bits of each factor, so they run as BF16 MMAs (twice the TF32 rate) on bf16 planes:
//
//     A*B ~= bf16(A - A_hi)*bf16(B) + bf16(A)*bf16(B - B_hi) + A_hi*B_hi
//
// Per 32-wide K block that is 2+2 BF16 MMAs (K = 16) and 4 TF32 MMAs (K = 8): 8 tensor-pipe
// slots instead of 12, with the same 8 bytes of planes per element (hi fp32 + two bf16 planes).
// The split error grows from 7e-8 to 7e-7 of max|result| (numpy emulation in DESIGN.md) -- still
// below the fp32 accumulation error of a K = 4096 product.  The kernel is power-bound (SM clocks
// settle near 1.7 GHz under the 1 kW cap), so a third fewer MMA cycles is a fifth less time.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include <cstdlib>

#include "common.cuh"
#include "tc_gemm.cuh"

namespace tnn {
namespace tc {

constexpr int BK = 32;                    // fp32 elements per K block = 128 bytes = swizzle row
constexpr int ROWS_A = 128;               // A rows staged per CTA
constexpr int UMMA_N = 256;               // accumulator columns per tile
constexpr int UMMA_K = 8;                 // tf32
constexpr int PLANE_ROW_BYTES = BK * 4;   // 128
constexpr int NUM_THREADS = 384;         // warpgroup 0: TMA warp, MMA warp, 2 idle; warpgroups 1-2: epilogue
#ifndef TNN_CHUNK_KB
#define TNN_CHUNK_KB 8
#endif
constexpr int CHUNK_KB = TNN_CHUNK_KB;    // K blocks accumulated inside the tensor core per chunk
constexpr uint32_t TMEM_COLS = 512;

template <int CG>
struct Cfg {
  static constexpr int ROWS_B = UMMA_N / CG;                      // B rows staged per CTA
  static constexpr int A_BYTES = ROWS_A * PLANE_ROW_BYTES;        // one plane
  static constexpr int B_BYTES = ROWS_B * PLANE_ROW_BYTES;
  static constexpr int STAGES = CG == 1 ? 2 : 3;
  static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // hi+lo of both operands
  static constexpr int A_PLANES_BYTES = 2 * A_BYTES;
  static constexpr int L16_OFF_A = A_BYTES / 2, L16_OFF_B = B_BYTES / 2;
  static constexpr int TILE_M = ROWS_A * CG;
  static constexpr int EPI_PATCH_BYTES = 8 * 4096;                // one 32x32 fp32 patch per epilogue warp
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/ + EPI_PATCH_BYTES;
};

// Operand tiles in shared memory (one plane of one 32-wide K block, rows = 128 M/N rows):
//   K-major  : one TMA box {32 k, rows}: row r at r*128 B, k contiguous, 128-byte swizzle.
//              Descriptor: 8-row groups 1024 B apart (SBO); a K=8 step advances 32 B in the row.
//   MN-major : rows/32 TMA boxes {32 mn, 32 k} of 4096 B each: inside a box k-row j at j*128 B with
//              32 consecutive M/N elements.  32-bit MN-major operands only exist in the
//              "128-byte swizzle with 32-byte atoms" layout (TMA SWIZZLE_128B_ATOM_32B, UMMA layout
//              type SWIZZLE_128B_BASE32B): the swizzle pattern spans 4 k-rows (512 B).  Descriptor:
//              4-k groups 512 B apart (SBO), 32-element M/N chunks 4096 B apart (LBO); a K=8 step
//              advances 1024 B.
template <bool MN>
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);                  // start address
  d |= (uint64_t)(MN ? (4096 >> 4) : 1) << 16;               // leading byte offset
  d |= (uint64_t)((MN ? 512 : 1024) >> 4) << 32;             // stride byte offset
  d |= (uint64_t)1 << 46;                                    // descriptor version (Blackwell)
  d |= (uint64_t)(MN ? 1 : 2) << 61;                         // SWIZZLE_128B_BASE32B : SWIZZLE_128B
  return d;
}
// bf16 planes (MIX variant), one 32-wide K block:
//   K-major  : one TMA box {32 k, rows} of 64-byte rows, 64-byte swizzle (period 8 rows = 512 B).
//              Descriptor: SWIZZLE_64B, 8-row groups 512 B apart (SBO); a K=16 step advances 32 B.
//   MN-major : rows/64 TMA boxes {64 mn, 32 k} of 4096 B (k-row j at j*128 B holding 64 consecutive
//              M/N elements), plain 128-byte swizzle.  Descriptor: SWIZZLE_128B, 8-k groups 1024 B
//              apart (SBO), 64-element M/N chunks 4096 B apart (LBO); a K=16 step advances 2048 B.
template <bool MN>
__device__ __forceinline__ uint64_t make_smem_desc16(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)(MN ? (4096 >> 4) : 1) << 16;
  d |= (uint64_t)((MN ? 1024 : 512) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(MN ? 2 : 4) << 61;                         // SWIZZLE_128B : SWIZZLE_64B
  return d;
}
constexpr int MN_BOX_BYTES = 32 * PLANE_ROW_BYTES;           // one {32 mn, 32 k} box
// instruction descriptor: D=F32, A=B=TF32, operand majors, N, M
__host__ __device__ constexpr uint32_t make_idesc(int m, int n, bool a_mn, bool b_mn) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// D=F32, A=B=BF16
__host__ __device__ constexpr uint32_t make_idesc16(int m, int n, bool a_mn, bool b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---- the GEMM kernel ---------------------------------------------------------------------------
// MIX = false: planes are (hi, lo) tf32, map_*_lo = the lo plane, map_*_l16 unused.
// MIX = true : planes are (hi tf32, h16 = bf16(x), l16 = bf16(x - hi)); map_*_lo = h16.
template <int CG, bool A_MN, bool B_MN, bool MIX>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap map_a_hi,
                   const __grid_constant__ CUtensorMap map_a_lo,
                   const __grid_constant__ CUtensorMap map_a_l16,
                   const __grid_constant__ CUtensorMap map_b_hi,
                   const __grid_constant__ CUtensorMap map_b_lo,
                   const __grid_constant__ CUtensorMap map_b_l16,
                   float* __restrict__ D, int64_t ldd, int M, int N, int K,
                   const float* __restrict__ bias, int flags, int t_full, int tail_split,
                   unsigned int* __restrict__ tile_flags, int group_m,
                   float* __restrict__ act_out, float* __restrict__ act_hi,
                   float* __restrict__ act_lo, __nv_bfloat16* __restrict__ act_l16, int64_t ld_act,
                   const float* __restrict__ mask_src, const int* __restrict__ cond_a,
                   const int* __restrict__ cond_b) {
  // conditional form (fallback behind the f16 product, gemm_f16.cu): nothing to do when both
  // operands were inside the f16 guard (word 3 of an operand's meta record = its `safe` flag)
  if (cond_a != nullptr && cond_a[3] && cond_b[3]) return;
  using C = Cfg<CG>;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B tiles need 1024-byte alignment
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const Barriers<C::STAGES> bar{smem_base + C::STAGES * C::STAGE_BYTES};

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t cta_rank = CG == 1 ? 0u : cluster_ctarank();
  const bool leader = cta_rank == 0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a_hi);
    tma_prefetch_desc(&map_a_lo);
    tma_prefetch_desc(&map_b_hi);
    tma_prefetch_desc(&map_b_lo);
    if constexpr (MIX) {
      tma_prefetch_desc(&map_a_l16);
      tma_prefetch_desc(&map_b_l16);
    }
    bar.init(1, 8 * CG);   // tmem_empty: one arrival per epilogue warp of every CTA in the group
  }
  const uint32_t tmem_base = tmem_setup<CG>(bar, smem_gen + C::STAGES * C::STAGE_BYTES, warp, TMEM_COLS);

  const int tiles_m = (M + C::TILE_M - 1) / C::TILE_M;
  const int tiles_n = (N + UMMA_N - 1) / UMMA_N;
  const int num_tiles = tiles_m * tiles_n;
  const int num_kb = (K + BK - 1) / BK;
  const int group = blockIdx.x / CG;            // CTA (pair) index
  const int num_groups = gridDim.x / CG;
  const WorkUnits work(t_full, tail_split, num_tiles, num_kb);

  // Register budget: the compiler is held to 168 registers per thread by the 384-thread block; the
  // epilogue warps carry 128 fp32 tile sums each, so warpgroup 0 (TMA + MMA issue, a handful of
  // registers) hands its share to warpgroups 1-2: 128*40 + 256*216 = 60,416 <= 65,536.
  // (setmaxnreg sits inside each role branch so the compiler scopes the budget to that role.)
  if (warp == 0) {
    // ================= TMA producer =================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = group; u < work.num_units; u += num_groups) {
        int t, sp, kb_begin, kb_end;
        work.decode(u, t, sp, kb_begin, kb_end);
        int tm, tn;
        tile_coords(t, tiles_m, tiles_n, group_m, tm, tn);
        const int row_a = tm * C::TILE_M + (int)cta_rank * ROWS_A;
        const int row_b = tn * UMMA_N + (int)cta_rank * C::ROWS_B;
        for (int kb = kb_begin; kb < kb_end; ++kb) {
          mbar_wait(bar.empty(stage), phase ^ 1u);
          const uint32_t sa_hi = smem_base + stage * C::STAGE_BYTES;
          const uint32_t sa_lo = sa_hi + C::A_BYTES;
          const uint32_t sb_hi = sa_hi + C::A_PLANES_BYTES;
          const uint32_t sb_lo = sb_hi + C::B_BYTES;
          // (flags & 64: timing experiment only -- the bf16(x) planes are not fetched, results are wrong)
          // flags & 64 / 128 / 256 / 512 are TIMING EXPERIMENTS (TNN_EXP_FLAGS, results are wrong): the
          // bf16(x) planes are not fetched / nothing is fetched / no MMA is issued / no chunk is drained
          const bool exp_skip_h16 = MIX && (flags & 64);
          const bool exp_skip_hi = MIX && (flags & 1024);   // timing experiment: 16-bit planes only
          const uint32_t tx_bytes = (uint32_t)(C::STAGE_BYTES - (exp_skip_h16 ? (C::A_BYTES + C::B_BYTES) / 2 : 0)
                                               - (exp_skip_hi ? (C::A_BYTES + C::B_BYTES) : 0)) * CG;
          if (leader) mbar_expect_tx(bar.full(stage), tx_bytes);
          const int k0 = kb * BK;
          if (flags & 128) {
            // timing experiment: no operand fetch at all (the MMAs run on whatever the stage holds);
            // the transaction count armed above is satisfied by hand
            if (leader)
              asm volatile("mbarrier.complete_tx.shared::cta.b64 [%0], %1;" ::"r"(bar.full(stage)), "r"(tx_bytes) : "memory");
          } else
          if constexpr (!MIX) {
            if constexpr (A_MN) {
#pragma unroll
              for (int j = 0; j < ROWS_A / 32; ++j) {
                tma_load_2d<CG>(sa_hi + j * MN_BOX_BYTES, &map_a_hi, bar.full(stage), row_a + 32 * j, k0);
                tma_load_2d<CG>(sa_lo + j * MN_BOX_BYTES, &map_a_lo, bar.full(stage), row_a + 32 * j, k0);
              }
            } else {
              tma_load_2d<CG>(sa_hi, &map_a_hi, bar.full(stage), k0, row_a);
              tma_load_2d<CG>(sa_lo, &map_a_lo, bar.full(stage), k0, row_a);
            }
            if constexpr (B_MN) {
#pragma unroll
              for (int j = 0; j < C::ROWS_B / 32; ++j) {
                tma_load_2d<CG>(sb_hi + j * MN_BOX_BYTES, &map_b_hi, bar.full(stage), row_b + 32 * j, k0);
                tma_load_2d<CG>(sb_lo + j * MN_BOX_BYTES, &map_b_lo, bar.full(stage), row_b + 32 * j, k0);
              }
            } else {
              tma_load_2d<CG>(sb_hi, &map_b_hi, bar.full(stage), k0, row_b);
              tma_load_2d<CG>(sb_lo, &map_b_lo, bar.full(stage), k0, row_b);
            }
          } else {
            // the second 32-bit plane's space holds the two bf16 planes
            const uint32_t sa_h16 = sa_lo, sa_l16 = sa_lo + C::L16_OFF_A;
            const uint32_t sb_h16 = sb_lo, sb_l16 = sb_lo + C::L16_OFF_B;
            if constexpr (A_MN) {
#pragma unroll
              for (int j = 0; j < ROWS_A / 32; ++j)
                if (!exp_skip_hi) tma_load_2d<CG>(sa_hi + j * MN_BOX_BYTES, &map_a_hi, bar.full(stage), row_a + 32 * j, k0);
#pragma unroll
              for (int j = 0; j < ROWS_A / 64; ++j) {
                if (!exp_skip_h16) tma_load_2d<CG>(sa_h16 + j * MN_BOX_BYTES, &map_a_lo, bar.full(stage), row_a + 64 * j, k0);
                tma_load_2d<CG>(sa_l16 + j * MN_BOX_BYTES, &map_a_l16, bar.full(stage), row_a + 64 * j, k0);
              }
            } else {
              if (!exp_skip_hi) tma_load_2d<CG>(sa_hi, &map_a_hi, bar.full(stage), k0, row_a);
              if (!exp_skip_h16) tma_load_2d<CG>(sa_h16, &map_a_lo, bar.full(stage), k0, row_a);
              tma_load_2d<CG>(sa_l16, &map_a_l16, bar.full(stage), k0, row_a);
            }
            if constexpr (B_MN) {
#pragma unroll
              for (int j = 0; j < C::ROWS_B / 32; ++j)
                if (!exp_skip_hi) tma_load_2d<CG>(sb_hi + j * MN_BOX_BYTES, &map_b_hi, bar.full(stage), row_b + 32 * j, k0);
#pragma unroll
              for (int j = 0; j < C::ROWS_B / 64; ++j) {
                if (!exp_skip_h16) tma_load_2d<CG>(sb_h16 + j * MN_BOX_BYTES, &map_b_lo, bar.full(stage), row_b + 64 * j, k0);
                tma_load_2d<CG>(sb_l16 + j * MN_BOX_BYTES, &map_b_l16, bar.full(stage), row_b + 64 * j, k0);
              }
            } else {
              if (!exp_skip_hi) tma_load_2d<CG>(sb_hi, &map_b_hi, bar.full(stage), k0, row_b);
              if (!exp_skip_h16) tma_load_2d<CG>(sb_h16, &map_b_lo, bar.full(stage), k0, row_b);
              tma_load_2d<CG>(sb_l16, &map_b_l16, bar.full(stage), k0, row_b);
            }
          }
          if (++stage == C::STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (leader CTA only) =================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (leader && lane == 0) {
      constexpr uint32_t idesc = make_idesc(C::TILE_M, UMMA_N, A_MN, B_MN);
      constexpr uint32_t idesc16 = make_idesc16(C::TILE_M, UMMA_N, A_MN, B_MN);
      (void)idesc16;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int u = group; u < work.num_units; u += num_groups) {
        int t, sp, kb_begin, kb_end;
        work.decode(u, t, sp, kb_begin, kb_end);
        for (int kb0 = kb_begin; kb0 < kb_end; kb0 += CHUNK_KB) {
          mbar_wait(bar.tempty(acc), acc_phase ^ 1u);   // epilogue has drained this accumulator
          tc_fence_after();
          const uint32_t tmem_d = tmem_base + (uint32_t)(acc * UMMA_N);
          const int kb1 = min(kb0 + CHUNK_KB, kb_end);
          for (int kb = kb0; kb < kb1; ++kb) {
            mbar_wait(bar.full(stage), phase);
            tc_fence_after();
            const uint32_t sa_hi = smem_base + stage * C::STAGE_BYTES;
            const uint32_t sa_lo = sa_hi + C::A_BYTES;
            const uint32_t sb_hi = sa_hi + C::A_PLANES_BYTES;
            const uint32_t sb_lo = sb_hi + C::B_BYTES;
            if (flags & 256) {
              // timing experiment: operands are fetched but no MMA is issued
            } else
            if constexpr (!MIX) {
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                // a K=8 step: 32 B along the row (K-major) or one 8-row group of 1024 B (MN-major)
                const uint32_t koff_a = (uint32_t)(k * (A_MN ? 1024 : UMMA_K * 4));
                const uint32_t koff_b = (uint32_t)(k * (B_MN ? 1024 : UMMA_K * 4));
                const uint64_t da_hi = make_smem_desc<A_MN>(sa_hi + koff_a);
                const uint64_t da_lo = make_smem_desc<A_MN>(sa_lo + koff_a);
                const uint64_t db_hi = make_smem_desc<B_MN>(sb_hi + koff_b);
                const uint64_t db_lo = make_smem_desc<B_MN>(sb_lo + koff_b);
                // small terms first; the first MMA of a chunk overwrites the accumulator
                umma_tf32<CG>(tmem_d, da_lo, db_hi, idesc, (kb != kb0 || k != 0) ? 1u : 0u);
                umma_tf32<CG>(tmem_d, da_hi, db_lo, idesc, 1u);
                umma_tf32<CG>(tmem_d, da_hi, db_hi, idesc, 1u);
              }
            } else {
              const uint32_t sa_h16 = sa_lo, sa_l16 = sa_lo + C::L16_OFF_A;
              const uint32_t sb_h16 = sb_lo, sb_l16 = sb_lo + C::L16_OFF_B;
              // cross terms on the bf16 planes (small terms first): two K=16 steps
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
                const uint32_t koff_a = (uint32_t)(k * (A_MN ? 2048 : 32));
                const uint32_t koff_b = (uint32_t)(k * (B_MN ? 2048 : 32));
                const uint64_t da_h = make_smem_desc16<A_MN>(sa_h16 + koff_a);
                const uint64_t da_l = make_smem_desc16<A_MN>(sa_l16 + koff_a);
                const uint64_t db_h = make_smem_desc16<B_MN>(sb_h16 + koff_b);
                const uint64_t db_l = make_smem_desc16<B_MN>(sb_l16 + koff_b);
                umma_bf16<CG>(tmem_d, da_l, db_h, idesc16, (kb != kb0 || k != 0) ? 1u : 0u);
                umma_bf16<CG>(tmem_d, da_h, db_l, idesc16, 1u);
                if (flags & 1024) umma_bf16<CG>(tmem_d, da_h, db_h, idesc16, 1u);
              }
              // main term on the tf32 planes: four K=8 steps
              if (!(flags & 1024))
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k) {
                const uint32_t koff_a = (uint32_t)(k * (A_MN ? 1024 : UMMA_K * 4));
                const uint32_t koff_b = (uint32_t)(k * (B_MN ? 1024 : UMMA_K * 4));
                umma_tf32<CG>(tmem_d, make_smem_desc<A_MN>(sa_hi + koff_a),
                              make_smem_desc<B_MN>(sb_hi + koff_b), idesc, 1u);
              }
            }
            umma_commit<CG>(bar.empty(stage));          // frees the smem slot when the MMAs retire
            if (++stage == C::STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
          umma_commit<CG>(bar.tfull(acc));              // chunk complete -> epilogue may drain it
          if (++acc == 2) {
            acc = 0;
            acc_phase ^= 1u;
          }
        }
      }
    }
  } else if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");   // idle warps of warpgroup 0
  } else {
    // ================= epilogue: TMEM chunks -> fp32 registers (RN adds) -> global =================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
    const int quad = warp & 3;                       // TMEM lanes [32*quad, 32*quad+32)
    const int half = (warp - 4) >> 2;                // accumulator columns [128*half, 128*half+128)
    int acc = 0;
    uint32_t acc_phase = 0;
    const bool relu = flags & 2;
    for (int u = group; u < work.num_units; u += num_groups) {
      int t, sp, kb_begin, kb_end;
      work.decode(u, t, sp, kb_begin, kb_end);
      const bool accumulate = (flags & 1) || sp > 0;
      // the unit that holds the complete sum also emits the fused activation outputs
      // act_out may be NULL with the planes present: the fp32 ReLU output is then never written
      // (the next products read its planes, the backward mask reads the pre-activation)
      const bool emit_act = (act_out != nullptr || act_hi != nullptr) && (u < t_full || sp + 1 == tail_split);
      const float* bias_u = sp == 0 ? bias : nullptr;
      int tm, tn;
      tile_coords(t, tiles_m, tiles_n, group_m, tm, tn);
      const int row = tm * C::TILE_M + (int)cta_rank * ROWS_A + quad * 32 + lane;
      const int col0 = tn * UMMA_N + half * 128;
      float sum[128];
#pragma unroll
      for (int j = 0; j < 128; ++j) sum[j] = 0.f;
      for (int kb0 = kb_begin; kb0 < kb_end; kb0 += CHUNK_KB) {
        mbar_wait(bar.tfull(acc), acc_phase);
        tc_fence_after();
        const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) +
                               (uint32_t)(acc * UMMA_N + half * 128);
        if (!(flags & 512)) {     // (512: timing experiment, accumulator chunks are not drained)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            uint32_t r[32];
            tmem_ld_32x32b_x32(taddr + (uint32_t)(c * 32), r);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) sum[c * 32 + j] += __uint_as_float(r[j]);
          }
        }
        tmem_hand_back<CG != 1>(bar.tempty(acc), 0, lane);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1u;
        }
      }
      if (sp > 0) {
        // wait until every epilogue warp of split sp-1 has stored this tile
        if (lane == 0) {
          const unsigned int need = (unsigned int)(sp * 8 * CG);
          unsigned int seen;
          long long t0 = clock64();
          do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(tile_flags + t) : "memory");
            if (clock64() - t0 > 8000000000LL) {
              printf("tnn gemm_tc: split-K ordering wait timed out (tile %d split %d)\n", t, sp);
              __trap();
            }
          } while (seen < need);
        }
        __syncwarp();
        __threadfence();
      }
      // ---- store the tile.  A thread owns one row x 128 columns, so a direct store would touch 32
      // rows with 16 bytes each per instruction (half-used sectors).  Each warp instead bounces its
      // 32 x 32 blocks through a private 4 KB swizzled shared-memory patch and comes back with 8
      // lanes per row: every global access is 4 full 128-byte lines.  While the epilogue warps are
      // here the MMA issuer can only run two chunks ahead, so this phase has to be short.
      {
        const int row_base = tm * C::TILE_M + (int)cta_rank * ROWS_A + quad * 32;
        float4* patch = reinterpret_cast<float4*>(smem_gen + C::STAGES * C::STAGE_BYTES + 256) +
                        (warp - 4) * 256;                       // 32 rows x 8 float4
        const bool rows_aligned = (ldd % 4 == 0) && ((reinterpret_cast<uintptr_t>(D) & 15) == 0);
        const bool act_aligned = !emit_act || (((reinterpret_cast<uintptr_t>(act_out) |
                                                  reinterpret_cast<uintptr_t>(mask_src)) & 15) == 0);
        if (!accumulate && !emit_act && rows_aligned) {
          // plain tile (bias / in-place ReLU only): ONE rolled copy of the store loop.  The general
          // form below is fully unrolled -- thousands of SASS instructions that a warp walks once
          // per tile, instruction-fetch-bound (r02, gemm_f16.cu) -- and is kept for the launches
          // that read back (accumulate, mask) or emit operand planes.
          const int rr = lane >> 3, c4l = lane & 7;
#pragma unroll 1
          for (int cb = 0; cb < 4; ++cb) {
            const int colb = col0 + cb * 32;
            if (colb >= N) break;                               // warp-uniform
            patch_write<false>(cb, sum, patch, lane, 1.f, 1.f, bias_u, colb, N);
            __syncwarp();
            const int gcol = colb + c4l * 4;
#pragma unroll 1
            for (int i = 0; i < 8; ++i) {
              const int r = 4 * i + rr, grow = row_base + r;
              if (grow >= M) break;
              float4 v = patch[r * 8 + (c4l ^ (r & 7))];
              if (relu) {
                v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f);
                v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
              }
              float* dp = D + (int64_t)grow * ldd + gcol;
              if (gcol + 3 < N) {
                *reinterpret_cast<float4*>(dp) = v;
              } else {
                if (gcol < N) dp[0] = v.x;
                if (gcol + 1 < N) dp[1] = v.y;
                if (gcol + 2 < N) dp[2] = v.z;
              }
            }
            __syncwarp();
          }
        } else
#pragma unroll
        for (int cb = 0; cb < 4; ++cb) {
          const int colb = col0 + cb * 32;                      // first column of this 32-wide block
          if (colb >= N) break;                                 // warp-uniform
          patch_write<false>(cb, sum, patch, lane, 1.f, 1.f, bias_u, colb, N);   // (cb is unrolled)
          __syncwarp();
          // whatever the store has to READ first (the previous D for accumulate, the pre-activation
          // for the ReLU mask) is fetched for all 8 row groups up front: 8-16 independent 128-bit
          // loads in flight instead of one exposed round trip per row group
          // (one register array serves either purpose; a launch that wants both -- never issued by
          // the engine -- reads the mask inside the loop)
          const bool fast_rows = rows_aligned && act_aligned;
          const bool want_mask = emit_act && mask_src != nullptr;
          const float* pre_src = accumulate ? D : (want_mask ? mask_src : nullptr);
          float4 pre[8];
          if (fast_rows && pre_src != nullptr) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int grow = row_base + 4 * i + (lane >> 3), gcol = colb + (lane & 7) * 4;
              if (grow < M && gcol + 3 < N)
                pre[i] = *reinterpret_cast<const float4*>(pre_src + (int64_t)grow * ldd + gcol);
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int r = 4 * i + (lane >> 3), c4 = lane & 7;
            float4 v = patch[r * 8 + (c4 ^ (r & 7))];
            const int grow = row_base + r, gcol = colb + c4 * 4;
            if (grow < M && gcol < N) {
              float* dp = D + (int64_t)grow * ldd + gcol;
              if (gcol + 3 < N && fast_rows) {
                if (accumulate) {
                  const float4 o = pre[i];
                  v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w;
                }
                if (relu) {
                  v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f);
                  v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f);
                }
                *reinterpret_cast<float4*>(dp) = v;
                if (emit_act) {
                  // ReLU(D) (NaN-propagating like np.clip) and, optionally, its tf32 planes: the
                  // next product consumes the activation without a separate relu / split pass
                  float4 a;
                  if (mask_src) {
                    // backward form: act = D * (pre-activation >= 0), the ReLU gradient mask of
                    // ops.py:336-343 (grad * mask, so a masked NaN/inf stays NaN like numpy's)
                    const float4 z = accumulate
                        ? *reinterpret_cast<const float4*>(mask_src + (int64_t)grow * ldd + gcol)
                        : pre[i];
                    a = make_float4(z.x >= 0.f ? v.x : v.x * 0.f, z.y >= 0.f ? v.y : v.y * 0.f,
                                    z.z >= 0.f ? v.z : v.z * 0.f, z.w >= 0.f ? v.w : v.w * 0.f);
                  } else {
                    a = make_float4(v.x < 0.f ? 0.f : v.x, v.y < 0.f ? 0.f : v.y,
                                    v.z < 0.f ? 0.f : v.z, v.w < 0.f ? 0.f : v.w);
                  }
                  if (act_out) *reinterpret_cast<float4*>(act_out + (int64_t)grow * ldd + gcol) = a;
                  if (act_hi) {
                    const float4 h = make_float4(to_tf32(a.x), to_tf32(a.y), to_tf32(a.z), to_tf32(a.w));
                    *reinterpret_cast<float4*>(act_hi + (int64_t)grow * ld_act + gcol) = h;
                    if constexpr (!MIX) {
                      const float4 l = make_float4(to_tf32(a.x - h.x), to_tf32(a.y - h.y),
                                                   to_tf32(a.z - h.z), to_tf32(a.w - h.w));
                      *reinterpret_cast<float4*>(act_lo + (int64_t)grow * ld_act + gcol) = l;
                    } else {
                      __nv_bfloat16* h16p = reinterpret_cast<__nv_bfloat16*>(act_lo);
                      union { __nv_bfloat162 b[2]; uint2 u; } ph, pl;
                      ph.b[0] = __floats2bfloat162_rn(a.x, a.y);
                      ph.b[1] = __floats2bfloat162_rn(a.z, a.w);
                      pl.b[0] = __floats2bfloat162_rn(a.x - h.x, a.y - h.y);
                      pl.b[1] = __floats2bfloat162_rn(a.z - h.z, a.w - h.w);
                      *reinterpret_cast<uint2*>(h16p + (int64_t)grow * ld_act + gcol) = ph.u;
                      *reinterpret_cast<uint2*>(act_l16 + (int64_t)grow * ld_act + gcol) = pl.u;
                    }
                  }
                }
              } else {
                const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  if (gcol + k < N) {
                    float x = e[k];
                    if (accumulate) x += dp[k];
                    if (relu) x = fmaxf(x, 0.f);
                    dp[k] = x;
                    if (emit_act) {
                      float a;
                      if (mask_src) a = mask_src[(int64_t)grow * ldd + gcol + k] >= 0.f ? x : x * 0.f;
                      else a = x < 0.f ? 0.f : x;
                      if (act_out) act_out[(int64_t)grow * ldd + gcol + k] = a;
                      if (act_hi) {
                        const float h = to_tf32(a);
                        act_hi[(int64_t)grow * ld_act + gcol + k] = h;
                        if constexpr (!MIX) {
                          act_lo[(int64_t)grow * ld_act + gcol + k] = to_tf32(a - h);
                        } else {
                          reinterpret_cast<__nv_bfloat16*>(act_lo)[(int64_t)grow * ld_act + gcol + k] =
                              __float2bfloat16_rn(a);
                          act_l16[(int64_t)grow * ld_act + gcol + k] = __float2bfloat16_rn(a - h);
                        }
                      }
                    }
                  }
                }
              }
            }
          }
          __syncwarp();
        }
      }
      if (u >= t_full && sp + 1 < tail_split) splitk_publish(tile_flags, t, lane);
    }
  }

  tmem_teardown<CG>(warp, tmem_base, TMEM_COLS);
}

// ---- fp32 -> tf32 hi/lo split (+ optional transposed copy) ----------------------------------------

// 64 x 64 tile per CTA, 256 threads; plain planes are written with 128-bit stores straight from
// registers, the transposed planes go through a padded shared-memory tile so both global sides
// stay coalesced.
__global__ void __launch_bounds__(256)
split_tf32_kernel(const float* __restrict__ x, int64_t R, int64_t C, float* __restrict__ hi,
                  float* __restrict__ lo, int64_t ldp, float* __restrict__ hiT,
                  float* __restrict__ loT, int64_t ldt, int vec_in) {
  __shared__ float tile[64][65];
  const int64_t r0 = (int64_t)blockIdx.y * 64, c0 = (int64_t)blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;  // 16 x 16, each thread 4 cols x 4 rows
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int lr = ty + 16 * i;
    const int64_t r = r0 + lr, c = c0 + tx * 4;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < R) {
      if (vec_in && c + 3 < C) {
        const float4 t = *reinterpret_cast<const float4*>(x + r * C + c);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (c + k < C) v[k] = x[r * C + c + k];
      }
      if (hi) {
        float h[4], l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          h[k] = to_tf32(v[k]);
          l[k] = to_tf32(v[k] - h[k]);
        }
        // ldp is a multiple of 4 and c is a multiple of 4: 16-byte aligned; columns in
        // [C, ldp) receive zeros (TMA never reads them, the tensor map ends at C)
        if (c < ldp) {
          *reinterpret_cast<float4*>(hi + r * ldp + c) = make_float4(h[0], h[1], h[2], h[3]);
          *reinterpret_cast<float4*>(lo + r * ldp + c) = make_float4(l[0], l[1], l[2], l[3]);
        }
      }
    }
    if (hiT) {
#pragma unroll
      for (int k = 0; k < 4; ++k) tile[lr][tx * 4 + k] = v[k];
    }
  }
  if (!hiT) return;
  __syncthreads();
  // transposed: output row = source column; each thread writes 4 consecutive source rows
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int lc = ty + 16 * i;            // source column inside the tile
    const int64_t c = c0 + lc, r = r0 + tx * 4;
    if (c < C && r < ldt) {
      float h[4], l[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float v = tile[tx * 4 + k][lc];   // zero beyond R
        h[k] = to_tf32(v);
        l[k] = to_tf32(v - h[k]);
      }
      *reinterpret_cast<float4*>(hiT + c * ldt + r) = make_float4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<float4*>(loT + c * ldt + r) = make_float4(l[0], l[1], l[2], l[3]);
    }
  }
}

// fp32 [R, C] -> hi = tf32(x) (fp32 plane), h16 = bf16(x), l16 = bf16(x - hi), all with pitch ld
// (a multiple of 8 >= C; the pad columns receive zeros).  One thread per 8 consecutive columns:
// two 128-bit loads, two 128-bit hi stores, one 128-bit store per bf16 plane.  12 B/element.
__device__ __forceinline__ void split_mix_body(const float* __restrict__ x, int64_t R, int64_t C,
                                               float* __restrict__ hi, __nv_bfloat16* __restrict__ h16,
                                               __nv_bfloat16* __restrict__ l16, int64_t ld, int vec_in,
                                               int relu_mode) {
  const int64_t gpr = ld / 8;   // 8-column groups per row
  const int64_t total = R * gpr;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
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
    if (relu_mode) {
#pragma unroll
      for (int k = 0; k < 8; ++k) v[k] = v[k] < 0.f ? 0.f : v[k];
    }
    float h[8];
    union { __nv_bfloat162 b[4]; uint4 u; } ph, pl;
#pragma unroll
    for (int k = 0; k < 8; ++k) h[k] = to_tf32(v[k]);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      ph.b[k] = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]);
      pl.b[k] = __floats2bfloat162_rn(v[2 * k] - h[2 * k], v[2 * k + 1] - h[2 * k + 1]);
    }
    float* hp = hi + r * ld + c;
    *reinterpret_cast<float4*>(hp) = make_float4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<float4*>(hp + 4) = make_float4(h[4], h[5], h[6], h[7]);
    *reinterpret_cast<uint4*>(h16 + r * ld + c) = ph.u;
    *reinterpret_cast<uint4*>(l16 + r * ld + c) = pl.u;
  }
}

__global__ void __launch_bounds__(256)
split_mix_kernel(const float* __restrict__ x, int64_t R, int64_t C, float* __restrict__ hi,
                 __nv_bfloat16* __restrict__ h16, __nv_bfloat16* __restrict__ l16, int64_t ld,
                 int vec_in) {
  split_mix_body(x, R, C, hi, h16, l16, ld, vec_in, 0);
}

// Conditional form, both operands of a product in one launch (blockIdx.y picks the operand): the
// fallback behind an f16 product (gemm_f16.cu).  Returns at once when both operands were inside
// the f16 guard (word 3 of an operand's meta record = its `safe` flag).  When it does run, the
// mixed-split product that follows leaves no statistics of its result, so word 1 of the result's
// record ("statistics missing") is set and tnn_f16_stats_cond recomputes them for the next split.
struct SplitArgs {
  const float* x; int64_t R, C; float* hi; __nv_bfloat16* h16; __nv_bfloat16* l16; int64_t ld;
  int vec_in, relu_mode;
};
__global__ void __launch_bounds__(256)
split_mix_cond2_kernel(SplitArgs a, SplitArgs b, const int* __restrict__ cond_a,
                       const int* __restrict__ cond_b, unsigned int* __restrict__ result_meta) {
  if (cond_a[3] && cond_b[3]) return;
  if (result_meta != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) result_meta[1] = 1u;
  const SplitArgs& s = blockIdx.y == 0 ? a : b;
  split_mix_body(s.x, s.R, s.C, s.hi, s.h16, s.l16, s.ld, s.vec_in, s.relu_mode);
}

// ---- host side ---------------------------------------------------------------------------------
// fp32 plane.  K-major [rows, K]: box {BK k, box_rows}, 128-byte swizzle.  MN-major [K, rows]: box
// {32 mn, BK k}, 128-byte swizzle with 32-byte atoms.
static int make_map(CUtensorMap* map, const float* ptr, int64_t rows, int64_t K, int64_t ld, int box_rows,
                    bool mn_major) {
  return tc::make_map(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, ptr, rows, K, ld, mn_major, mn_major ? 32 : BK,
                      mn_major ? BK : box_rows,
                      mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                      "tf32x3 GEMM: operand plane", "tf32x3 GEMM: operand pitch", "");
}

// bf16 plane.  K-major [rows, K]: box {BK k, box_rows}, 64-byte swizzle (a row of the box is 32 bf16 =
// 64 B).  MN-major [K, rows]: box {64 mn, BK k}, 128-byte swizzle.
static int make_map16(CUtensorMap* map, const void* ptr, int64_t rows, int64_t K, int64_t ld, int box_rows,
                      bool mn_major) {
  return tc::make_map(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, ptr, rows, K, ld, mn_major, mn_major ? 64 : BK,
                      mn_major ? BK : box_rows, mn_major ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                      "mixed GEMM: bf16 plane", "mixed GEMM: bf16 plane pitch", " (bf16)");
}

constexpr int DEFAULT_CG = 2;  // CTA pairs: measured 0.98 ms vs 1.10 ms per 8192x4096x4096 product
static int g_group_m = 1;                      // tile rasterisation group; measured on 8192x4096x4096:
                                               // 1 -> 0.95 ms, 4 -> 0.96-1.04, 8 -> 1.10, 16 -> 1.08
static int g_force_ksplit = 0;                 // 0 = auto (tail split), 1 = off, 2/4 = every tile (TNN_GEMM_KSPLIT)
static int g_force_cg = 0;  // 0 = default, 1 / 2 = forced (TNN_GEMM_CG or tnn_set_gemm_cta_group)
static int g_exp_flags = 0;  // timing experiments (TNN_EXP_*): OR-ed into the kernel's flags

struct ActOut {
  float* out = nullptr;   // relu(D), pitch ldd
  float* hi = nullptr;    // tf32 planes of relu(D), pitch ld
  float* lo = nullptr;    // MIX: the bf16(x) plane
  void* l16 = nullptr;    // MIX: the bf16(x - hi) plane
  int64_t ld = 0;
  const float* mask_src = nullptr;   // when set: out = D * (mask_src >= 0) instead of relu(D)
};

// planes: MIX = false -> (hi, lo) tf32 planes, l16 unused; MIX = true -> (hi tf32, h16, l16)
struct Planes {
  const float* hi;
  const void* lo;     // tf32 lo plane, or the bf16(x) plane
  const void* l16;    // bf16(x - hi) plane (MIX only)
  int64_t ld;
};

template <int CG, bool A_MN, bool B_MN, bool MIX>
static int launch_gemm(float* D, int64_t ldd, const Planes& a, const Planes& b, int64_t M, int64_t N,
                       int64_t K, const float* bias, int flags, const ActOut& act,
                       const int* cond_a = nullptr, const int* cond_b = nullptr) {
  using C = Cfg<CG>;
  CUtensorMap ma_hi, ma_lo, ma_l16, mb_hi, mb_lo, mb_l16;
  if (make_map(&ma_hi, a.hi, M, K, a.ld, ROWS_A, A_MN)) return 1;
  if (make_map(&mb_hi, b.hi, N, K, b.ld, C::ROWS_B, B_MN)) return 1;
  if constexpr (MIX) {
    if (make_map16(&ma_lo, a.lo, M, K, a.ld, ROWS_A, A_MN)) return 1;
    if (make_map16(&ma_l16, a.l16, M, K, a.ld, ROWS_A, A_MN)) return 1;
    if (make_map16(&mb_lo, b.lo, N, K, b.ld, C::ROWS_B, B_MN)) return 1;
    if (make_map16(&mb_l16, b.l16, N, K, b.ld, C::ROWS_B, B_MN)) return 1;
  } else {
    if (make_map(&ma_lo, (const float*)a.lo, M, K, a.ld, ROWS_A, A_MN)) return 1;
    if (make_map(&mb_lo, (const float*)b.lo, N, K, b.ld, C::ROWS_B, B_MN)) return 1;
    ma_l16 = ma_lo;
    mb_l16 = mb_lo;
  }
  const int64_t tiles = ceil_div(M, C::TILE_M) * ceil_div(N, UMMA_N);
  const int64_t num_kb = ceil_div(K, BK);
  const int groups = max_groups(CG);
  // Splitting EVERY tile instead of the tail lost time (1.20 ms vs 1.03 ms on the 4096x4096x8192 dW
  // product: the read-modify-write epilogue of the second range costs more than the idle tail), so a
  // forced whole-matrix split (TNN_GEMM_KSPLIT) is only taken when asked for.
  TailPlan plan{(int)tiles, 1};
  if (g_force_ksplit > 1) {
    if (!(flags & 2) && tiles <= MAX_FLAG_TILES && num_kb / g_force_ksplit >= 1) plan = {0, g_force_ksplit};
  } else if (g_force_ksplit != 1) {
    plan = plan_tail(flags, tiles, tiles, groups, num_kb, 16);
  }
  if (clear_tile_flags(plan, tiles)) return 1;
  // (a conditional launch is the fallback behind an f16 product: family 4, so that the per-launch
  // GEMM timing of family 1 only sees launches that do the product)
  return launch_persistent<gemm_tf32x3_kernel<CG, A_MN, B_MN, MIX>>(
      CG, NUM_THREADS, C::SMEM_BYTES, plan.t_full + (tiles - plan.t_full) * plan.tail_split, groups, false,
      cond_a ? 4 : 1, ma_hi, ma_lo, ma_l16, mb_hi, mb_lo, mb_l16, D, ldd, (int)M, (int)N, (int)K, bias,
      flags | g_exp_flags, plan.t_full, plan.tail_split, g_tile_flags, g_group_m, act.out, act.hi, act.lo,
      (__nv_bfloat16*)act.l16, act.ld, act.mask_src, cond_a, cond_b);
}

}  // namespace tc
}  // namespace tnn

using namespace tnn;

template <int CG, bool MIX>
static int launch_by_layout(int layout, float* D, int64_t ldd, const tnn::tc::Planes& a,
                            const tnn::tc::Planes& b, int64_t M, int64_t N, int64_t K, const float* bias,
                            int flags, const tnn::tc::ActOut& act, const int* cond_a, const int* cond_b) {
  switch (layout & 3) {
    case 0: return tnn::tc::launch_gemm<CG, false, false, MIX>(D, ldd, a, b, M, N, K, bias, flags, act, cond_a, cond_b);
    case 1: return tnn::tc::launch_gemm<CG, true, false, MIX>(D, ldd, a, b, M, N, K, bias, flags, act, cond_a, cond_b);
    case 2: return tnn::tc::launch_gemm<CG, false, true, MIX>(D, ldd, a, b, M, N, K, bias, flags, act, cond_a, cond_b);
    default: return tnn::tc::launch_gemm<CG, true, true, MIX>(D, ldd, a, b, M, N, K, bias, flags, act, cond_a, cond_b);
  }
}

static int gemm_common(const char* who, bool mix, float* D, int64_t ldd, const tnn::tc::Planes& a,
                       const tnn::tc::Planes& b, int64_t M, int64_t N, int64_t K, const float* bias,
                       int flags, int layout, const tnn::tc::ActOut& act_in,
                       const int* cond_a = nullptr, const int* cond_b = nullptr) {
  bool empty;
  if (tc::gemm_entry_checks(who, M, N, K, empty)) return 1;
  if (empty) return 0;
  static bool env_read = false;
  if (!env_read) {
    const char* e = getenv("TNN_GEMM_CG");
    if (e && !tc::g_force_cg) tc::g_force_cg = atoi(e);
    const char* rs = getenv("TNN_GEMM_RESERVED_SMS");
    if (rs && !tc::g_reserved_sms) tc::g_reserved_sms = atoi(rs);
    const char* ex2 = getenv("TNN_EXP_FLAGS");     // timing experiments only, see the kernel
    if (ex2) tc::g_exp_flags |= atoi(ex2) & (64 | 128 | 256 | 512 | 1024);
    const char* ks = getenv("TNN_GEMM_KSPLIT");
    if (ks && !tc::g_force_ksplit) tc::g_force_ksplit = atoi(ks);
    env_read = true;
  }
  tc::ActOut act = act_in;
  if (!act.out && act.hi && act.mask_src) TNN_FAIL(std::string(who) + ": the mask_src form needs act_out");
  if (act.out || act.hi) {
    const int64_t need = mix ? 8 : 4;
    if ((act.hi == nullptr) != (act.lo == nullptr)) TNN_FAIL(std::string(who) + ": activation planes come together");
    if (mix && (act.hi == nullptr) != (act.l16 == nullptr)) TNN_FAIL(std::string(who) + ": activation planes come together");
    if (act.hi && (act.ld % need != 0 || act.ld < N)) TNN_FAIL(std::string(who) + ": ld_act must be >= N and suitably padded");
    if (flags & 2) TNN_FAIL(std::string(who) + ": act_out and the relu-in-place flag are exclusive");
  } else {
    act = tc::ActOut();
  }
  const int cg = tc::g_force_cg ? tc::g_force_cg : tc::DEFAULT_CG;
  if (mix) {
    if (cg == 2) return launch_by_layout<2, true>(layout, D, ldd, a, b, M, N, K, bias, flags, act, cond_a, cond_b);
    return launch_by_layout<1, true>(layout, D, ldd, a, b, M, N, K, bias, flags, act, cond_a, cond_b);
  }
  if (cg == 2) return launch_by_layout<2, false>(layout, D, ldd, a, b, M, N, K, bias, flags, act, cond_a, cond_b);
  return launch_by_layout<1, false>(layout, D, ldd, a, b, M, N, K, bias, flags, act, cond_a, cond_b);
}

extern "C" {

int tnn_split_tf32(const float* x, int64_t R, int64_t C, float* hi, float* lo, int64_t ldp,
                   float* hiT, float* loT, int64_t ldt) {
  TNN_REQUIRE_INIT();
  if (R <= 0 || C <= 0) return 0;
  if ((hi == nullptr) != (lo == nullptr) || (hiT == nullptr) != (loT == nullptr))
    TNN_FAIL("tnn_split_tf32: hi/lo planes come in pairs");
  if (hi && (ldp % 4 != 0 || ldp < C)) TNN_FAIL("tnn_split_tf32: ldp must be >= C and a multiple of 4");
  if (hiT && (ldt % 4 != 0 || ldt < R)) TNN_FAIL("tnn_split_tf32: ldt must be >= R and a multiple of 4");
  dim3 grid((unsigned)ceil_div(C, 64), (unsigned)ceil_div(R, 64));
  if (grid.y > 65535) TNN_FAIL("tnn_split_tf32: more than 65535*64 rows");
  int vec_in = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  prof_begin(3);
  tc::split_tf32_kernel<<<grid, 256, 0, ctx().stream>>>(x, R, C, hi, lo, ldp, hiT, loT, ldt, vec_in);
  TNN_POST_LAUNCH();
  prof_end(3);
  return 0;
}

int tnn_set_gemm_group_m(int gm) {
  if (gm == 0 || gm > 64 || gm < -64) TNN_FAIL("tnn_set_gemm_group_m: 1..64 (row groups) or -1..-64 (column panels)");
  tc::g_group_m = gm;
  return 0;
}

int tnn_set_gemm_ksplit(int ks) {
  if (ks != 0 && ks != 1 && ks != 2 && ks != 4) TNN_FAIL("tnn_set_gemm_ksplit: 0 (auto), 1 (off), 2 or 4");
  tc::g_force_ksplit = ks;
  return 0;
}

int tnn_set_gemm_reserved_sms(int n) {
  if (n < 0 || n > 64) TNN_FAIL("tnn_set_gemm_reserved_sms: 0..64");
  tc::g_reserved_sms = n;
  return 0;
}

int tnn_set_gemm_cta_group(int cg) {
  if (cg != 0 && cg != 1 && cg != 2) TNN_FAIL("tnn_set_gemm_cta_group: 0 (default), 1 or 2");
  tc::g_force_cg = cg;
  return 0;
}

int tnn_gemm_tf32x3(float* D, int64_t ldd, const float* a_hi, const float* a_lo, int64_t lda,
                    const float* b_hi, const float* b_lo, int64_t ldb, int64_t M, int64_t N,
                    int64_t K, const float* bias, int flags, int layout, float* act_out,
                    float* act_hi, float* act_lo, int64_t ld_act, const float* mask_src) {
  tc::Planes a{a_hi, a_lo, nullptr, lda}, b{b_hi, b_lo, nullptr, ldb};
  tc::ActOut act;
  act.out = act_out;
  act.hi = act_hi;
  act.lo = act_lo;
  act.ld = ld_act;
  act.mask_src = mask_src;
  return gemm_common("tnn_gemm_tf32x3", false, D, ldd, a, b, M, N, K, bias, flags, layout, act);
}

int tnn_split_tf32_bf16(const float* x, int64_t R, int64_t C, float* hi, void* h16, void* l16,
                        int64_t ld) {
  TNN_REQUIRE_INIT();
  if (R <= 0 || C <= 0) return 0;
  if (!hi || !h16 || !l16) TNN_FAIL("tnn_split_tf32_bf16: all three planes are required");
  if (ld % 8 != 0 || ld < C) TNN_FAIL("tnn_split_tf32_bf16: ld must be >= C and a multiple of 8");
  const int vec_in = (C % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  prof_begin(3);
  tc::split_mix_kernel<<<ew_grid(R * (ld / 8), 256), 256, 0, ctx().stream>>>(
      x, R, C, hi, (__nv_bfloat16*)h16, (__nv_bfloat16*)l16, ld, vec_in);
  TNN_POST_LAUNCH();
  prof_end(3);
  return 0;
}

int tnn_split_tf32_bf16_cond(const float* xa, int64_t Ra, int64_t Ca, float* hia, void* h16a, void* l16a,
                             int64_t lda, int relu_a, const float* xb, int64_t Rb, int64_t Cb, float* hib,
                             void* h16b, void* l16b, int64_t ldb, int relu_b, const void* meta_a,
                             const void* meta_b, void* result_meta) {
  TNN_REQUIRE_INIT();
  if (Ra <= 0 || Ca <= 0 || Rb <= 0 || Cb <= 0) return 0;
  if (!hia || !h16a || !l16a || !hib || !h16b || !l16b) TNN_FAIL("tnn_split_tf32_bf16_cond: all planes are required");
  if (!meta_a || !meta_b) TNN_FAIL("tnn_split_tf32_bf16_cond: both operand meta records are required");
  if (lda % 8 != 0 || lda < Ca || ldb % 8 != 0 || ldb < Cb)
    TNN_FAIL("tnn_split_tf32_bf16_cond: pitches must be >= C and multiples of 8");
  tc::SplitArgs a{xa, Ra, Ca, hia, (__nv_bfloat16*)h16a, (__nv_bfloat16*)l16a, lda,
                  (Ca % 4 == 0) && ((reinterpret_cast<uintptr_t>(xa) & 15) == 0), relu_a};
  tc::SplitArgs b{xb, Rb, Cb, hib, (__nv_bfloat16*)h16b, (__nv_bfloat16*)l16b, ldb,
                  (Cb % 4 == 0) && ((reinterpret_cast<uintptr_t>(xb) & 15) == 0), relu_b};
  // a small grid: this launch returns at once in all but exceptional steps
  dim3 grid((unsigned)ew_grid(std::max(Ra * (lda / 8), Rb * (ldb / 8)), 256, 4), 2);
  prof_begin(3);
  tc::split_mix_cond2_kernel<<<grid, 256, 0, ctx().stream>>>(a, b, (const int*)meta_a, (const int*)meta_b,
                                                             (unsigned int*)result_meta);
  TNN_POST_LAUNCH();
  prof_end(3);
  return 0;
}

int tnn_gemm_tf32_bf16x2(float* D, int64_t ldd, const float* a_hi, const void* a_h16, const void* a_l16,
                         int64_t lda, const float* b_hi, const void* b_h16, const void* b_l16,
                         int64_t ldb, int64_t M, int64_t N, int64_t K, const float* bias, int flags,
                         int layout, float* act_out, float* act_hi, void* act_h16, void* act_l16,
                         int64_t ld_act, const float* mask_src) {
  tc::Planes a{a_hi, a_h16, a_l16, lda}, b{b_hi, b_h16, b_l16, ldb};
  tc::ActOut act;
  act.out = act_out;
  act.hi = act_hi;
  act.lo = (float*)act_h16;
  act.l16 = act_l16;
  act.ld = ld_act;
  act.mask_src = mask_src;
  return gemm_common("tnn_gemm_tf32_bf16x2", true, D, ldd, a, b, M, N, K, bias, flags, layout, act);
}

int tnn_gemm_tf32_bf16x2_cond(float* D, int64_t ldd, const float* a_hi, const void* a_h16, const void* a_l16,
                              int64_t lda, const float* b_hi, const void* b_h16, const void* b_l16,
                              int64_t ldb, int64_t M, int64_t N, int64_t K, const float* bias, int flags,
                              int layout, float* act_out, const float* mask_src, const void* meta_a,
                              const void* meta_b) {
  if (!meta_a || !meta_b) TNN_FAIL("tnn_gemm_tf32_bf16x2_cond: both operand meta records are required");
  tc::Planes a{a_hi, a_h16, a_l16, lda}, b{b_hi, b_h16, b_l16, ldb};
  tc::ActOut act;
  act.out = act_out;
  act.mask_src = mask_src;
  return gemm_common("tnn_gemm_tf32_bf16x2_cond", true, D, ldd, a, b, M, N, K, bias, flags, layout, act,
                     (const int*)meta_a, (const int*)meta_b);
}

}  // extern "C"

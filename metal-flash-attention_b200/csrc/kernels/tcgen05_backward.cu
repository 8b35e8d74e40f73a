// FlashAttention backward for sm_100a: the reference's atomics-free split backward (README.md:11,39) as two
// TMA + tcgen05 + TMEM kernels for 16-bit row-major operands.
//
//   backwardQuery     loopBackwardQuery     AttentionKernel+Source.swift:202-242, computeD +Softmax.swift:32-221
//       per 128-row block of Q, over key blocks c:   S = Q K^T, dP = dO V^T  ->  P = exp2(s2 S - L),
//       dS = P (s dP - D)  ->  dQ += dS K;   also writes D = rowsum(dO * O) / sqrt(D)
//   backwardKeyValue  loopBackwardKeyValue  AttentionKernel+Source.swift:244-293
//       per 128-row block of K/V, over query blocks r:   S^T = K Q^T, dP^T = V dO^T  ->  P^T, dS^T
//       ->  dV += P^T dO,  dK += dS^T Q
//
// Shared structure (384 threads): warps 0-3 / 4-7 are two elementwise warpgroups (thread = TMEM lane = one row of
// the 128 x 128 block; warpgroup h owns columns [64 h, 64 h + 64)); warp 8 issues every tcgen05.mma; warps 9-10 are
// TMA producers (dQ: K ring / V ring; dK-dV: Q and dO rings / the L, D vector loader); warps 10-11 also rewrite BF16 dO
// tiles as FP16 when the reference's mixed policy is in use.  No row reductions are needed in the backward pass (L and
// D are inputs).  All four "accumulate" GEMMs take their A operand (P, dS, P^T, dS^T: 16-bit) straight from TMEM,
// written over the FP32 S / dP they came from.  Each elementwise pass is split in two -- the exponentials need only S,
// the dS half needs dP -- and the tensor-pipe issue order and operand rings are arranged so that what the next pass
// starts with is issued a pass ahead (kernel headers below; measurements in DESIGN.md 4.1c).  Small grids are split
// along the traversal axis (blockIdx.z) and merged by sum_splits.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include "accumulator_store.cuh"
#include "attention_params.h"
#include "backward_common.cuh"
#include "device_state.h"
#include "sm100_ptx.cuh"
#include "tma_host.h"

namespace mfa {
namespace bwd {

using namespace ptx;

constexpr uint32_t kTile = 128;   // rows of the parallelised operand per CTA and rows per traversal block
constexpr uint32_t kHalf = 64;    // columns per elementwise warpgroup
constexpr uint32_t kSubTileBytes = 128 * 128;  // [128 rows][64 x 16-bit]: one 128B-swizzled TMA box
constexpr uint32_t kThreads = 384;
constexpr uint32_t kElemThreads = 256;
constexpr uint32_t kLaunchRegs = 168, kElemRegs = 208, kOtherRegs = 88;
static_assert(kElemRegs * 256 + kOtherRegs * 128 <= kLaunchRegs * kThreads, "setmaxnreg over-subscribed");

// kPoly (template parameter of both kernels, from the parameter-table row): of every 4 element pairs of P, how many
// take exp2 on the FMA pipe (exp2_poly2, sm100_ptx.cuh) instead of the MUFU pipe.  At D = 64 a block's MMAs need 768
// (dQ) / 1024 (dK/dV) tensor-pipe cycles but its 128 x 128 exponentials 1024 MUFU cycles (16 ex2 / clk / SM): the P half
// of the elementwise pass is MUFU-bound, so part of the pairs go to the FMA pipe.  At D = 128 the kernels are
// tensor-bound and the extra FMA-pipe instructions only cost issue slots.  Swept on B200 (scripts/sweep.py; round-2
// numbers with packed dS arithmetic, TFLOP/s, dQ | dK/dV, N = 4096):  D=128: 0 -> 1330 | 1280, 1 -> 1300 | 1290,
// 3 -> 1270 | 1235;  D=64: 0 -> 924 | 873, 1 -> 962 | 911, 2 -> 946 | 948, 3 -> 862 | 846.
// p0, p1 <- exp2(p * scale - l) for pair index `pair` (a compile-time constant once the caller's loop is unrolled)
template <uint32_t kPoly>
__device__ __forceinline__ void exp2_pair(uint32_t pair, float &p0, float &p1, float scale, float l0, float l1) {
  const float2 x = ffma2(make_float2(p0, p1), make_float2(scale, scale), make_float2(-l0, -l1));
  if (kPoly > 0 && (pair & 3) < kPoly) {
    const float2 r = exp2_poly2<false>(x);  // x = s - L <= ~0: no upper clamp needed
    p0 = r.x;
    p1 = r.y;
  } else {
    p0 = ex2_approx(x.x);
    p1 = ex2_approx(x.y);
  }
}

struct BackwardArgs {
  const void *dO;   // [batch][R][D] 16-bit (element type of Q/K/V, or BF16 beside FP16 Q/K/V: kConvertDO)
  const float *O;   // [batch][R][D] FP32
  const void *L;    // [batch][R]
  void *Dterm;      // [batch][R]
  float *dQ, *dV, *dK;  // FP32 outputs
  uint32_t R, C, D;
  float scale, scale_log2;
  int l_prec, d_prec;
  // traversal split (small grids): blockIdx.z = split s handles traversal blocks [s * blocks_per_split, ...) and writes
  // its partial accumulators to slice s of the outputs (which then point at scratch; split_stride floats apart)
  uint32_t blocks_per_split;
  size_t split_stride;
  // work decomposition: item -> (split, head, tile)
  uint32_t tiles, batch, num_splits, num_items;
};

// ================================================================================================
// backwardQuery
//   TMEM columns: [0,128) S (single buffer, released as soon as it is in registers),
//                 [128,256) [256,384) dP double buffer (dS is written in place over dP),  [384,384+D) dQ
//   Shared memory: Q and dO tiles resident; K in a ring of THREE stages (block j's tile is read by S(j) and, two
//   pipeline steps later, by dQ(j): with two stages the load of K(j+1) had to wait for dQ(j-1) to retire and S(j+1)
//   -- which the next block's elementwise pass waits for -- sat behind a TMA round trip); V in a ring of two.
//   Tensor-pipe order per block j:  dQ(j-1)  ->  S(j+1)  ->  dP(j+1).  The elementwise warps split their pass so that
//   the exponentials (which need only S) run while dP is still on the pipe: measured 2310 -> see DESIGN.md.
// ================================================================================================
template <uint32_t DPAD, bool kOffload = false>
struct QueryConfig {
  static constexpr uint32_t kSubTiles = DPAD / 64;
  static constexpr uint32_t kTileBytes = kSubTiles * kSubTileBytes;  // one 128 x DPAD 16-bit tile
  static constexpr uint32_t kStagesK = 3, kStagesV = 2;
  // D <= 64: persistent CTAs.  Q / dO are double-buffered in shared memory and the dQ accumulator in TMEM, so the next
  // work item's tiles land -- and its first S / dP are computed -- while the elementwise warps finish and store the
  // current one; the epilogue then needs a scratch tile of its own (the K ring is live).  D = 128 has no room for
  // either (224 KB of operand tiles, 512 TMEM columns): one work item per CTA, scratch overlays the dead K ring.
  static constexpr bool kPersistent = DPAD <= 64;
  static constexpr uint32_t kBuffers = kPersistent ? 2 : 1;
  static constexpr uint32_t kSmemQ = 0;
  static constexpr uint32_t kSmemdO = kBuffers * kTileBytes;
  static constexpr uint32_t kSmemK = 2 * kBuffers * kTileBytes;
  static constexpr uint32_t kSmemV = kSmemK + kStagesK * kTileBytes;
  static constexpr uint32_t kSmemScratch = kPersistent ? kSmemV + kStagesV * kTileBytes : kSmemK;  // 8 warps x 4 KB
  // persistent: warp 11 stages the next item's O (FP32) and dO rows here for D = rowsum(dO * O)
  static constexpr bool kOffloadD = kOffload;  // (its own instantiation: the staging area costs the inline form ~4 %)
  static_assert(!kOffload || kPersistent, "the D-term is only offloaded in the persistent form");
  static constexpr uint32_t kStageBytes = kOffloadD ? kTile * DPAD * 6 : 0;
  static constexpr uint32_t kSmemStage = kSmemV + kStagesV * kTileBytes + (kPersistent ? 8 * 4096 : 0);
  static constexpr uint32_t kSmemVec = kSmemStage + kStageBytes;  // float D[128] (persistent: one per item parity)
  static constexpr uint32_t kSmemBar = kSmemVec + 2 * kTile * 4;
  static constexpr uint32_t kNumBars = 30;
  static constexpr uint32_t kSmemTmemPtr = kSmemBar + kNumBars * 8;
  static constexpr uint32_t kSmemBytes = kSmemTmemPtr + 16;
  static_assert(kSmemBytes <= 232448, "shared memory over budget");
  static_assert(8 * 4096 <= kStagesK * kTileBytes, "epilogue scratch does not fit the K stages");
  static_assert(384 + kBuffers * DPAD <= 512, "dQ accumulators do not fit TMEM");
};

template <uint32_t DPAD, bool kBF16, bool kConvertDO, uint32_t kPoly, bool kOffload>
__global__ void __launch_bounds__(kThreads, 1)
    attention_backward_query_tcgen05(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapdO,
                                     const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapV,
                                     const BackwardArgs a) {
  using Cfg = QueryConfig<DPAD, kOffload>;
  constexpr uint32_t kDB = Cfg::kBuffers;
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t total_blocks = (a.C + kTile - 1) / kTile;
  constexpr uint32_t kTmemS = 0, kTmemdP = 128, kTmemdQ = 384, kTmemCols = 512;
  // work item -> (traversal split, head, 128-row tile of Q); items blockIdx.x, blockIdx.x + gridDim.x, ... (the
  // non-persistent instantiation is launched with one CTA per item).  `g0` counts the key blocks this CTA has processed
  // before the current item: every ring stage and barrier phase below is a function of the global block index g0 + j.
  auto decode = [&](uint32_t item, uint32_t &r0, uint32_t &head, uint32_t &split, uint32_t &blk0, uint32_t &num_blocks) {
    r0 = (item % a.tiles) * kTile;
    head = (item / a.tiles) % a.batch;
    split = item / (a.tiles * a.batch);
    blk0 = split * a.blocks_per_split;  // first key block of this split (host: never empty)
    num_blocks = min(a.blocks_per_split, total_blocks - blk0);
  };

  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::kSmemBar);
  uint64_t *q_full = bars;            // [2] Q and dO tiles of the item landed
  uint64_t *q_empty = bars + 2;       // [2] every MMA of the item has completed: the buffers may be reloaded
  uint64_t *k_full = bars + 4;        // [3]
  uint64_t *k_empty = bars + 7;       // [3]
  uint64_t *v_full = bars + 10;       // [2]
  uint64_t *v_empty = bars + 12;      // [2]
  uint64_t *s_full = bars + 14;       // S(g) in TMEM
  uint64_t *s_free = bars + 15;       // S(g) is in registers (256 arrivals)
  uint64_t *dp_full = bars + 16;      // [2] dP(g) in TMEM
  uint64_t *ds_full = bars + 18;      // [2] dS(g) written over dP(g) (256 arrivals)
  uint64_t *dq_final = bars + 20;     // one phase per item: the item's last dQ += dS K has completed
  uint64_t *do_ready = bars + 21;     // kConvertDO, one phase per item: the dO tile has been rewritten as FP16 (256)
  uint64_t *dq_free = bars + 22;      // [2] the epilogue has read this dQ accumulator out of TMEM (256 arrivals)
  uint64_t *dterm_full = bars + 24;   // [2] persistent form: warp 11 has written the item's D vector (32 arrivals)
  uint64_t *dterm_empty = bars + 26;  // [2] ... and every elementwise thread has read it (256 arrivals)
  uint64_t *stage_full = bars + 28;   // persistent form: the item's O and dO rows have landed in the staging area
  static_assert(!(kBF16 && kConvertDO), "dO is only converted when Q, K, V are FP16");
  constexpr bool kDOisBF16 = kBF16 || kConvertDO;  // element type of dO in global memory
  uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(smem + Cfg::kSmemTmemPtr);

  if (threadIdx.x == 0) {
    for (uint32_t s = 0; s < 2; ++s) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], 1);
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], 1);
      mbar_init(&dp_full[s], 1);
      mbar_init(&ds_full[s], kElemThreads);
      mbar_init(&dq_free[s], kElemThreads);
      mbar_init(&dterm_full[s], 32);
      mbar_init(&dterm_empty[s], kElemThreads);
    }
    for (uint32_t s = 0; s < Cfg::kStagesK; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(s_free, kElemThreads);
    mbar_init(dq_final, 1);
    mbar_init(do_ready, kElemThreads);
    mbar_init(stage_full, 1);
    fence_barrier_init();
  }
  if (warp == 8) {
    tmem_alloc(tmem_ptr_smem, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  // traversal split: let the sum kernel (launched with programmatic stream serialisation) be set up now; its
  // griddepcontrol.wait still holds it until this grid has completed and flushed
  if (a.num_splits > 1) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp < 8) {
    // ---------------- elementwise warpgroups ----------------
    setmaxnreg_inc<kElemRegs>();
    const uint32_t h = warp >> 2, quarter = warp & 3;
    const uint32_t row_in_tile = quarter * 32 + lane;
    const uint32_t tLane = tmem_base + ((quarter * 32) << 16);

    uint32_t g0 = 0;
    float Lnext = 0.f;
    for (uint32_t item = blockIdx.x, it = 0; item < a.num_items; item += gridDim.x, ++it) {
      uint32_t r0, head, split, blk0, num_blocks;
      decode(item, r0, head, split, blk0, num_blocks);
      const uint32_t qb = it % kDB, q_phase = (it / kDB) & 1;
      const uint32_t row = r0 + row_in_tile;
      const uint32_t row_c = min(row, a.R - 1);  // clamped like clampedParallelizationThreadOffset (AttentionKernel.swift:224-226)

      if constexpr (kConvertDO) {
        // BF16 dO tile (TMA) -> FP16 in place; elementwise, so the 128 B swizzle is irrelevant.  Generic-proxy writes
        // must be fenced before the tensor core (async proxy) reads them.
        mbar_wait(&q_full[qb], q_phase);
        uint4 *tile = reinterpret_cast<uint4 *>(smem + Cfg::kSmemdO + qb * Cfg::kTileBytes);
#pragma unroll
        for (uint32_t i = 0; i < Cfg::kTileBytes / (kElemThreads * 16); ++i)
          tile[i * kElemThreads + threadIdx.x] = bf16x8_to_f16x8(tile[i * kElemThreads + threadIdx.x]);
        fence_proxy_async_smem();
        mbar_arrive(do_ready);
      }

      // computeD (AttentionKernel+Softmax.swift:32-221): D = (sum_d dO * O) / sqrt(D), kept in FP32 for this kernel and
      // stored (possibly as BF16) for the dK/dV kernel.  A row per thread (what the MMA layout would suggest) makes every
      // warp load touch 32 different cache lines -- the profile showed the elementwise warps spending 17 % of the kernel
      // here -- so each warp instead takes 16 rows and spreads the columns over its lanes (one 512 B line of O per load),
      // reduces with shuffles and hands the results to the row owners through shared memory.
      float Dterm;
      constexpr bool offload = Cfg::kOffloadD;
      if constexpr (offload) {
        // computed off the critical path by warp 11, one item ahead (see there)
        const uint32_t db = it & 1;
        mbar_wait(&dterm_full[db], (it >> 1) & 1);
        Dterm = reinterpret_cast<const float *>(smem + Cfg::kSmemVec)[db * kTile + row_in_tile];
        mbar_arrive(&dterm_empty[db]);
      } else
      {
        float *dvec = reinterpret_cast<float *>(smem + Cfg::kSmemVec);
        constexpr uint32_t kRowsPerWarp = kTile / 8;
        float4 o4[kRowsPerWarp];
        uint2 g4[kRowsPerWarp];
        const bool active = 4 * lane < a.D;
#pragma unroll
        for (uint32_t i = 0; i < kRowsPerWarp; ++i) {
          const uint32_t rr = min(r0 + warp * kRowsPerWarp + i, a.R - 1);
          const size_t base = (static_cast<size_t>(head) * a.R + rr) * a.D + 4 * lane;
          o4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
          g4[i] = make_uint2(0u, 0u);
          if (active) {
            o4[i] = ldg_stream_f32x4(a.O + base);
            g4[i] = ldg_stream_u32x2(static_cast<const uint16_t *>(a.dO) + base);
          }
        }
#pragma unroll
        for (uint32_t i = 0; i < kRowsPerWarp; ++i) {
          float v0, v1, v2, v3;
          if (kDOisBF16) {
            v0 = __uint_as_float(g4[i].x << 16);
            v1 = __uint_as_float(g4[i].x & 0xFFFF0000u);
            v2 = __uint_as_float(g4[i].y << 16);
            v3 = __uint_as_float(g4[i].y & 0xFFFF0000u);
          } else {
            const __half2 lo = *reinterpret_cast<const __half2 *>(&g4[i].x), hi = *reinterpret_cast<const __half2 *>(&g4[i].y);
            v0 = __low2float(lo); v1 = __high2float(lo); v2 = __low2float(hi); v3 = __high2float(hi);
          }
          float acc = fmaf(v0, o4[i].x, fmaf(v1, o4[i].y, fmaf(v2, o4[i].z, v3 * o4[i].w)));
#pragma unroll
          for (uint32_t off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
          if (lane == i) dvec[warp * kRowsPerWarp + i] = acc * a.scale;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kElemThreads) : "memory");  // the eight elementwise warps only
        Dterm = dvec[row_in_tile];
      }
      const size_t stat_idx = static_cast<size_t>(head) * a.R + row_c;
      // (persistent form: fetched during the previous item's epilogue, see below)
      const float Lrow = (Cfg::kPersistent && it > 0) ? Lnext : load_stat(a.L, stat_idx, a.l_prec);
      if (!offload && h == 0 && row < a.R && split == 0) store_stat(a.Dterm, stat_idx, a.d_prec, Dterm);

      for (uint32_t j = 0; j < num_blocks; ++j) {
        const uint32_t g = g0 + j, bf = g & 1;
        const uint32_t tS = tLane + kTmemS + h * kHalf;
        const uint32_t tdP = tLane + kTmemdP + bf * kTile + h * kHalf;
        // ---- first half of the pass: P = exp2(S * log2e/sqrt(D) - L) needs only S ----
        mbar_wait(s_full, g & 1);
        tc_fence_after();
        float p[kHalf];
#pragma unroll
        for (uint32_t c = 0; c < kHalf; c += 32) tmem_ld32(tS + c, *reinterpret_cast<uint32_t(*)[32]>(&p[c]));
        tc_wait_ld();
        tc_fence_before();
        mbar_arrive(s_free);  // S(g+1) may overwrite the S buffer now

        const uint32_t col0 = (blk0 + j) * kTile + h * kHalf;
        if (blk0 + j + 1 == total_blocks && col0 + kHalf > a.C) {  // padded key columns (maskAttentionMatrixEdge): P = 0 there
#pragma unroll
          for (uint32_t c = 0; c < kHalf; ++c)
            if (col0 + c >= a.C) p[c] = -INFINITY;
        }
        // P = exp2(S * log2e/sqrt(D) - L)   (+Softmax.swift:419-427)
#pragma unroll
        for (uint32_t i = 0; i < kHalf / 2; ++i) exp2_pair<kPoly>(i, p[2 * i], p[2 * i + 1], a.scale_log2, Lrow, Lrow);

        // ---- second half: dS = P * (dP/sqrt(D) - D), written in place over dP as the 16-bit A operand of dQ += dS K ----
        mbar_wait(&dp_full[bf], (g >> 1) & 1);
        tc_fence_after();
        uint32_t dp[kHalf];
#pragma unroll
        for (uint32_t c = 0; c < kHalf; c += 32) tmem_ld32(tdP + c, *reinterpret_cast<uint32_t(*)[32]>(&dp[c]));
        tc_wait_ld();
        const float2 scale2 = make_float2(a.scale, a.scale), negD2 = make_float2(-Dterm, -Dterm);
#pragma unroll
        for (uint32_t c = 0; c < kHalf; c += 32) {
          uint32_t packed[16];
#pragma unroll
          for (uint32_t k = 0; k < 16; ++k) {
            // packed FP32x2 arithmetic: the elementwise pass is bound by instruction issue (one 32-wide FP32
            // instruction per two cycles and sub-partition), so two elements per FFMA2 / FMUL2 halve its cost
            const float2 t = ffma2(make_float2(__uint_as_float(dp[c + 2 * k]), __uint_as_float(dp[c + 2 * k + 1])), scale2, negD2);
            const float2 ds = fmul2(make_float2(p[c + 2 * k], p[c + 2 * k + 1]), t);
            packed[k] = kBF16 ? pack_bf16x2(ds.x, ds.y) : pack_f16x2(ds.x, ds.y);
          }
          tmem_st16(tdP + (c >> 1), packed);  // dS of keys [64h + c, +32) -> columns [64h + c/2, +16) of the dP buffer
        }
        tc_wait_st();
        tc_fence_before();
        mbar_arrive(&ds_full[bf]);
      }

      // the next item's L: issued now so that its latency hides under the wait for the last MMA and the epilogue
      if (Cfg::kPersistent && item + gridDim.x < a.num_items) {
        uint32_t nr0, nhead, nsplit, nblk0, nblocks;
        decode(item + gridDim.x, nr0, nhead, nsplit, nblk0, nblocks);
        Lnext = load_stat(a.L, static_cast<size_t>(nhead) * a.R + min(nr0 + row_in_tile, a.R - 1), a.l_prec);
      }
      // epilogue: dQ -> global (FP32); warpgroup h writes columns [h D/2, (h+1) D/2)
      mbar_wait(dq_final, it & 1);
      tc_fence_after();
      {
        float4 *scratch = reinterpret_cast<float4 *>(smem + Cfg::kSmemScratch) + warp * 256;
        const uint32_t warp_row0 = r0 + quarter * 32;
        store_accumulator_coalesced(tLane + kTmemdQ + qb * DPAD, h * (DPAD / 2), DPAD / 2, scratch,
                                    a.dQ + split * a.split_stride + (static_cast<size_t>(head) * a.R + warp_row0) * a.D,
                                    warp_row0, a.R, a.D, lane);
      }
      // this dQ accumulator is out of TMEM: a later item's first dQ = dS K (accumulate off) may overwrite it
      tc_fence_before();
      mbar_arrive(&dq_free[qb]);
      g0 += num_blocks;
    }  // work items
  } else {
    setmaxnreg_dec<kOtherRegs>();
    if (warp == 9) {
      // ---------------- TMA producer: Q, dO of every item, and the K ring ----------------
      uint32_t g0 = 0;
      for (uint32_t item = blockIdx.x, it = 0; item < a.num_items; item += gridDim.x, ++it) {
        uint32_t r0, head, split, blk0, num_blocks;
        decode(item, r0, head, split, blk0, num_blocks);
        const uint32_t qb = it % kDB;
        mbar_wait(&q_empty[qb], ((it / kDB) & 1) ^ 1);  // the item that used these buffers last is done with them
        if (elect_one()) {
          mbar_arrive_expect_tx(&q_full[qb], 2 * Cfg::kTileBytes);
#pragma unroll
          for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds) {
            tma_load_3d(smem + Cfg::kSmemQ + qb * Cfg::kTileBytes + ds * kSubTileBytes, &mapQ, &q_full[qb], ds * 64, r0, head);
            tma_load_3d(smem + Cfg::kSmemdO + qb * Cfg::kTileBytes + ds * kSubTileBytes, &mapdO, &q_full[qb], ds * 64, r0, head);
          }
        }
        for (uint32_t j = 0; j < num_blocks; ++j) {
          const uint32_t g = g0 + j, stage = g % Cfg::kStagesK, phase = (g / Cfg::kStagesK) & 1;
          mbar_wait(&k_empty[stage], phase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&k_full[stage], Cfg::kTileBytes);
#pragma unroll
            for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
              tma_load_3d(smem + Cfg::kSmemK + stage * Cfg::kTileBytes + ds * kSubTileBytes, &mapK, &k_full[stage],
                          ds * 64, (blk0 + j) * kTile, head);
          }
        }
        g0 += num_blocks;
      }
    } else if (warp == 10) {
      // ---------------- TMA producer for the V ring ----------------
      uint32_t g0 = 0;
      for (uint32_t item = blockIdx.x; item < a.num_items; item += gridDim.x) {
        uint32_t r0, head, split, blk0, num_blocks;
        decode(item, r0, head, split, blk0, num_blocks);
        for (uint32_t j = 0; j < num_blocks; ++j) {
          const uint32_t g = g0 + j, stage = g & 1, phase = (g >> 1) & 1;
          mbar_wait(&v_empty[stage], phase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&v_full[stage], Cfg::kTileBytes);
#pragma unroll
            for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
              tma_load_3d(smem + Cfg::kSmemV + stage * Cfg::kTileBytes + ds * kSubTileBytes, &mapV, &v_full[stage],
                          ds * 64, (blk0 + j) * kTile, head);
          }
        }
        g0 += num_blocks;
      }
    } else if (warp == 11) {
      // ---------------- persistent form: D = rowsum(dO * O) / sqrt(D) of every item, one item ahead ----------------
      // (computeD, AttentionKernel+Softmax.swift:32-221.)  In the one-item-per-CTA form the elementwise warps compute it
      // while the first tiles are in flight anyway; with persistent CTAs it sat at the head of every item (global-load
      // latency with nothing to overlap: ~2 k of the ~7 k cycles between two items' block loops), so the otherwise idle
      // warp 11 produces the vector of item it+1 while item it is being processed.  The item's rows of O and dO are one
      // contiguous range each (row-major, leading dimension D): two bulk copies bring them into a staging area -- no
      // registers in flight, so the whole 48 KB is outstanding at once (register-staged loads, eight per lane, took longer
      // than an N = 2048 item lasts) -- and the warp then reduces from shared memory, four rows per lane.
      if constexpr (Cfg::kOffloadD) {
        float *dvec = reinterpret_cast<float *>(smem + Cfg::kSmemVec);
        const float *stO = reinterpret_cast<const float *>(smem + Cfg::kSmemStage);
        const uint16_t *stG = reinterpret_cast<const uint16_t *>(smem + Cfg::kSmemStage + kTile * DPAD * 4);
        const uint32_t chunks = a.D / 4;  // float4 chunks per row
        for (uint32_t item = blockIdx.x, it = 0; item < a.num_items; item += gridDim.x, ++it) {
          uint32_t r0, head, split, blk0, num_blocks;
          decode(item, r0, head, split, blk0, num_blocks);
          const uint32_t db = it & 1;
          const uint32_t rows = min(kTile, a.R - r0);  // rows past R keep whatever the staging area held: never stored
          if (elect_one()) {
            const size_t first = (static_cast<size_t>(head) * a.R + r0) * a.D;
            mbar_arrive_expect_tx(stage_full, rows * a.D * 6);
            bulk_load_1d(smem + Cfg::kSmemStage, a.O + first, rows * a.D * 4, stage_full);
            bulk_load_1d(smem + Cfg::kSmemStage + kTile * DPAD * 4, static_cast<const uint16_t *>(a.dO) + first,
                         rows * a.D * 2, stage_full);
          }
          __syncwarp();
          mbar_wait(&dterm_empty[db], ((it >> 1) & 1) ^ 1);
          mbar_wait(stage_full, it & 1);
          // lane = rows lane, lane + 32, lane + 64, lane + 96; the lanes walk their rows' chunks on a diagonal so that a
          // warp access spreads over the banks (rows are D * 4 bytes apart).  No shuffles, no branches: the four
          // accumulators are independent FMA chains.
          float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
          for (uint32_t step = 0; step < chunks; ++step) {
            uint32_t c = step + lane;
            c -= (c / chunks) * chunks;
#pragma unroll
            for (uint32_t q = 0; q < 4; ++q) {
              const uint32_t rt = lane + 32 * q;
              const float4 o = *reinterpret_cast<const float4 *>(stO + rt * a.D + 4 * c);
              const uint2 g = *reinterpret_cast<const uint2 *>(stG + rt * a.D + 4 * c);
              const float2 lo = kDOisBF16 ? unpack_bf16x2(g.x) : unpack_f16x2(g.x);
              const float2 hi = kDOisBF16 ? unpack_bf16x2(g.y) : unpack_f16x2(g.y);
              acc[q] = fmaf(lo.x, o.x, fmaf(lo.y, o.y, fmaf(hi.x, o.z, fmaf(hi.y, o.w, acc[q]))));
            }
          }
#pragma unroll
          for (uint32_t q = 0; q < 4; ++q) {
            const uint32_t rt = lane + 32 * q;
            const float d = acc[q] * a.scale;
            dvec[db * kTile + rt] = d;
            if (split == 0 && r0 + rt < a.R) store_stat(a.Dterm, static_cast<size_t>(head) * a.R + r0 + rt, a.d_prec, d);
          }
          __syncwarp();  // every lane has read the staging area before the next item's copies overwrite it
          mbar_arrive(&dterm_full[db]);  // (release: orders this lane's vector writes before the readers' acquire)
        }
      }
    } else if (warp == 8) {
      // ---------------- MMA issuer ----------------
      constexpr uint32_t kFormat = kBF16 ? 1u : 0u;
      constexpr uint32_t idescNT = make_idesc_f16(kTile, kTile, kFormat, 0, 0);  // [128 x D] . [128 x D]^T
      constexpr uint32_t idescAcc = make_idesc_f16(kTile, DPAD, kFormat, 0, 1);  // TMEM A . MN-major B -> [128 x DPAD]
      const uint64_t descQ = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemQ), 16, 1024);
      const uint64_t descdO = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemdO), 16, 1024);
      const uint64_t descK = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemK), 16, 1024);
      const uint64_t descV = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemV), 16, 1024);
      const uint64_t descKmn = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemK), kSubTileBytes, 1024);

      auto issue_nt = [&](uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc) {
#pragma unroll
        for (uint32_t k = 0; k < DPAD / 16; ++k) {
          const uint32_t off = ((k >> 2) * kSubTileBytes + (k & 3) * 32) >> 4;
          umma_ss(d_tmem, a_desc + off, b_desc + off, idescNT, k > 0);
        }
      };
      auto issue_dQ = [&](uint32_t qb, uint32_t bf, uint32_t stage, uint32_t accumulate) {
        const uint64_t b0 = descKmn + ((stage * Cfg::kTileBytes) >> 4);
#pragma unroll
        for (uint32_t k = 0; k < kTile / 16; ++k) {
          // dS of keys [64 hh, 64 hh + 64) sits in columns [64 hh, 64 hh + 32) of the dP buffer
          const uint32_t a_tmem = tmem_base + kTmemdP + bf * kTile + (k >> 2) * kHalf + (k & 3) * 8;
          umma_ts(tmem_base + kTmemdQ + qb * DPAD, a_tmem, b0 + ((k * 2048) >> 4), idescAcc, k > 0 ? 1u : accumulate);
        }
      };

      uint32_t g0 = 0;
      for (uint32_t item = blockIdx.x, it = 0; item < a.num_items; item += gridDim.x, ++it) {
        uint32_t r0, head, split, blk0, num_blocks;
        decode(item, r0, head, split, blk0, num_blocks);
        const uint32_t qb = it % kDB, q_phase = (it / kDB) & 1;
        const uint64_t descQb = descQ + ((qb * Cfg::kTileBytes) >> 4), descdOb = descdO + ((qb * Cfg::kTileBytes) >> 4);

        // prologue: S(g0), dP(g0).  For every item but the first they are issued while the elementwise warps are still
        // storing the previous item's dQ: the S buffer only needs the previous item's last S to have been read out
        // (s_free), the dP buffer's last reader dQ(g0 - 2) is ahead on the in-order tensor pipe.
        {
          const uint32_t ks = g0 % Cfg::kStagesK, vs = g0 & 1;
          mbar_wait(&q_full[qb], q_phase);
          if (it > 0) mbar_wait(s_free, (g0 - 1) & 1);
          mbar_wait(&k_full[ks], (g0 / Cfg::kStagesK) & 1);
          tc_fence_after();
          if (elect_one()) {
            issue_nt(tmem_base + kTmemS, descQb, descK + ((ks * Cfg::kTileBytes) >> 4));
            umma_commit(s_full);
          }
          __syncwarp();
          mbar_wait(&v_full[vs], (g0 >> 1) & 1);
          if constexpr (kConvertDO) mbar_wait(do_ready, it & 1);
          tc_fence_after();
          if (elect_one()) {
            issue_nt(tmem_base + kTmemdP + vs * kTile, descdOb, descV + ((vs * Cfg::kTileBytes) >> 4));
            umma_commit(&dp_full[vs]);
            umma_commit(&v_empty[vs]);
          }
          __syncwarp();
        }

        for (uint32_t j = 0; j < num_blocks; ++j) {
          const uint32_t g = g0 + j;
          // (a) dQ += dS(g-1) K(g-1): frees K's stage and the dP buffer that dP(g+1) is about to overwrite
          if (j > 0) {
            const uint32_t pg = g - 1, ks = pg % Cfg::kStagesK;
            mbar_wait(&ds_full[pg & 1], (pg >> 1) & 1);
            // the item's first dQ MMA overwrites the accumulator: its previous user's epilogue must have read it out
            if (j == 1) mbar_wait(&dq_free[qb], q_phase ^ 1);
            tc_fence_after();
            if (elect_one()) {
              issue_dQ(qb, pg & 1, ks, j > 1 ? 1u : 0u);
              umma_commit(&k_empty[ks]);
            }
            __syncwarp();
          }
          if (j + 1 < num_blocks) {
            const uint32_t ng = g + 1, ks = ng % Cfg::kStagesK, vs = ng & 1;
            // (b) S(g+1) as soon as S(g) has been read out: first in line for the next elementwise pass
            mbar_wait(s_free, g & 1);
            mbar_wait(&k_full[ks], (ng / Cfg::kStagesK) & 1);
            tc_fence_after();
            if (elect_one()) {
              issue_nt(tmem_base + kTmemS, descQb, descK + ((ks * Cfg::kTileBytes) >> 4));
              umma_commit(s_full);
            }
            __syncwarp();
            // (c) dP(g+1) into the buffer dS(g-1) just left (in-order tensor pipe: after dQ(g-1))
            mbar_wait(&v_full[vs], (ng >> 1) & 1);
            tc_fence_after();
            if (elect_one()) {
              issue_nt(tmem_base + kTmemdP + vs * kTile, descdOb, descV + ((vs * Cfg::kTileBytes) >> 4));
              umma_commit(&dp_full[vs]);
              umma_commit(&v_empty[vs]);
            }
            __syncwarp();
          }
        }
        {
          const uint32_t pg = g0 + num_blocks - 1, ks = pg % Cfg::kStagesK;
          mbar_wait(&ds_full[pg & 1], (pg >> 1) & 1);
          if (num_blocks == 1) mbar_wait(&dq_free[qb], q_phase ^ 1);
          tc_fence_after();
          if (elect_one()) {
            issue_dQ(qb, pg & 1, ks, num_blocks > 1 ? 1u : 0u);
            umma_commit(&k_empty[ks]);
            umma_commit(dq_final);
            umma_commit(&q_empty[qb]);  // (every MMA that read this item's Q / dO has completed as well)
          }
          __syncwarp();
        }
        g0 += num_blocks;
      }  // work items
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ================================================================================================
// backwardKeyValue
//   TMEM columns: two 128-column regions X = [0,128), Y = [128,256) that swap roles every block, dV [256,256+D),
//   dK [256+D,256+2D).  For query block r (Rs = X, Rd = Y when r is even, swapped when odd):
//     S^T(r) (FP32) lands in Rs, dP^T(r) in Rd.  Once both warpgroups hold S^T(r) in registers, P^T(r) (16-bit) goes
//     to Rs[0,64) and, later, dS^T(r) to Rs[64,128) -- the two 16-bit A operands share ONE region, so Rd is free the
//     moment dP^T(r) has been read and S^T(r+1) = K Q(r+1)^T is issued into it while the warps are still computing
//     dS^T(r).  dP^T(r+1) follows dV(r), dK(r) into Rs (in-order tensor pipe).
//   Tensor-pipe order per block:  dV(r) [after the P half of the pass]  ->  S^T(r+1)  ->  dK(r)  ->  dP^T(r+1).
//   The previous form (S^T, dP^T -> one elementwise pass -> dV, dK, everything serialised) left the tensor pipe
//   idle for the whole pass: 45 % active, the elementwise warps waiting 57 % of the time (profiles/).
// ================================================================================================
template <uint32_t DPAD>
struct KeyValueConfig {
  static constexpr uint32_t kSubTiles = DPAD / 64;
  static constexpr uint32_t kTileBytes = kSubTiles * kSubTileBytes;  // one 128 x DPAD 16-bit tile
  // Q(r) is first read by S^T(r) in the middle of pass r-1 and last by dK(r) at the end of pass r, dO(r) first by
  // dP^T(r) at the end of pass r-1 and last by dV(r) in the middle of pass r: with one shared two-stage ring the load of
  // Q(r+1) could not start before dK(r-1) had retired and S^T(r+1) waited for a TMA round trip (22 % of the elementwise
  // warps' time in the profile).  Separate rings, three stages of Q, two of dO.
  static constexpr uint32_t kStagesQ = 3, kStagesdO = 2;
  // D <= 64: persistent CTAs with K / V double-buffered, so the next work item's tiles land and its first S^T / dP^T are
  // computed while the elementwise warps store the current item's dV and dK (which then need a scratch tile of their
  // own).  D = 128: no shared memory left for that; one work item per CTA, scratch overlays the dead Q ring.
  static constexpr bool kPersistent = DPAD <= 64;
  static constexpr uint32_t kBuffers = kPersistent ? 2 : 1;
  static constexpr uint32_t kSmemK = 0;
  static constexpr uint32_t kSmemV = kBuffers * kTileBytes;
  static constexpr uint32_t kSmemQ = 2 * kBuffers * kTileBytes;
  static constexpr uint32_t kSmemdO = kSmemQ + kStagesQ * kTileBytes;
  static constexpr uint32_t kSmemScratch = kPersistent ? kSmemdO + kStagesdO * kTileBytes : kSmemQ;  // 8 warps x 4 KB
  static constexpr uint32_t kSmemVec = kSmemdO + kStagesdO * kTileBytes + (kPersistent ? 8 * 4096 : 0);  // float L[2][128], D[2][128]
  static constexpr uint32_t kSmemBar = kSmemVec + 4 * kTile * 4;
  static constexpr uint32_t kNumBars = 32;
  static constexpr uint32_t kSmemTmemPtr = kSmemBar + kNumBars * 8;
  static constexpr uint32_t kSmemBytes = kSmemTmemPtr + 16;
  static_assert(kSmemBytes <= 232448, "shared memory over budget");
  static_assert(8 * 4096 <= kStagesQ * kTileBytes, "epilogue scratch does not fit the Q stages");
};

template <uint32_t DPAD, bool kBF16, bool kConvertDO, uint32_t kPoly>
__global__ void __launch_bounds__(kThreads, 1)
    attention_backward_key_value_tcgen05(const __grid_constant__ CUtensorMap mapQ,
                                         const __grid_constant__ CUtensorMap mapdO,
                                         const __grid_constant__ CUtensorMap mapK,
                                         const __grid_constant__ CUtensorMap mapV, const BackwardArgs a) {
  using Cfg = KeyValueConfig<DPAD>;
  constexpr uint32_t kDB = Cfg::kBuffers;
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t total_blocks = (a.R + kTile - 1) / kTile;
  // work item -> (traversal split, head, 128-row tile of K / V); items blockIdx.x, blockIdx.x + gridDim.x, ...  `g0`
  // counts the query blocks this CTA has processed before the current item: every ring stage, TMEM region and barrier
  // phase below is a function of the global block index g = g0 + r.
  auto decode = [&](uint32_t item, uint32_t &c0, uint32_t &head, uint32_t &split, uint32_t &blk0, uint32_t &num_blocks) {
    c0 = (item % a.tiles) * kTile;
    head = (item / a.tiles) % a.batch;
    split = item / (a.tiles * a.batch);
    blk0 = split * a.blocks_per_split;  // first query block of this split (host: never empty)
    num_blocks = min(a.blocks_per_split, total_blocks - blk0);
  };
  // At D <= 64 the accumulators leave room for a THIRD 128-column region: dP^T then has a region of its own (Z) and
  // S^T / P^T / dS^T alternate between X and Y, so S^T(g+2) is issued a whole pass ahead and dP^T(g+1) in the middle of
  // pass g -- the elementwise warps never wait for the tensor pipe in steady state (they waited 24 % of the time at
  // D = 64 with two regions).  At D = 128 TMEM is full (128 + 128 + 128 + 128) and the two-region scheme above applies.
  constexpr bool kThird = DPAD <= 64;
  constexpr uint32_t kTmemX = 0, kTmemY = 128, kTmemZ = 256;
  constexpr uint32_t kTmemdV = kThird ? 384 : 256, kTmemdK = kTmemdV + DPAD, kTmemCols = 512;
  static_assert(kTmemdK + DPAD <= kTmemCols, "accumulators do not fit TMEM");

  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::kSmemBar);
  uint64_t *kv_full = bars;           // [2] K and V tiles of the item landed
  uint64_t *kv_empty = bars + 2;      // [2] every MMA of the item has completed: the buffers may be reloaded
  uint64_t *q_full = bars + 4;        // [3] Q(g) landed
  uint64_t *q_empty = bars + 7;       // [3]
  uint64_t *do_full = bars + 10;      // [2] dO(g) landed
  uint64_t *do_empty = bars + 12;     // [2]
  uint64_t *vec_full = bars + 14;     // [2] L(g), D(g) vectors in shared memory (32 arrivals)
  uint64_t *vec_empty = bars + 16;    // [2] (256 arrivals)
  uint64_t *do_ready = bars + 18;     // [2] kConvertDO: staged dO(g) rewritten as FP16 (warps 10 and 11: 64 arrivals)
  uint64_t *st_full = bars + 20;      // S^T(g) in TMEM (kThird: st_full for even g, st_full2 for odd g -- one per region)
  uint64_t *st_full2 = bars + 21;
  uint64_t *p_full = bars + 22;       // P^T(g) written (256 arrivals)
  uint64_t *acc_final = bars + 23;    // one phase per item: the item's last dK += dS^T Q has completed
  uint64_t *dpt_full = bars + 24;     // dP^T(g) in TMEM
  uint64_t *rd_free = bars + 25;      // dP^T(g) is in registers: its region may be overwritten (256 arrivals)
  uint64_t *ds_full = bars + 26;      // dS^T(g) written (256 arrivals)
  uint64_t *acc_free = bars + 27;     // one phase per item: the epilogue has read dV and dK out of TMEM (256 arrivals)
  static_assert(!(kBF16 && kConvertDO), "dO is only converted when Q, K, V are FP16");
  float *vecL = reinterpret_cast<float *>(smem + Cfg::kSmemVec);  // [stage][128]
  float *vecD = vecL + 2 * kTile;
  uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(smem + Cfg::kSmemTmemPtr);

  if (threadIdx.x == 0) {
    for (uint32_t s = 0; s < Cfg::kStagesQ; ++s) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], 1);
    }
    for (uint32_t s = 0; s < 2; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
      mbar_init(&do_full[s], 1);
      mbar_init(&do_empty[s], 1);
      mbar_init(&vec_full[s], 32);
      mbar_init(&vec_empty[s], kElemThreads);
      mbar_init(&do_ready[s], 64);
    }
    mbar_init(st_full, 1);
    mbar_init(st_full2, 1);
    mbar_init(p_full, kElemThreads);
    mbar_init(acc_final, 1);
    mbar_init(dpt_full, 1);
    mbar_init(rd_free, kElemThreads);
    mbar_init(ds_full, kElemThreads);
    mbar_init(acc_free, kElemThreads);
    fence_barrier_init();
  }
  if (warp == 8) {
    tmem_alloc(tmem_ptr_smem, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  if (a.num_splits > 1) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp < 8) {
    // ---------------- elementwise warpgroups: thread = key row, columns = queries ----------------
    setmaxnreg_inc<kElemRegs>();
    const uint32_t h = warp >> 2, quarter = warp & 3;
    const uint32_t tLane = tmem_base + ((quarter * 32) << 16);

    uint32_t g0 = 0;
    for (uint32_t item = blockIdx.x, it = 0; item < a.num_items; item += gridDim.x, ++it) {
      uint32_t c0, head, split, blk0, num_blocks;
      decode(item, c0, head, split, blk0, num_blocks);
      for (uint32_t r = 0; r < num_blocks; ++r) {
        const uint32_t g = g0 + r, stage = g & 1;
        const uint32_t rs = (g & 1) ? kTmemY : kTmemX, rd = kThird ? kTmemZ : ((g & 1) ? kTmemX : kTmemY);
        const float *Lq = vecL + stage * kTile + h * kHalf, *Dq = vecD + stage * kTile + h * kHalf;
        // ---- first half: P^T = exp2(S^T * log2e/sqrt(D) - L[q])   (+Softmax.swift:419-427) ----
        if (kThird)
          mbar_wait((g & 1) ? st_full2 : st_full, (g >> 1) & 1);  // one barrier per S^T region: two S^T can be outstanding
        else
          mbar_wait(st_full, g & 1);
        mbar_wait(&vec_full[stage], (g >> 1) & 1);
        tc_fence_after();
        float p[kHalf];
#pragma unroll
        for (uint32_t c = 0; c < kHalf; c += 32) tmem_ld32(tLane + rs + h * kHalf + c, *reinterpret_cast<uint32_t(*)[32]>(&p[c]));
        tc_wait_ld();
        // both warpgroups hold S^T(g) in registers before either overwrites the region with P^T / dS^T (warpgroup 1's
        // P^T columns [32,64) lie inside warpgroup 0's S^T columns [0,64))
        asm volatile("bar.sync 1, %0;" ::"n"(kElemThreads) : "memory");
        const uint32_t q0 = (blk0 + r) * kTile + h * kHalf;
        if (blk0 + r + 1 == total_blocks && q0 + kHalf > a.R) {  // padded query rows: P^T = 0 there
#pragma unroll
          for (uint32_t c = 0; c < kHalf; ++c)
            if (q0 + c >= a.R) p[c] = -INFINITY;
        }
#pragma unroll
        for (uint32_t c = 0; c < kHalf; c += 32) {
          uint32_t pp[16];
#pragma unroll
          for (uint32_t k = 0; k < 16; ++k) {
            exp2_pair<kPoly>(k, p[c + 2 * k], p[c + 2 * k + 1], a.scale_log2, Lq[c + 2 * k], Lq[c + 2 * k + 1]);
            pp[k] = kBF16 ? pack_bf16x2(p[c + 2 * k], p[c + 2 * k + 1]) : pack_f16x2(p[c + 2 * k], p[c + 2 * k + 1]);
          }
          tmem_st16(tLane + rs + h * (kHalf / 2) + (c >> 1), pp);  // P^T of queries [64h + c, +32) -> columns [32h + c/2, +16)
        }
        tc_wait_st();
        tc_fence_before();
        mbar_arrive(p_full);

        // ---- second half: dS^T = P^T * (dP^T/sqrt(D) - D[q]) ----
        mbar_wait(dpt_full, g & 1);
        tc_fence_after();
        uint32_t dp[kHalf];
#pragma unroll
        for (uint32_t c = 0; c < kHalf; c += 32) tmem_ld32(tLane + rd + h * kHalf + c, *reinterpret_cast<uint32_t(*)[32]>(&dp[c]));
        tc_wait_ld();
        tc_fence_before();
        mbar_arrive(rd_free);  // the dP^T region may be overwritten now
        const float2 scale2 = make_float2(a.scale, a.scale);
#pragma unroll
        for (uint32_t c = 0; c < kHalf; c += 32) {
          uint32_t dd[16];
#pragma unroll
          for (uint32_t k = 0; k < 16; ++k) {
            // (the vector loader stores -D, so the pair of D terms is one 64-bit shared-memory load and the
            // subtraction folds into the packed FMA; see backwardQuery for why packed arithmetic)
            const float2 negD2 = *reinterpret_cast<const float2 *>(&Dq[c + 2 * k]);
            const float2 t = ffma2(make_float2(__uint_as_float(dp[c + 2 * k]), __uint_as_float(dp[c + 2 * k + 1])), scale2, negD2);
            const float2 ds = fmul2(make_float2(p[c + 2 * k], p[c + 2 * k + 1]), t);
            dd[k] = kBF16 ? pack_bf16x2(ds.x, ds.y) : pack_f16x2(ds.x, ds.y);
          }
          tmem_st16(tLane + rs + kHalf + h * (kHalf / 2) + (c >> 1), dd);  // dS^T -> columns [64 + 32h + c/2, +16)
        }
        tc_wait_st();
        tc_fence_before();
        mbar_arrive(ds_full);
        mbar_arrive(&vec_empty[stage]);
      }

      // epilogue: dV, dK -> global (FP32); warpgroup h writes columns [h D/2, (h+1) D/2) of both
      mbar_wait(acc_final, it & 1);
      tc_fence_after();
      {
        float4 *scratch = reinterpret_cast<float4 *>(smem + Cfg::kSmemScratch) + warp * 256;
        const uint32_t warp_row0 = c0 + quarter * 32;
        const size_t base = split * a.split_stride + (static_cast<size_t>(head) * a.C + warp_row0) * a.D;
        store_accumulator_coalesced(tLane + kTmemdV, h * (DPAD / 2), DPAD / 2, scratch, a.dV + base, warp_row0, a.C, a.D, lane);
        store_accumulator_coalesced(tLane + kTmemdK, h * (DPAD / 2), DPAD / 2, scratch, a.dK + base, warp_row0, a.C, a.D, lane);
      }
      // the accumulators are out of TMEM: the next item's first dV / dK MMAs (accumulate off) may overwrite them
      tc_fence_before();
      mbar_arrive(acc_free);
      g0 += num_blocks;
    }  // work items
  } else {
    setmaxnreg_dec<kOtherRegs>();
    // kConvertDO: warps 10 and 11 each rewrite one half of the staged BF16 dO tile as FP16 once the TMA has landed it
    // (the tile cannot be reloaded before the MMAs that wait on do_ready have retired: do_empty)
    auto convert_dO = [&](uint32_t stage, uint32_t phase, uint32_t half) {
      mbar_wait(&do_full[stage], phase);
      uint4 *tile = reinterpret_cast<uint4 *>(smem + Cfg::kSmemdO + stage * Cfg::kTileBytes + half * (Cfg::kTileBytes / 2));
#pragma unroll 8
      for (uint32_t i = 0; i < Cfg::kTileBytes / 2 / 512; ++i) tile[i * 32 + lane] = bf16x8_to_f16x8(tile[i * 32 + lane]);
      fence_proxy_async_smem();
      mbar_arrive(&do_ready[stage]);
    };
    if (warp == 9) {
      // ---------------- TMA producer: K, V of every item, and the Q and dO rings ----------------
      uint32_t g0 = 0;
      for (uint32_t item = blockIdx.x, it = 0; item < a.num_items; item += gridDim.x, ++it) {
        uint32_t c0, head, split, blk0, num_blocks;
        decode(item, c0, head, split, blk0, num_blocks);
        const uint32_t kb = it % kDB;
        mbar_wait(&kv_empty[kb], ((it / kDB) & 1) ^ 1);  // the item that used these buffers last is done with them
        if (elect_one()) {
          mbar_arrive_expect_tx(&kv_full[kb], 2 * Cfg::kTileBytes);
#pragma unroll
          for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds) {
            tma_load_3d(smem + Cfg::kSmemK + kb * Cfg::kTileBytes + ds * kSubTileBytes, &mapK, &kv_full[kb], ds * 64, c0, head);
            tma_load_3d(smem + Cfg::kSmemV + kb * Cfg::kTileBytes + ds * kSubTileBytes, &mapV, &kv_full[kb], ds * 64, c0, head);
          }
        }
        for (uint32_t r = 0; r < num_blocks; ++r) {
          const uint32_t g = g0 + r;
          const uint32_t qs = g % Cfg::kStagesQ, qphase = (g / Cfg::kStagesQ) & 1;
          const uint32_t os = g & 1, ophase = (g >> 1) & 1;
          mbar_wait(&q_empty[qs], qphase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&q_full[qs], Cfg::kTileBytes);
#pragma unroll
            for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
              tma_load_3d(smem + Cfg::kSmemQ + qs * Cfg::kTileBytes + ds * kSubTileBytes, &mapQ, &q_full[qs], ds * 64,
                          (blk0 + r) * kTile, head);
          }
          mbar_wait(&do_empty[os], ophase ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&do_full[os], Cfg::kTileBytes);
#pragma unroll
            for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
              tma_load_3d(smem + Cfg::kSmemdO + os * Cfg::kTileBytes + ds * kSubTileBytes, &mapdO, &do_full[os], ds * 64,
                          (blk0 + r) * kTile, head);
          }
        }
        g0 += num_blocks;
      }
    } else if (warp == 10) {
      // ---------------- L / D vector loader (values are read back in their memory precision,
      //                  AttentionKernel+Softmax.swift:356-404, 453-468) ----------------
      uint32_t g0 = 0;
      for (uint32_t item = blockIdx.x; item < a.num_items; item += gridDim.x) {
        uint32_t c0, head, split, blk0, num_blocks;
        decode(item, c0, head, split, blk0, num_blocks);
        for (uint32_t r = 0; r < num_blocks; ++r) {
          const uint32_t g = g0 + r, stage = g & 1, phase = (g >> 1) & 1;
          mbar_wait(&vec_empty[stage], phase ^ 1);
#pragma unroll
          for (uint32_t i = 0; i < kTile / 32; ++i) {
            const uint32_t q = (blk0 + r) * kTile + i * 32 + lane;
            const size_t idx = static_cast<size_t>(head) * a.R + min(q, a.R - 1);
            vecL[stage * kTile + i * 32 + lane] = load_stat(a.L, idx, a.l_prec);
            vecD[stage * kTile + i * 32 + lane] = -load_stat(a.Dterm, idx, a.d_prec);  // negated: see the dS^T pass
          }
          mbar_arrive(&vec_full[stage]);  // release semantics order the shared-memory writes above
          if constexpr (kConvertDO) convert_dO(stage, phase, 0);
        }
        g0 += num_blocks;
      }
    } else if (warp == 11) {
      if constexpr (kConvertDO) {
        uint32_t g0 = 0;
        for (uint32_t item = blockIdx.x; item < a.num_items; item += gridDim.x) {
          uint32_t c0, head, split, blk0, num_blocks;
          decode(item, c0, head, split, blk0, num_blocks);
          for (uint32_t r = 0; r < num_blocks; ++r) convert_dO((g0 + r) & 1, ((g0 + r) >> 1) & 1, 1);
          g0 += num_blocks;
        }
      }
    } else if (warp == 8) {
      // ---------------- MMA issuer ----------------
      constexpr uint32_t kFormat = kBF16 ? 1u : 0u;
      constexpr uint32_t idescNT = make_idesc_f16(kTile, kTile, kFormat, 0, 0);
      constexpr uint32_t idescAcc = make_idesc_f16(kTile, DPAD, kFormat, 0, 1);
      const uint64_t descK0 = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemK), 16, 1024);
      const uint64_t descV0 = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemV), 16, 1024);
      const uint64_t descQ = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemQ), 16, 1024);
      const uint64_t descdO = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemdO), 16, 1024);
      const uint64_t descQmn = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemQ), kSubTileBytes, 1024);
      const uint64_t descdOmn = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemdO), kSubTileBytes, 1024);

      auto issue_nt = [&](uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc) {
#pragma unroll
        for (uint32_t k = 0; k < DPAD / 16; ++k) {
          const uint32_t off = ((k >> 2) * kSubTileBytes + (k & 3) * 32) >> 4;
          umma_ss(d_tmem, a_desc + off, b_desc + off, idescNT, k > 0);
        }
      };
      // A = 128 queries (K) of 16-bit values in 64 consecutive TMEM columns starting at a_base
      auto issue_acc = [&](uint32_t d_tmem, uint32_t a_base, uint64_t b_desc, uint32_t accumulate) {
#pragma unroll
        for (uint32_t k = 0; k < kTile / 16; ++k)
          umma_ts(d_tmem, a_base + k * 8, b_desc + ((k * 2048) >> 4), idescAcc, k > 0 ? 1u : accumulate);
      };
      auto q_at = [&](uint32_t g) { return descQ + (((g % Cfg::kStagesQ) * Cfg::kTileBytes) >> 4); };
      auto do_at = [&](uint32_t g) { return descdO + (((g & 1) * Cfg::kTileBytes) >> 4); };
      auto region = [&](uint32_t g) { return tmem_base + ((g & 1) ? kTmemY : kTmemX); };

      uint32_t g0 = 0;
      for (uint32_t item = blockIdx.x, it = 0; item < a.num_items; item += gridDim.x, ++it) {
        uint32_t c0, head, split, blk0, num_blocks;
        decode(item, c0, head, split, blk0, num_blocks);
        const uint32_t kb = it % kDB;
        const uint64_t descK = descK0 + ((kb * Cfg::kTileBytes) >> 4), descV = descV0 + ((kb * Cfg::kTileBytes) >> 4);

        // prologue: S^T(g0) and dP^T(g0) (and S^T(g0 + 1) with three regions).  For every item but the first they are
        // issued while the elementwise warps are still storing the previous item's dV / dK: the S^T regions' last readers
        // (dK of the previous item's last two blocks) are ahead on the in-order tensor pipe, the dP^T region only needs
        // the previous item's last dP^T to have been read out (rd_free).
        mbar_wait(&kv_full[kb], (it / kDB) & 1);
        mbar_wait(&q_full[g0 % Cfg::kStagesQ], (g0 / Cfg::kStagesQ) & 1);
        tc_fence_after();
        if (elect_one()) {
          issue_nt(region(g0), descK, q_at(g0));  // S^T = K Q^T
          umma_commit(kThird && (g0 & 1) ? st_full2 : st_full);
        }
        __syncwarp();
        mbar_wait(&do_full[g0 & 1], (g0 >> 1) & 1);
        if constexpr (kConvertDO) mbar_wait(&do_ready[g0 & 1], (g0 >> 1) & 1);
        if (it > 0) mbar_wait(rd_free, (g0 - 1) & 1);
        tc_fence_after();
        if (elect_one()) {
          issue_nt(kThird ? tmem_base + kTmemZ : region(g0 + 1), descV, do_at(g0));  // dP^T = V dO^T
          umma_commit(dpt_full);
        }
        __syncwarp();

        if constexpr (kThird) {
          // three regions: S^T(g0 + 1) straight away, then per block  dV(g) -> dP^T(g+1) -> dK(g) -> S^T(g+2)
          if (num_blocks > 1) {
            mbar_wait(&q_full[(g0 + 1) % Cfg::kStagesQ], ((g0 + 1) / Cfg::kStagesQ) & 1);
            tc_fence_after();
            if (elect_one()) {
              issue_nt(region(g0 + 1), descK, q_at(g0 + 1));
              umma_commit(((g0 + 1) & 1) ? st_full2 : st_full);
            }
            __syncwarp();
          }
          for (uint32_t r = 0; r < num_blocks; ++r) {
            const uint32_t g = g0 + r;
            // (a) dV += P^T(g) dO(g); dO(g) is done with after this
            mbar_wait(p_full, g & 1);
            if (r == 0) mbar_wait(acc_free, (it & 1) ^ 1);  // the previous item's epilogue has read the accumulators out
            tc_fence_after();
            if (elect_one()) {
              issue_acc(tmem_base + kTmemdV, region(g), descdOmn + (((g & 1) * Cfg::kTileBytes) >> 4), r > 0 ? 1u : 0u);
              umma_commit(&do_empty[g & 1]);
            }
            __syncwarp();
            // (b) dP^T(g+1) = V dO(g+1)^T into Z as soon as dP^T(g) has been read out of it
            if (r + 1 < num_blocks) {
              mbar_wait(rd_free, g & 1);
              mbar_wait(&do_full[(g + 1) & 1], ((g + 1) >> 1) & 1);
              if constexpr (kConvertDO) mbar_wait(&do_ready[(g + 1) & 1], ((g + 1) >> 1) & 1);
              tc_fence_after();
              if (elect_one()) {
                issue_nt(tmem_base + kTmemZ, descV, do_at(g + 1));
                umma_commit(dpt_full);
              }
              __syncwarp();
            }
            // (c) dK += dS^T(g) Q(g); Q(g) is done with after this
            mbar_wait(ds_full, g & 1);
            tc_fence_after();
            if (elect_one()) {
              issue_acc(tmem_base + kTmemdK, region(g) + kHalf, descQmn + (((g % Cfg::kStagesQ) * Cfg::kTileBytes) >> 4),
                        r > 0 ? 1u : 0u);
              umma_commit(&q_empty[g % Cfg::kStagesQ]);
              if (r + 1 == num_blocks) {
                umma_commit(acc_final);
                umma_commit(&kv_empty[kb]);
              }
            }
            __syncwarp();
            // (d) S^T(g+2) = K Q(g+2)^T into the region P^T(g) / dS^T(g) occupied (in-order pipe: after dV(g), dK(g))
            if (r + 2 < num_blocks) {
              mbar_wait(&q_full[(g + 2) % Cfg::kStagesQ], ((g + 2) / Cfg::kStagesQ) & 1);
              tc_fence_after();
              if (elect_one()) {
                issue_nt(region(g), descK, q_at(g + 2));
                umma_commit((g & 1) ? st_full2 : st_full);
              }
              __syncwarp();
            }
          }
        } else {
          for (uint32_t r = 0; r < num_blocks; ++r) {
            const uint32_t g = g0 + r;
            const bool has_next = r + 1 < num_blocks;
            // (a) dV += P^T(g) dO(g); dO(g) is done with after this
            mbar_wait(p_full, g & 1);
            if (r == 0) mbar_wait(acc_free, (it & 1) ^ 1);
            tc_fence_after();
            if (elect_one()) {
              issue_acc(tmem_base + kTmemdV, region(g), descdOmn + (((g & 1) * Cfg::kTileBytes) >> 4), r > 0 ? 1u : 0u);
              umma_commit(&do_empty[g & 1]);
            }
            __syncwarp();
            // (b) S^T(g+1) = K Q(g+1)^T into the region dP^T(g) has just been read out of
            if (has_next) {
              mbar_wait(rd_free, g & 1);
              mbar_wait(&q_full[(g + 1) % Cfg::kStagesQ], ((g + 1) / Cfg::kStagesQ) & 1);
              tc_fence_after();
              if (elect_one()) {
                issue_nt(region(g + 1), descK, q_at(g + 1));
                umma_commit(st_full);
              }
              __syncwarp();
            }
            // (c) dK += dS^T(g) Q(g); Q(g) is done with after this
            mbar_wait(ds_full, g & 1);
            tc_fence_after();
            if (elect_one()) {
              issue_acc(tmem_base + kTmemdK, region(g) + kHalf, descQmn + (((g % Cfg::kStagesQ) * Cfg::kTileBytes) >> 4),
                        r > 0 ? 1u : 0u);
              umma_commit(&q_empty[g % Cfg::kStagesQ]);
              if (!has_next) {
                umma_commit(acc_final);
                umma_commit(&kv_empty[kb]);
              }
            }
            __syncwarp();
            // (d) dP^T(g+1) = V dO(g+1)^T into the region P^T(g) / dS^T(g) occupied (in-order pipe: after dV(g), dK(g))
            if (has_next) {
              mbar_wait(&do_full[(g + 1) & 1], ((g + 1) >> 1) & 1);
              if constexpr (kConvertDO) mbar_wait(&do_ready[(g + 1) & 1], ((g + 1) >> 1) & 1);
              tc_fence_after();
              if (elect_one()) {
                issue_nt(region(g), descV, do_at(g + 1));
                umma_commit(dpt_full);
              }
              __syncwarp();
            }
          }
        }
        g0 += num_blocks;
      }  // work items
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

template <uint32_t DPAD, bool kBF16, bool kConvertDO, uint32_t kPoly>
cudaError_t launch(const AttentionParams &p, cudaStream_t stream, bool key_value) {
  auto kernel_q = attention_backward_query_tcgen05<DPAD, kBF16, kConvertDO, kPoly, false>;
  auto kernel_kv = attention_backward_key_value_tcgen05<DPAD, kBF16, kConvertDO, kPoly>;
  size_t smem_q = QueryConfig<DPAD, false>::kSmemBytes;
  const int device = current_device();
  cudaError_t e;

  // parallelised dimension -> CTAs; traversed dimension -> blocks, possibly split over blockIdx.z
  const uint32_t par = key_value ? p.C : p.R, trav = key_value ? p.R : p.C;
  const uint32_t tiles = (par + kTile - 1) / kTile, total_blocks = (trav + kTile - 1) / kTile;
  const uint32_t per = choose_blocks_per_split(tiles * p.batch, total_blocks, device_sm_count(device), p.split_min_blocks, p.split_max);
  const uint32_t splits = (total_blocks + per - 1) / per;
  // D-term of the persistent dQ kernel (D <= 64): computed one item ahead by warp 11 (kOffload) or by the elementwise
  // warps at the head of every item.  A/B on one box (profiles/r2_sweep_dq_dterm*.jsonl, TFLOP/s, offload | inline): N=512
  // 580 | 473, N=1024 750 | 670, N=2048 880 | 840 (reference policy 900 | 834), N=4096 915 | 955, N=8192 975 | 1030: the
  // head of an item that the offload removes matters for short items; the 48 KB staging area it needs costs long items ~4 %
  // (also with the offload switched off at run time, and with no-allocate loads: it is the shared-memory footprint, 225
  // instead of 177 KB), so the two forms are separate instantiations and long items take the inline one.
  if constexpr (QueryConfig<DPAD>::kPersistent) {
    if (!key_value && per <= 24) {
      kernel_q = attention_backward_query_tcgen05<DPAD, kBF16, kConvertDO, kPoly, true>;
      smem_q = QueryConfig<DPAD, true>::kSmemBytes;
    }
  }
  if (!key_value)
    e = ensure_max_dynamic_smem(reinterpret_cast<const void *>(kernel_q), smem_q, device);
  else
    e = ensure_max_dynamic_smem(reinterpret_cast<const void *>(kernel_kv), KeyValueConfig<DPAD>::kSmemBytes, device);
  if (e != cudaSuccess) return e;

  CUtensorMap mapQ, mapdO, mapK, mapV;
  if ((e = make_tensor_map_16bit(&mapQ, p.buf[sQ], p.R, p.D, p.batch, kTile)) != cudaSuccess) return e;
  if ((e = make_tensor_map_16bit(&mapdO, p.buf[sdO], p.R, p.D, p.batch, kTile)) != cudaSuccess) return e;
  if ((e = make_tensor_map_16bit(&mapK, p.buf[sK], p.C, p.D, p.batch, kTile)) != cudaSuccess) return e;
  if ((e = make_tensor_map_16bit(&mapV, p.buf[sV], p.C, p.D, p.batch, kTile)) != cudaSuccess) return e;

  BackwardArgs a;
  a.dO = p.buf[sdO];
  a.O = static_cast<const float *>(p.buf[sO]);
  a.L = p.buf[sL];
  a.Dterm = p.buf[sD];
  a.dQ = static_cast<float *>(p.buf[sdQ]);
  a.dV = static_cast<float *>(p.buf[sdV]);
  a.dK = static_cast<float *>(p.buf[sdK]);
  a.R = p.R;
  a.C = p.C;
  a.D = p.D;
  a.scale = p.scale;
  a.scale_log2 = p.scale_log2;
  a.l_prec = p.prec[sL];
  a.d_prec = p.prec[sD];

  a.blocks_per_split = per;
  a.split_stride = 0;
  a.tiles = tiles;
  a.batch = p.batch;
  a.num_splits = splits;
  a.num_items = tiles * p.batch * splits;
  // both kernels walk work items (split, head, tile): persistent CTAs, one per SM, where the kernel can overlap
  // consecutive items (D <= 64); otherwise one CTA per item
  const uint32_t sm_count = device_sm_count(device);
  const dim3 grid_q(QueryConfig<DPAD>::kPersistent && a.num_items > sm_count ? sm_count : a.num_items, 1, 1);
  const dim3 grid = grid_q;
  static_assert(QueryConfig<DPAD>::kPersistent == KeyValueConfig<DPAD>::kPersistent, "one grid rule for both kernels");
  const size_t smem = key_value ? KeyValueConfig<DPAD>::kSmemBytes : smem_q;
  if (splits == 1) {
    if (!key_value)
      kernel_q<<<grid_q, kThreads, smem, stream>>>(mapQ, mapdO, mapK, mapV, a);
    else
      kernel_kv<<<grid, kThreads, smem, stream>>>(mapQ, mapdO, mapK, mapV, a);
    return cudaGetLastError();
  }

  // partial accumulators in the library's per-(device, stream) workspace: [split][tensor][batch][rows][D] FP32,
  // tensor = dQ | (dV, dK)
  const size_t tensor_elems = static_cast<size_t>(p.batch) * par * p.D;
  const uint32_t tensors = key_value ? 2 : 1;
  void *ws = nullptr;
  if ((e = workspace_for(device, stream, splits * tensors * tensor_elems * sizeof(float), &ws)) != cudaSuccess) return e;
  float *scratch = static_cast<float *>(ws);
  a.split_stride = tensors * tensor_elems;
  a.dQ = scratch;
  a.dV = scratch;
  a.dK = scratch + tensor_elems;
  if (!key_value)
    kernel_q<<<grid_q, kThreads, smem, stream>>>(mapQ, mapdO, mapK, mapV, a);
  else
    kernel_kv<<<grid, kThreads, smem, stream>>>(mapQ, mapdO, mapK, mapV, a);
  e = cudaGetLastError();
  if (e == cudaSuccess)
    e = launch_sum_splits(scratch, static_cast<float *>(key_value ? p.buf[sdV] : p.buf[sdQ]),
                          static_cast<float *>(key_value ? p.buf[sdK] : p.buf[sdQ]), tensor_elems, tensors, a.split_stride,
                          splits, stream);
  return e;
}

}  // namespace bwd

uint32_t tcgen05_backward_max_head() { return 256; }  // (128, 256]: tcgen05_backward_generic.cu

bool tcgen05_backward_supported(const AttentionParams &p) {
  // dO: the element type of Q/K/V, or BF16 beside FP16 Q/K/V (the reference's policy; converted on chip)
  const bool dO_ok = p.prec[sdO] == p.prec[sQ] || (p.prec[sQ] == FP16 && p.prec[sdO] == BF16);
  const bool types = (p.prec[sQ] == FP16 || p.prec[sQ] == BF16) && p.prec[sK] == p.prec[sQ] &&
                     p.prec[sV] == p.prec[sQ] && dO_ok && p.prec[sO] == FP32 &&
                     p.prec[sdQ] == FP32 && p.prec[sdK] == FP32 && p.prec[sdV] == FP32;
  // derived operands follow their primal (dO ~ O, dQ ~ Q, dK ~ K, dV ~ V: AttentionKernel.swift:189-195)
  const bool layout = tcgen05_backward_transposes_ok(p.R, p.C, p.transposed[sQ] || p.transposed[sdQ], p.transposed[sK] || p.transposed[sdK],
                                                     p.transposed[sV] || p.transposed[sdV], p.transposed[sO] || p.transposed[sdO]);
  return types && layout && p.D % 8 == 0 && p.D <= tcgen05_backward_max_head();
}

// dK/dV, FP16 Q/K/V beside BF16 dO: convert dO in a pass of its own when the key tiles fill more than one wave of SMs
bool tcgen05_backward_converts_dO_first(uint32_t C, uint32_t batch) {
  const uint64_t tiles = static_cast<uint64_t>((C + bwd::kTile - 1) / bwd::kTile) * batch;
  return tiles > static_cast<uint64_t>(device_sm_count(current_device()));
}

cudaError_t launch_tcgen05_backward(const AttentionParams &p, cudaStream_t stream, bool key_value) {
  const bool bf16 = p.prec[sQ] == BF16;
  const bool convert = p.prec[sdO] != p.prec[sQ];  // FP16 Q/K/V with BF16 dO
  // dK/dV with the reference's policy: every streamed dO block has to be rewritten as FP16 by two helper warps before
  // dP^T = V dO^T may start -- 15 % at config 3 (N = 2048, D = 64: 802 against 941 TFLOP/s all-FP16).  When the grid is
  // more than one wave, dO is converted ONCE into the workspace instead (O(N D), ~3 % of the kernel) and the all-FP16
  // instantiation runs; small grids (latency-bound, an extra launch costs more than it saves) keep the in-kernel rewrite,
  // as does dQ, whose resident dO tile is rewritten once per item by all eight elementwise warps (2 %).
  if (convert && key_value && tcgen05_backward_converts_dO_first(p.C, p.batch)) {
    AttentionParams q = p;
    const uint64_t elements = static_cast<uint64_t>(p.batch) * p.R * p.D;
    void *ws = nullptr;
    cudaError_t e = workspace_for(current_device(), stream, elements * 2, &ws, /*slot=*/2);
    if (e != cudaSuccess) return e;
    if ((e = launch_bf16_to_f16(p.buf[sdO], ws, elements, stream)) != cudaSuccess) return e;
    q.buf[sdO] = ws;
    q.prec[sdO] = q.prec[sQ];
    return launch_tcgen05_backward(q, stream, key_value);
  }
  // the row's exp2 column selects the instantiation (kernel creation has checked the range)
#define MFA_BWD_MODES(DPAD_, POLY_)                                                          \
  if (convert) return bwd::launch<DPAD_, false, true, POLY_>(p, stream, key_value);         \
  return bf16 ? bwd::launch<DPAD_, true, false, POLY_>(p, stream, key_value)                 \
              : bwd::launch<DPAD_, false, false, POLY_>(p, stream, key_value);
#define MFA_BWD_DISPATCH(DPAD_)                \
  switch (p.exp2_fma_quarters) {               \
    case 0: { MFA_BWD_MODES(DPAD_, 0) }        \
    case 1: { MFA_BWD_MODES(DPAD_, 1) }        \
    case 2: { MFA_BWD_MODES(DPAD_, 2) }        \
    default: { MFA_BWD_MODES(DPAD_, 3) }       \
  }
  if (p.D <= 64) {
    MFA_BWD_DISPATCH(64)
  }
  MFA_BWD_DISPATCH(128)
#undef MFA_BWD_DISPATCH
#undef MFA_BWD_MODES
}

// 1 launch, or 2 (kernel + sum_splits) when the traversal split engages for this problem size
uint32_t tcgen05_backward_launch_count(int type, uint32_t R, uint32_t C, uint32_t batch, uint32_t min_blocks,
                                       uint32_t max_splits, bool convert_dO) {
  const bool key_value = type == 2;  // MFA_BACKWARD_KEY_VALUE
  const uint32_t par = key_value ? C : R, trav = key_value ? R : C;
  const uint32_t tiles = (par + bwd::kTile - 1) / bwd::kTile, total_blocks = (trav + bwd::kTile - 1) / bwd::kTile;
  const uint32_t extra = (key_value && convert_dO && tcgen05_backward_converts_dO_first(C, batch)) ? 1 : 0;
  return extra + (bwd::choose_blocks_per_split(tiles * batch, total_blocks, device_sm_count(current_device()), min_blocks, max_splits) < total_blocks ? 2 : 1);
}

void tcgen05_backward_geometry(int type, uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par,
                               uint32_t *trav, uint32_t *head) {
  *threads = bwd::kThreads;
  if (type == 1)  // MFA_BACKWARD_QUERY
    *smem_bytes = D <= 64 ? bwd::QueryConfig<64, true>::kSmemBytes  // (the larger of its two forms)
                          : bwd::QueryConfig<128>::kSmemBytes;
  else
    *smem_bytes = D <= 64 ? bwd::KeyValueConfig<64>::kSmemBytes : bwd::KeyValueConfig<128>::kSmemBytes;
  *par = bwd::kTile;
  *trav = bwd::kTile;
  *head = D <= 64 ? 64 : 128;
  const uint32_t padded = (D + 7) / 8 * 8;
  if (*head > padded) *head = padded;
}

}  // namespace mfa

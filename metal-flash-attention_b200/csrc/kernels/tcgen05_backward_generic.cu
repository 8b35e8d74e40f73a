// FlashAttention backward for sm_100a, the layout-generic / wide-head kernels: head dimensions 128 < D <= 256 and
// TRANSPOSED operands (stored [D][seq], AttentionKernel.swift:189-195) at any D <= 256, D % 8 == 0.  The reference serves
// these cases by blocking the head dimension and spilling the accumulators (AttentionDescriptor+Parameters.swift:182-285,
// the rows past D = 128; loopBackwardQuery / loopBackwardKeyValue, AttentionKernel+Source.swift:202-293); on B200 the
// limits are 512 TMEM columns and 227 KB of shared memory, and they force these changes against tcgen05_backward.cu:
//
//   * the traversed operands come in blocks of 64 rows, not 128 (a 128 x 256 16-bit tile is 64 KB; two resident tiles
//     plus a ring of 128-row blocks do not fit).  The S / dP MMAs are then M128 x N64, which the tensor pipe runs at
//     the N = 128 cost (64 cycles per k-step): these kernels top out near 60 % of the MMA peak by construction;
//   * at D > 128, dK and dV together would need 512 accumulator columns, leaving none for S^T / dP^T: backwardKeyValue runs
//     as TWO passes over the query blocks -- a dV pass (S^T -> P^T -> dV += P^T dO) and a dK pass (S^T, dP^T -> dS^T ->
//     dK += dS^T Q) -- one accumulator each.  S^T is computed twice: 5 GEMMs instead of 4;
//   * all passes are ONE kernel template.  With (A1, A2) the resident 128-row tiles and (B1, B2) the streamed
//     64-row blocks:
//         kQuery   A1 = Q, A2 = dO, B1 = K, B2 = V      S  = A1 B1^T, dP  = A2 B2^T, dQ += dS B1
//         kKey     A1 = K, A2 = V,  B1 = Q, B2 = dO     S^T = A1 B1^T, dP^T = A2 B2^T, dK += dS^T B1
//         kValue   A1 = K,          B1 = Q, B2 = dO     S^T = A1 B1^T,                 dV += P^T B2
//         kKeyValue (D <= 128, where dK and dV fit TMEM side by side: 256 + 2 D <= 512): kKey plus dV += P^T B2 -- one
//                  pass, four GEMMs; P^T is written over S^T and dS^T over dP^T, both A operands live in TMEM at once
//     L and D are per ROW in kQuery (registers; D is computed here, computeD +Softmax.swift:32-221) and per COLUMN in
//     the others (64-entry vectors staged in shared memory one block ahead).
//
// A transposed operand is fetched through a tensor map of the transposed view and consumed through the other UMMA
// major-ness (K-major <-> MN-major), exactly as in the layout-generic forward kernel (tcgen05_forward_d256.cu); a
// transposed output is stored straight from registers (a warp's 32 rows are contiguous in memory then).
//
// TMEM: S double buffer [0,128) (2 x 64 columns), dP double buffer [128,256), accumulator [256, 256 + DPAD) (kKeyValue: dK
// there, dV behind it).  P / dS
// (16-bit) overwrite S / dP in place and feed the accumulate MMA from TMEM.  Warps 0-7: elementwise (thread = TMEM lane
// x 32 of the block's 64 columns), warp 8: MMA issuer, warp 9: TMA producer for the resident tiles and ring 1, warp 10:
// TMA producer for ring 2.  (The reference's FP16 + BF16-dO policy: the host converts dO once, see the launcher.)
// Tensor-pipe order per block j:  dP(j+1) -> S(j+1) -> acc(j): the elementwise pass of block j runs under the first two.
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
namespace bwdg {

using namespace ptx;
using bwd::load_16bit;
using bwd::load_stat;
using bwd::store_stat;

constexpr uint32_t kTile = 128;   // rows of the parallelised operand per CTA
constexpr uint32_t kBlock = 64;   // rows of the traversed operands per block
constexpr uint32_t kCols = 32;    // block columns per elementwise thread
constexpr uint32_t kThreads = 384, kElemThreads = 256;
constexpr uint32_t kLaunchRegs = 168, kElemRegs = 208, kOtherRegs = 88;
static_assert(kElemRegs * 256 + kOtherRegs * 128 <= kLaunchRegs * kThreads, "setmaxnreg over-subscribed");
enum Mode : uint32_t { kQuery = 0, kKey = 1, kValue = 2, kKeyValue = 3 };

// tmask bits
constexpr uint32_t kTransA1 = 1, kTransA2 = 2, kTransB1 = 4, kTransB2 = 8, kTransOut = 16, kTransO = 32, kTransdO = 64,
                   kTransOut2 = 128;

struct GenericArgs {
  const void *dO;   // global dO (kQuery: for D = rowsum(dO * O))
  const float *O;   // global O (kQuery)
  const void *L;    // [batch][R]
  void *Dterm;      // [batch][R]: written by kQuery, read by kKey
  float *out;       // dQ | dK | dV (FP32)
  float *out2;      // kKeyValue: dV (out = dK)
  uint32_t R, C, D;
  float scale, scale_log2;
  int l_prec, d_prec;
  uint32_t blocks_per_split;  // traversal split, in 64-row blocks
  size_t split_stride;        // floats between split slices of `out` (0: no split)
  uint32_t tiles, batch, num_splits, num_items;
  uint32_t tmask;
};

template <uint32_t DPAD, uint32_t kMode>
struct Config {
  static constexpr uint32_t kResidents = kMode == kValue ? 1 : 2;
  static constexpr uint32_t kResBytes = DPAD * 256;  // 128 x DPAD 16-bit
  static constexpr uint32_t kBlkBytes = DPAD * 128;  // 64 x DPAD 16-bit
  // ring 1 = the S operand (and, kQuery / kKey, the accumulate operand: alive from S(j) to acc(j)); ring 2 = the dP
  // operand, or kValue's accumulate operand.  D = 256, kQuery / kKey: 2 x 64 + 2 x 32 + 32 = 224 KB.
  static constexpr uint32_t kStages1 = 2;
  static constexpr uint32_t kStages2 = (kMode == kValue || DPAD <= 128) ? 2 : 1;
  static_assert(kMode != kKeyValue || DPAD <= 128, "dK and dV do not fit TMEM beside S^T / dP^T");
  static constexpr uint32_t kSmemRes = 0;
  static constexpr uint32_t kSmemRing1 = kResidents * kResBytes;
  static constexpr uint32_t kSmemRing2 = kSmemRing1 + kStages1 * kBlkBytes;
  static constexpr uint32_t kSmemScratch = kSmemRing1;  // epilogue: 8 warps x 4 KB over the dead rings
  static constexpr uint32_t kSmemVec = kSmemRing2 + kStages2 * kBlkBytes;  // 256 floats
  static constexpr uint32_t kSmemBar = kSmemVec + 1024;
  static constexpr uint32_t kNumBars = 24;
  static constexpr uint32_t kSmemTmemPtr = kSmemBar + kNumBars * 8;
  static constexpr uint32_t kSmemBytes = kSmemTmemPtr + 16;
  static_assert(kSmemBytes <= 232448, "shared memory over budget");
  static_assert(8 * 4096 <= (kStages1 + kStages2) * kBlkBytes, "epilogue scratch does not fit the rings");
  static constexpr uint32_t kTmemS = 0, kTmemdP = 128, kTmemAcc = 256, kTmemAcc2 = 256 + DPAD, kTmemCols = 512;
  static_assert(kTmemAcc + (kMode == kKeyValue ? 2 : 1) * DPAD <= kTmemCols, "accumulators do not fit TMEM");
};

template <uint32_t DPAD, bool kBF16, uint32_t kMode>
__global__ void __launch_bounds__(kThreads, 1)
    attention_backward_generic_tcgen05(const __grid_constant__ CUtensorMap mapA1, const __grid_constant__ CUtensorMap mapA2,
                                       const __grid_constant__ CUtensorMap mapB1, const __grid_constant__ CUtensorMap mapB2,
                                       const GenericArgs a) {
  using Cfg = Config<DPAD, kMode>;
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t par_len = kMode == kQuery ? a.R : a.C, trav_len = kMode == kQuery ? a.C : a.R;
  const uint32_t total_blocks = (trav_len + kBlock - 1) / kBlock;
  const bool tA1 = a.tmask & kTransA1, tA2 = a.tmask & kTransA2, tB1 = a.tmask & kTransB1, tB2 = a.tmask & kTransB2;

  // work item (one per CTA) -> (traversal split, head, 128-row tile)
  const uint32_t item = blockIdx.x;
  const uint32_t p0 = (item % a.tiles) * kTile;
  const uint32_t head = (item / a.tiles) % a.batch;
  const uint32_t split = item / (a.tiles * a.batch);
  const uint32_t blk0 = split * a.blocks_per_split;
  const uint32_t num_blocks = min(a.blocks_per_split, total_blocks - blk0);

  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::kSmemBar);
  uint64_t *res_full = bars;          // resident tiles landed
  uint64_t *r1_full = bars + 1;       // [2]
  uint64_t *r1_empty = bars + 3;      // [2]
  uint64_t *r2_full = bars + 5;       // [2]
  uint64_t *r2_empty = bars + 7;      // [2]
  uint64_t *s_full = bars + 9;        // [2] S(j) in TMEM
  uint64_t *s_free = bars + 11;       // [2] S(j) is in registers (256 arrivals; kQuery / kKey)
  uint64_t *dp_full = bars + 13;      // [2] dP(j) in TMEM
  uint64_t *ds_full = bars + 15;      // [2] dS(j) -- kValue: P(j) -- written (256 arrivals)
  uint64_t *acc_final = bars + 17;    // the last accumulate MMA has completed
  uint64_t *p_full = bars + 18;       // [2] kKeyValue: P(j) written over S(j) (256 arrivals)
  constexpr bool kDOisBF16 = kBF16;  // dO has the element type of Q, K, V here (the host converts a BF16 dO beside FP16 inputs)
  uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(smem + Cfg::kSmemTmemPtr);

  if (threadIdx.x == 0) {
    mbar_init(res_full, 1);
    for (uint32_t s = 0; s < 2; ++s) {
      mbar_init(&r1_full[s], 1);
      mbar_init(&r1_empty[s], 1);
      mbar_init(&r2_full[s], 1);
      mbar_init(&r2_empty[s], 1);
      mbar_init(&s_full[s], 1);
      mbar_init(&s_free[s], kElemThreads);
      mbar_init(&dp_full[s], 1);
      mbar_init(&ds_full[s], kElemThreads);
      mbar_init(&p_full[s], kElemThreads);
    }
    mbar_init(acc_final, 1);
    fence_barrier_init();
  }
  if (warp == 8) {
    tmem_alloc(tmem_ptr_smem, Cfg::kTmemCols);
    tmem_relinquish();
  }
  if (warp == 9 && lane == 0) {
    prefetch_tensormap(&mapA1);
    prefetch_tensormap(&mapB1);
    prefetch_tensormap(&mapB2);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;
  if (a.num_splits > 1) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp < 8) {
    // ---------------- elementwise warps ----------------
    setmaxnreg_inc<kElemRegs>();
    const uint32_t h = warp >> 2, quarter = warp & 3;
    const uint32_t row_in_tile = quarter * 32 + lane;
    const uint32_t tLane = tmem_base + ((quarter * 32) << 16);
    const uint32_t row = p0 + row_in_tile;
    float *vec = reinterpret_cast<float *>(smem + Cfg::kSmemVec);
    float Lrow = 0.f, Dterm = 0.f;

    // statistics of traversal block `blk` for this thread's slot of the staging vector: [0,64) L, [64,128) D
    auto load_column_stat = [&](uint32_t blk) -> float {
      const uint32_t t = threadIdx.x, q = blk * kBlock + (t & 63);
      if (t < 64) return q < a.R ? load_stat(a.L, static_cast<size_t>(head) * a.R + q, a.l_prec) : INFINITY;  // P = 0 there
      if ((kMode == kKey || kMode == kKeyValue) && q < a.R) return load_stat(a.Dterm, static_cast<size_t>(head) * a.R + q, a.d_prec);
      return 0.f;
    };

    if constexpr (kMode == kQuery) {
      // computeD: D = (sum_d dO * O) / sqrt(D)
      if ((a.tmask & (kTransO | kTransdO)) == 0) {
        // row-major: each warp takes 16 rows and spreads the columns over its lanes (full cache lines per load)
        // (eight rows in flight at a time: sixteen would not fit the 168 registers ptxas allocates against)
        constexpr uint32_t kRowsPerWarp = kTile / 8, kBatch = 8;
#pragma unroll 1
        for (uint32_t r8 = 0; r8 < kRowsPerWarp; r8 += kBatch) {
          float acc[kBatch];
#pragma unroll
          for (uint32_t i = 0; i < kBatch; ++i) acc[i] = 0.f;
          for (uint32_t cb = 0; cb < a.D; cb += 128) {
            const bool active = cb + 4 * lane < a.D;
            float4 o4[kBatch];
            uint2 g4[kBatch];
#pragma unroll
            for (uint32_t i = 0; i < kBatch; ++i) {
              const uint32_t rr = min(p0 + warp * kRowsPerWarp + r8 + i, a.R - 1);
              const size_t base = (static_cast<size_t>(head) * a.R + rr) * a.D + cb + 4 * lane;
              o4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
              g4[i] = make_uint2(0u, 0u);
              if (active) {
                o4[i] = ldg_stream_f32x4(a.O + base);
                g4[i] = ldg_stream_u32x2(static_cast<const uint16_t *>(a.dO) + base);
              }
            }
#pragma unroll
            for (uint32_t i = 0; i < kBatch; ++i) {
              const float2 lo = kDOisBF16 ? unpack_bf16x2(g4[i].x) : unpack_f16x2(g4[i].x);
              const float2 hi = kDOisBF16 ? unpack_bf16x2(g4[i].y) : unpack_f16x2(g4[i].y);
              acc[i] += fmaf(lo.x, o4[i].x, fmaf(lo.y, o4[i].y, fmaf(hi.x, o4[i].z, hi.y * o4[i].w)));
            }
          }
#pragma unroll
          for (uint32_t i = 0; i < kBatch; ++i) {
            float v = acc[i];
#pragma unroll
            for (uint32_t off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            if (lane == i) vec[warp * kRowsPerWarp + r8 + i] = v * a.scale;
          }
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kElemThreads) : "memory");
        Dterm = vec[row_in_tile];
      } else {
        // a transposed O or dO: thread = (row, half of the head dimension); along a transposed operand a warp's 32 rows
        // are contiguous
        const uint32_t rc = min(row, a.R - 1), d0 = h * (a.D / 2), d1 = d0 + a.D / 2;
        const size_t hb = static_cast<size_t>(head) * a.R * a.D;
        // four columns (D % 8 == 0: D / 2 is a multiple of 4) x two unrolled steps: sixteen loads in flight per thread -- one
        // load at a time made this loop a fifth of the kernel (64 dependent round trips to memory at D = 128)
        const bool tO = a.tmask & kTransO, tG = a.tmask & kTransdO;
        float part = 0.f;
#pragma unroll 2
        for (uint32_t d = d0; d < d1; d += 4) {
          float o[4], g[4];
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k) {
            const size_t io = tO ? static_cast<size_t>(d + k) * a.R + rc : static_cast<size_t>(rc) * a.D + d + k;
            const size_t ig = tG ? static_cast<size_t>(d + k) * a.R + rc : static_cast<size_t>(rc) * a.D + d + k;
            o[k] = __ldg(a.O + hb + io);
            g[k] = load_16bit(a.dO, hb + ig, kDOisBF16);
          }
#pragma unroll
          for (uint32_t k = 0; k < 4; ++k) part = fmaf(o[k], g[k], part);
        }
        vec[h * kTile + row_in_tile] = part;
        asm volatile("bar.sync 1, %0;" ::"n"(kElemThreads) : "memory");
        Dterm = (vec[row_in_tile] + vec[kTile + row_in_tile]) * a.scale;
      }
      const size_t stat_idx = static_cast<size_t>(head) * a.R + min(row, a.R - 1);
      Lrow = load_stat(a.L, stat_idx, a.l_prec);
      if (h == 0 && row < a.R && split == 0) store_stat(a.Dterm, stat_idx, a.d_prec, Dterm);
    } else {
      if (threadIdx.x < 128) vec[threadIdx.x] = load_column_stat(blk0);
    }

    for (uint32_t j = 0; j < num_blocks; ++j) {
      const uint32_t b = j & 1, ph = (j >> 1) & 1;
      const uint32_t tS = tLane + Cfg::kTmemS + b * kBlock + h * kCols;
      const uint32_t tdP = tLane + Cfg::kTmemdP + b * kBlock + h * kCols;
      float next_stat = 0.f;
      if constexpr (kMode != kQuery) {
        // vec[b] (this block's statistics) is complete, vec[b ^ 1] is no longer read: fetch the next block's
        asm volatile("bar.sync 1, %0;" ::"n"(kElemThreads) : "memory");
        if (j + 1 < num_blocks && threadIdx.x < 128) next_stat = load_column_stat(blk0 + j + 1);
      }
      mbar_wait(&s_full[b], ph);
      tc_fence_after();
      float p[kCols];
      tmem_ld32(tS, *reinterpret_cast<uint32_t(*)[32]>(&p[0]));
      tc_wait_ld();
      if constexpr (kMode == kQuery || kMode == kKey) {
        tc_fence_before();
        mbar_arrive(&s_free[b]);  // S(j+2) may overwrite this buffer
      }

      if constexpr (kMode == kQuery) {
        const uint32_t col0 = (blk0 + j) * kBlock + h * kCols;
        if (col0 + kCols > a.C) {  // padded key columns (maskAttentionMatrixEdge): P = 0 there
#pragma unroll
          for (uint32_t c = 0; c < kCols; ++c)
            if (col0 + c >= a.C) p[c] = -INFINITY;
        }
        const float2 scale2 = make_float2(a.scale_log2, a.scale_log2), negL = make_float2(-Lrow, -Lrow);
#pragma unroll
        for (uint32_t c = 0; c < kCols; c += 2) {
          const float2 x = ffma2(make_float2(p[c], p[c + 1]), scale2, negL);
          p[c] = ex2_approx(x.x);
          p[c + 1] = ex2_approx(x.y);
        }
      } else {
        const float4 *Lc = reinterpret_cast<const float4 *>(vec + b * 128 + h * kCols);
        const float2 scale2 = make_float2(a.scale_log2, a.scale_log2);
#pragma unroll
        for (uint32_t c = 0; c < kCols; c += 4) {
          const float4 l4 = Lc[c >> 2];
          const float2 x0 = ffma2(make_float2(p[c], p[c + 1]), scale2, make_float2(-l4.x, -l4.y));
          const float2 x1 = ffma2(make_float2(p[c + 2], p[c + 3]), scale2, make_float2(-l4.z, -l4.w));
          p[c] = ex2_approx(x0.x);
          p[c + 1] = ex2_approx(x0.y);
          p[c + 2] = ex2_approx(x1.x);
          p[c + 3] = ex2_approx(x1.y);
        }
      }

      uint32_t packed[kCols / 2];
      if constexpr (kMode == kValue) {
        // P^T (16-bit) over S^T: columns [32 h, 32 h + 32) -> 32-bit columns [32 h, 32 h + 16) of the same buffer
#pragma unroll
        for (uint32_t k = 0; k < kCols / 2; ++k)
          packed[k] = kBF16 ? pack_bf16x2(p[2 * k], p[2 * k + 1]) : pack_f16x2(p[2 * k], p[2 * k + 1]);
        tmem_st16(tS, packed);
      } else {
        if constexpr (kMode == kKeyValue) {
          // P^T over S^T first: dV += P^T dO can run while dS^T is being computed
#pragma unroll
          for (uint32_t k = 0; k < kCols / 2; ++k)
            packed[k] = kBF16 ? pack_bf16x2(p[2 * k], p[2 * k + 1]) : pack_f16x2(p[2 * k], p[2 * k + 1]);
          tmem_st16(tS, packed);
          tc_wait_st();
          tc_fence_before();
          mbar_arrive(&p_full[b]);
        }
        // dS = P * (dP / sqrt(D) - D), written over dP as the 16-bit A operand of the accumulate MMA
        mbar_wait(&dp_full[b], ph);
        tc_fence_after();
        uint32_t dp[kCols];
        tmem_ld32(tdP, dp);
        tc_wait_ld();
        const float2 scale2 = make_float2(a.scale, a.scale);
        const float4 *Dc = reinterpret_cast<const float4 *>(vec + b * 128 + 64 + h * kCols);
#pragma unroll
        for (uint32_t k = 0; k < kCols / 2; ++k) {
          float2 negD;
          if constexpr (kMode == kQuery) {
            negD = make_float2(-Dterm, -Dterm);
          } else {
            const float4 d4 = Dc[k >> 1];
            negD = (k & 1) ? make_float2(-d4.z, -d4.w) : make_float2(-d4.x, -d4.y);
          }
          const float2 t = ffma2(make_float2(__uint_as_float(dp[2 * k]), __uint_as_float(dp[2 * k + 1])), scale2, negD);
          const float2 ds = fmul2(make_float2(p[2 * k], p[2 * k + 1]), t);
          packed[k] = kBF16 ? pack_bf16x2(ds.x, ds.y) : pack_f16x2(ds.x, ds.y);
        }
        tmem_st16(tdP, packed);
      }
      tc_wait_st();
      tc_fence_before();
      mbar_arrive(&ds_full[b]);
      if constexpr (kMode != kQuery) {
        if (j + 1 < num_blocks && threadIdx.x < 128) vec[(b ^ 1) * 128 + threadIdx.x] = next_stat;
      }
    }

    // ---------------- epilogue: accumulator -> global (FP32) ----------------
    mbar_wait(acc_final, 0);
    tc_fence_after();
    auto store_accumulator = [&](uint32_t t_col, float *out, bool transposed) {
      float *out_head = out + split * a.split_stride + static_cast<size_t>(head) * par_len * a.D;
      if (transposed) {
        float *o_col = out_head + row;
#pragma unroll 1
        for (uint32_t cc = 0; cc < DPAD / 2; cc += 32) {
          const uint32_t c = h * (DPAD / 2) + cc;
          uint32_t o[32];
          tmem_ld32(tLane + t_col + c, o);
          tc_wait_ld();
          if (row < par_len) {
#pragma unroll
            for (uint32_t k = 0; k < 32; ++k)
              if (c + k < a.D) o_col[static_cast<size_t>(c + k) * par_len] = __uint_as_float(o[k]);
          }
        }
      } else {
        float4 *scratch = reinterpret_cast<float4 *>(smem + Cfg::kSmemScratch) + warp * 256;
        const uint32_t warp_row0 = p0 + quarter * 32;
        store_accumulator_coalesced(tLane + t_col, h * (DPAD / 2), DPAD / 2, scratch,
                                    out_head + static_cast<size_t>(warp_row0) * a.D, warp_row0, par_len, a.D, lane);
      }
    };
    store_accumulator(Cfg::kTmemAcc, a.out, a.tmask & kTransOut);
    if constexpr (kMode == kKeyValue) store_accumulator(Cfg::kTmemAcc2, a.out2, a.tmask & kTransOut2);
  } else {
    setmaxnreg_dec<kOtherRegs>();
    // 128-row resident tile / 64-row block -> shared memory.  Row-major: one [rows][64 columns of D] box per 64-column
    // sub-tile; transposed: boxes of [DPAD rows of D][64 sequence elements].
    auto load_resident = [&](uint8_t *dst, const CUtensorMap *map, uint64_t *bar, bool t) {
      if (t) {
        tma_load_3d(dst, map, bar, p0, 0, head);
        tma_load_3d(dst + DPAD * 128, map, bar, p0 + 64, 0, head);
      } else {
#pragma unroll
        for (uint32_t ds = 0; ds < DPAD / 64; ++ds) tma_load_3d(dst + ds * (kTile * 128), map, bar, ds * 64, p0, head);
      }
    };
    auto load_block = [&](uint8_t *dst, const CUtensorMap *map, uint64_t *bar, bool t, uint32_t row0) {
      if (t) {
        tma_load_3d(dst, map, bar, row0, 0, head);
      } else {
#pragma unroll
        for (uint32_t ds = 0; ds < DPAD / 64; ++ds) tma_load_3d(dst + ds * (kBlock * 128), map, bar, ds * 64, row0, head);
      }
    };

    if (warp == 9) {
      // ---------------- TMA producer: resident tiles, ring 1 ----------------
      if (elect_one()) {
        mbar_arrive_expect_tx(res_full, Cfg::kResidents * Cfg::kResBytes);
        load_resident(smem + Cfg::kSmemRes, &mapA1, res_full, tA1);
        if (Cfg::kResidents == 2) load_resident(smem + Cfg::kSmemRes + Cfg::kResBytes, &mapA2, res_full, tA2);
      }
      for (uint32_t j = 0; j < num_blocks; ++j) {
        const uint32_t st = j & 1, ph = (j >> 1) & 1;
        mbar_wait(&r1_empty[st], ph ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&r1_full[st], Cfg::kBlkBytes);
          load_block(smem + Cfg::kSmemRing1 + st * Cfg::kBlkBytes, &mapB1, &r1_full[st], tB1, (blk0 + j) * kBlock);
        }
      }
    } else if (warp == 10) {
      // ---------------- TMA producer for ring 2 ----------------
      for (uint32_t j = 0; j < num_blocks; ++j) {
        const uint32_t st = j % Cfg::kStages2, ph = (j / Cfg::kStages2) & 1;
        mbar_wait(&r2_empty[st], ph ^ 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&r2_full[st], Cfg::kBlkBytes);
          load_block(smem + Cfg::kSmemRing2 + st * Cfg::kBlkBytes, &mapB2, &r2_full[st], tB2, (blk0 + j) * kBlock);
        }
      }
    } else if (warp == 8) {
      // ---------------- MMA issuer ----------------
      constexpr uint32_t kFormat = kBF16 ? 1u : 0u;
      // [128 x 64] = A[128 x D] . B[64 x D]^T.  Row-major tiles are K-major operands (16 elements of D = 32 B inside
      // the 128 B swizzle row, 64-column sub-tiles rows x 128 B apart); transposed tiles are MN-major (16 rows of D =
      // 2048 B; the two 64-row halves of A are DPAD x 128 B apart: LBO).
      auto issue_nt = [&](uint32_t d_tmem, uint32_t a_off, bool tA, uint32_t b_off, bool tB) {
        const uint32_t idesc = make_idesc_f16(kTile, kBlock, kFormat, tA ? 1u : 0u, tB ? 1u : 0u);
        const uint64_t da = make_smem_desc_sw128(smem_u32(smem + a_off), tA ? DPAD * 128 : 16, 1024);
        const uint64_t db = make_smem_desc_sw128(smem_u32(smem + b_off), 16, 1024);
#pragma unroll 4
        for (uint32_t k = 0; k < DPAD / 16; ++k) {
          const uint32_t ao = tA ? k * 2048 : (k >> 2) * (kTile * 128) + (k & 3) * 32;
          const uint32_t bo = tB ? k * 2048 : (k >> 2) * (kBlock * 128) + (k & 3) * 32;
          umma_ss(d_tmem, da + (ao >> 4), db + (bo >> 4), idesc, k > 0);
        }
      };
      // acc[128 x DPAD] (+)= A[128 x 64] (TMEM, 16-bit) . B[64 x DPAD].  A row-major block is an MN-major B (16 rows =
      // 2048 B, 64-column blocks 64 x 128 B apart: LBO); a transposed block ([DPAD rows of D][64]) is K-major.
      // The thread's columns [32 h, 32 h + 32) sit in 32-bit columns [32 h, 32 h + 16) of the buffer.
      auto issue_acc = [&](uint32_t d_col, uint32_t a_tmem, uint32_t b_off, bool tB, uint32_t accumulate) {
        const uint32_t idesc = make_idesc_f16(kTile, DPAD, kFormat, 0, tB ? 0u : 1u);
        const uint64_t db = make_smem_desc_sw128(smem_u32(smem + b_off), tB ? 16 : kBlock * 128, 1024);
#pragma unroll
        for (uint32_t k = 0; k < kBlock / 16; ++k) {
          const uint32_t bo = tB ? k * 32 : k * 2048;
          umma_ts(tmem_base + d_col, a_tmem + (k >> 1) * kCols + (k & 1) * 8, db + (bo >> 4), idesc,
                  k > 0 ? 1u : accumulate);
        }
      };
      auto issue_S = [&](uint32_t j) {
        const uint32_t st = j & 1;
        mbar_wait(&r1_full[st], (j >> 1) & 1);
        if ((kMode == kQuery || kMode == kKey) && j >= 2) mbar_wait(&s_free[j & 1], ((j - 2) >> 1) & 1);
        tc_fence_after();
        if (elect_one()) {
          issue_nt(tmem_base + Cfg::kTmemS + (j & 1) * kBlock, Cfg::kSmemRes, tA1, Cfg::kSmemRing1 + st * Cfg::kBlkBytes, tB1);
          umma_commit(&s_full[j & 1]);
          if (kMode == kValue) umma_commit(&r1_empty[st]);
        }
        __syncwarp();
      };
      auto issue_dP = [&](uint32_t j) {
        const uint32_t st = j % Cfg::kStages2, ph = (j / Cfg::kStages2) & 1;
        mbar_wait(&r2_full[st], ph);
        tc_fence_after();
        if (elect_one()) {
          issue_nt(tmem_base + Cfg::kTmemdP + (j & 1) * kBlock, Cfg::kSmemRes + Cfg::kResBytes, tA2,
                   Cfg::kSmemRing2 + st * Cfg::kBlkBytes, tB2);
          umma_commit(&dp_full[j & 1]);
          if (kMode != kKeyValue) umma_commit(&r2_empty[st]);  // (kKeyValue: dV += P^T dO still reads the block)
        }
        __syncwarp();
      };

      mbar_wait(res_full, 0);
      if constexpr (kMode != kValue) issue_dP(0);
      issue_S(0);
      for (uint32_t j = 0; j < num_blocks; ++j) {
        if (j + 1 < num_blocks) {
          // the dP buffer of block j+1 was last read by acc(j-1), the S buffer (kValue: P) likewise: both ahead of
          // these on the in-order tensor pipe
          if constexpr (kMode != kValue) issue_dP(j + 1);
          issue_S(j + 1);
        }
        if constexpr (kMode == kKeyValue) {
          // dV += P^T(j) dO(j) as soon as P^T is written; dS^T(j) is still being computed
          const uint32_t st = j % Cfg::kStages2;
          mbar_wait(&p_full[j & 1], (j >> 1) & 1);
          tc_fence_after();
          if (elect_one()) {
            issue_acc(Cfg::kTmemAcc2, tmem_base + Cfg::kTmemS + (j & 1) * kBlock, Cfg::kSmemRing2 + st * Cfg::kBlkBytes, tB2,
                      j > 0 ? 1u : 0u);
            umma_commit(&r2_empty[st]);
          }
          __syncwarp();
        }
        mbar_wait(&ds_full[j & 1], (j >> 1) & 1);
        if constexpr (kMode == kValue) {
          const uint32_t st = j % Cfg::kStages2, ph = (j / Cfg::kStages2) & 1;
          mbar_wait(&r2_full[st], ph);
          tc_fence_after();
          if (elect_one()) {
            issue_acc(Cfg::kTmemAcc, tmem_base + Cfg::kTmemS + (j & 1) * kBlock, Cfg::kSmemRing2 + st * Cfg::kBlkBytes, tB2,
                      j > 0 ? 1u : 0u);
            umma_commit(&r2_empty[st]);
            if (j + 1 == num_blocks) umma_commit(acc_final);
          }
        } else {
          tc_fence_after();
          if (elect_one()) {
            issue_acc(Cfg::kTmemAcc, tmem_base + Cfg::kTmemdP + (j & 1) * kBlock, Cfg::kSmemRing1 + (j & 1) * Cfg::kBlkBytes, tB1,
                      j > 0 ? 1u : 0u);
            umma_commit(&r1_empty[j & 1]);
            if (j + 1 == num_blocks) umma_commit(acc_final);
          }
        }
        __syncwarp();
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static cudaError_t operand_map(CUtensorMap *map, const AttentionParams &p, int slot, uint32_t seq, uint32_t box_rows,
                               uint32_t dpad) {
  return p.transposed[slot] ? make_tensor_map_16bit_transposed(map, p.buf[slot], seq, p.D, p.batch, dpad)
                            : make_tensor_map_16bit(map, p.buf[slot], seq, p.D, p.batch, box_rows);
}

template <uint32_t DPAD, bool kBF16, uint32_t kMode>
cudaError_t launch_pass(const AttentionParams &p, cudaStream_t stream) {
  using Cfg = Config<DPAD, kMode>;
  auto kernel = attention_backward_generic_tcgen05<DPAD, kBF16, kMode>;
  const int device = current_device();
  cudaError_t e = ensure_max_dynamic_smem(reinterpret_cast<const void *>(kernel), Cfg::kSmemBytes, device);
  if (e != cudaSuccess) return e;

  // (A1, A2) resident, (B1, B2) streamed -- see the table in the file header
  const int sA1 = kMode == kQuery ? sQ : sK, sA2 = kMode == kQuery ? sdO : sV;
  const int sB1 = kMode == kQuery ? sK : sQ, sB2 = kMode == kQuery ? sV : sdO;
  const int sOut = kMode == kQuery ? sdQ : (kMode == kValue ? sdV : sdK);  // (kKeyValue: dK, and dV as the second output)
  const uint32_t par = kMode == kQuery ? p.R : p.C, trav = kMode == kQuery ? p.C : p.R;
  CUtensorMap mapA1, mapA2, mapB1, mapB2;
  if ((e = operand_map(&mapA1, p, sA1, par, kTile, DPAD)) != cudaSuccess) return e;
  if ((e = operand_map(&mapA2, p, sA2, par, kTile, DPAD)) != cudaSuccess) return e;
  if ((e = operand_map(&mapB1, p, sB1, trav, kBlock, DPAD)) != cudaSuccess) return e;
  if ((e = operand_map(&mapB2, p, sB2, trav, kBlock, DPAD)) != cudaSuccess) return e;

  GenericArgs a;
  a.dO = p.buf[sdO];
  a.O = static_cast<const float *>(p.buf[sO]);
  a.L = p.buf[sL];
  a.Dterm = p.buf[sD];
  a.out = static_cast<float *>(p.buf[sOut]);
  a.out2 = static_cast<float *>(p.buf[sdV]);
  a.R = p.R;
  a.C = p.C;
  a.D = p.D;
  a.scale = p.scale;
  a.scale_log2 = p.scale_log2;
  a.l_prec = p.prec[sL];
  a.d_prec = p.prec[sD];
  a.tmask = (p.transposed[sA1] ? kTransA1 : 0u) | (p.transposed[sA2] ? kTransA2 : 0u) | (p.transposed[sB1] ? kTransB1 : 0u) |
            (p.transposed[sB2] ? kTransB2 : 0u) | (p.transposed[sOut] ? kTransOut : 0u) | (p.transposed[sO] ? kTransO : 0u) |
            (p.transposed[sdO] ? kTransdO : 0u) | (p.transposed[sdV] ? kTransOut2 : 0u);

  const uint32_t tiles = (par + kTile - 1) / kTile, total_blocks = (trav + kBlock - 1) / kBlock;
  // the row's split policy counts 128-row blocks
  const uint32_t per = bwd::choose_blocks_per_split(tiles * p.batch, total_blocks, device_sm_count(device),
                                                    2u * p.split_min_blocks, p.split_max);
  const uint32_t splits = (total_blocks + per - 1) / per;
  a.blocks_per_split = per;
  a.split_stride = 0;
  a.tiles = tiles;
  a.batch = p.batch;
  a.num_splits = splits;
  a.num_items = tiles * p.batch * splits;
  if (splits == 1) {
    kernel<<<a.num_items, kThreads, Cfg::kSmemBytes, stream>>>(mapA1, mapA2, mapB1, mapB2, a);
    return cudaGetLastError();
  }
  const size_t tensor_elems = static_cast<size_t>(p.batch) * par * p.D;
  constexpr uint32_t tensors = kMode == kKeyValue ? 2 : 1;  // partial accumulators: [split][tensor][batch][rows][D]
  void *ws = nullptr;
  if ((e = workspace_for(device, stream, splits * tensors * tensor_elems * sizeof(float), &ws)) != cudaSuccess) return e;
  float *scratch = static_cast<float *>(ws);
  a.split_stride = tensors * tensor_elems;
  a.out = scratch;
  a.out2 = scratch + tensor_elems;
  kernel<<<a.num_items, kThreads, Cfg::kSmemBytes, stream>>>(mapA1, mapA2, mapB1, mapB2, a);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  return bwd::launch_sum_splits(scratch, static_cast<float *>(p.buf[sOut]), static_cast<float *>(p.buf[sdV]), tensor_elems,
                                tensors, a.split_stride, splits, stream);
}

template <uint32_t DPAD, bool kBF16>
cudaError_t launch(const AttentionParams &p, cudaStream_t stream, bool key_value) {
  if (!key_value) return launch_pass<DPAD, kBF16, kQuery>(p, stream);
  if constexpr (DPAD <= 128) {
    return launch_pass<DPAD, kBF16, kKeyValue>(p, stream);  // dK and dV fit TMEM side by side: one pass
  } else {
    cudaError_t e = launch_pass<DPAD, kBF16, kValue>(p, stream);
    if (e != cudaSuccess) return e;
    return launch_pass<DPAD, kBF16, kKey>(p, stream);
  }
}

static uint32_t pass_launches(uint32_t par, uint32_t trav, uint32_t batch, uint32_t min_blocks, uint32_t max_splits) {
  const uint32_t tiles = (par + kTile - 1) / kTile, total_blocks = (trav + kBlock - 1) / kBlock;
  return bwd::choose_blocks_per_split(tiles * batch, total_blocks, device_sm_count(current_device()), 2u * min_blocks,
                                      max_splits) < total_blocks ? 2 : 1;
}

}  // namespace bwdg

// TMA addresses a transposed operand through its [D][seq] view: the row pitch (seq elements) must be 16-byte aligned
bool tcgen05_backward_transposes_ok(uint32_t R, uint32_t C, bool tQ, bool tK, bool tV, bool tO) {
  if ((tQ || tO) && R % 8 != 0) return false;  // dO follows O, Q^T and dO^T are fetched by TMA
  if ((tK || tV) && C % 8 != 0) return false;
  return true;
}

cudaError_t launch_tcgen05_backward_generic(const AttentionParams &p_in, cudaStream_t stream, bool key_value) {
  AttentionParams p = p_in;
  // The reference's policy (FP16 Q/K/V beside BF16 dO): tcgen05 kind::f16 cannot mix the two types in one MMA.  These
  // kernels stream dO blocks through a one- or two-stage ring with only two spare warps to rewrite them (measured: the dK
  // pass at D = 256 fell from 762 to 533 TFLOP/s with the in-kernel rewrite), so dO is converted ONCE into the workspace
  // (O(N D) against O(N^2 D)) and the all-FP16 instantiations run.
  if (p.prec[sdO] != p.prec[sQ]) {
    const uint64_t elements = static_cast<uint64_t>(p.batch) * p.R * p.D;
    void *ws = nullptr;
    cudaError_t e = workspace_for(current_device(), stream, elements * 2, &ws, /*slot=*/2);
    if (e != cudaSuccess) return e;
    if ((e = launch_bf16_to_f16(p.buf[sdO], ws, elements, stream)) != cudaSuccess) return e;
    p.buf[sdO] = ws;
    p.prec[sdO] = p.prec[sQ];
  }
  const bool bf16 = p.prec[sQ] == BF16;
#define MFA_BWDG_MODES(DPAD_) \
  return bf16 ? bwdg::launch<DPAD_, true>(p, stream, key_value) : bwdg::launch<DPAD_, false>(p, stream, key_value);
  if (p.D <= 64) {
    MFA_BWDG_MODES(64)
  }
  if (p.D <= 128) {
    MFA_BWDG_MODES(128)
  }
  MFA_BWDG_MODES(256)
#undef MFA_BWDG_MODES
}

// backwardQuery: 1 launch (+1 when the traversal split engages); backwardKeyValue: one pass at D <= 128, else the dV pass
// and the dK pass
uint32_t tcgen05_backward_generic_launch_count(int type, uint32_t R, uint32_t C, uint32_t D, uint32_t batch,
                                               uint32_t min_blocks, uint32_t max_splits, bool convert_dO) {
  const uint32_t extra = convert_dO ? 1 : 0;  // the BF16 -> FP16 copy of dO
  if (type == 1) return extra + bwdg::pass_launches(R, C, batch, min_blocks, max_splits);
  return extra + (D <= 128 ? 1 : 2) * bwdg::pass_launches(C, R, batch, min_blocks, max_splits);
}

void tcgen05_backward_generic_geometry(int type, uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par,
                                       uint32_t *trav, uint32_t *head) {
  *threads = bwdg::kThreads;
  const uint32_t block = D <= 64 ? 64u : (D <= 128 ? 128u : 256u);
  if (type == 1)
    *smem_bytes = block == 64 ? bwdg::Config<64, bwdg::kQuery>::kSmemBytes
                              : (block == 128 ? bwdg::Config<128, bwdg::kQuery>::kSmemBytes : bwdg::Config<256, bwdg::kQuery>::kSmemBytes);
  else  // the larger of the two passes
    *smem_bytes = block == 64 ? bwdg::Config<64, bwdg::kKeyValue>::kSmemBytes
                              : (block == 128 ? bwdg::Config<128, bwdg::kKeyValue>::kSmemBytes : bwdg::Config<256, bwdg::kKey>::kSmemBytes);
  *par = bwdg::kTile;
  *trav = bwdg::kBlock;
  const uint32_t padded = (D + 7) / 8 * 8;
  *head = block < padded ? block : padded;
}

}  // namespace mfa

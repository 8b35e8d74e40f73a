// FlashAttention forward for sm_100a, large head dimensions (128 < D <= 256): the reference's "nothing cached /
// intentional spill" regime (AttentionDescriptor+Parameters.swift:113,120: the 384 rows) re-expressed for B200.
//
// At D = 256 one query tile's O accumulator alone takes 256 of the 512 TMEM columns and a 128-key K or V tile takes
// 64 KB of shared memory, so the residency choices change relative to tcgen05_forward.cu:
//   * one 128-row tcgen05 M-tile per CTA (not two), O resident in TMEM columns [256, 512);
//   * keys are walked in blocks of 128 (S = Q K^T as M128 x N128 MMAs: an N = 64 MMA costs the tensor pipe as many
//     cycles as an N = 128 one -- measured, 64 cycles each -- so 64-key blocks ran S at half rate);
//   * K and V are SINGLE-buffered (Q 64 KB + K 64 KB + V 64 KB) but recycled at sub-tile granularity: S walks K's four
//     64-column sub-tiles in order and releases each as soon as its four k-steps have retired, O += P V releases V in
//     two 64-key halves; because S and P V alternate on the in-order tensor pipe, every reload has at least one whole
//     GEMM (~1000 cycles) to land before it is needed;
//   * S is double-buffered in TMEM (2 x 128 columns), so S(i+1) runs while the softmax warps work on S(i); P (16-bit)
//     overwrites S in place and feeds O += P V straight from TMEM.
// Warp roles (384 threads): warps 0-7 softmax -- two warpgroups that split every block's 128 key columns in half
// (thread = query row x 64 columns; the two warps of a row quarter agree on rescales through a 64-thread named
// barrier with an OR reduction) -- warp 8 MMA issuer, warp 9 TMA producer for Q and K, warp 10 for V.  One softmax
// warp per SM sub-partition cannot issue ex2 faster than about one per 16 cycles (half the pipe's rate), hence two.
// Softmax conventions are those of tcgen05_forward.cu (log2 domain, lazy rescale on a half-row-sum check,
// L = m + log2 l).  History of this kernel (N = 8192, D = 256, 16 heads, TFLOP/s): 64-key blocks, one softmax
// warpgroup, one TMA producer 956; two warpgroups 970; separate K / V producers and P V decoupled from the next S
// 1155-1257; 128-key blocks: see DESIGN.md.
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include "attention_params.h"
#include "device_state.h"
#include "sm100_ptx.cuh"
#include "tma_host.h"

namespace mfa {
namespace fwd256 {

using namespace ptx;

constexpr uint32_t kTileM = 128;       // rows per tcgen05 M-tile (one per CTA)
constexpr uint32_t kBlockN = 128;      // keys per traversal block
constexpr uint32_t kSBuffers = 2;      // S/P buffers
constexpr uint32_t kSubTileBytes = 128 * 128;  // [128 rows][64 x 16-bit]: one 128B-swizzled sub-tile
constexpr uint32_t kVHalfBytes = 64 * 128;     // [64 keys][64 x 16-bit]: half a V sub-tile (one TMA box)
constexpr uint32_t kThreads = 384;
// setmaxnreg budget: the CTA is launched with floor(65536 / 384 / 8) * 8 = 168 registers per thread; the two
// softmax warpgroups grow to kSoftmaxRegs after the producer warpgroup has shrunk to kOtherRegs.  The sum
// must not exceed the launch allocation or the second setmaxnreg.inc never returns.
constexpr uint32_t kLaunchRegs = 168, kSoftmaxRegs = 208, kOtherRegs = 88;
static_assert(kSoftmaxRegs * 256 + kOtherRegs * 128 <= kLaunchRegs * kThreads, "setmaxnreg over-subscribed");
constexpr float kLazySumLimit = 256.0f;  // a half-row of P summing to <= 2^8 proves every element is <= 2^8

// named barrier over `count` threads with an OR reduction of `flag` (all participating warps get the result)
__device__ __forceinline__ bool bar_red_or(uint32_t id, uint32_t count, bool flag) {
  uint32_t out;
  asm volatile(
      "{\n"
      ".reg .pred p, q;\n"
      "setp.ne.u32 q, %3, 0;\n"
      "barrier.cta.red.or.pred p, %1, %2, q;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(out)
      : "r"(id), "r"(count), "r"(static_cast<uint32_t>(flag))
      : "memory");
  return out != 0;
}
__device__ __forceinline__ void bar_sync(uint32_t id, uint32_t count) {
  asm volatile("barrier.cta.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}

template <uint32_t DPAD>
struct Config {
  static constexpr uint32_t kSubTiles = DPAD / 64;                  // 64-element sub-tiles along D
  static constexpr uint32_t kTileBytes = kSubTiles * kSubTileBytes;  // one 128 x DPAD operand tile
  static constexpr uint32_t kSmemQ = 0;
  static constexpr uint32_t kSmemK = kSmemQ + kTileBytes;
  static constexpr uint32_t kSmemV = kSmemK + kTileBytes;
  static constexpr uint32_t kSmemXch = kSmemV + kTileBytes;  // float [2][128]: row max / row sum exchange
  static constexpr uint32_t kSmemBar = kSmemXch + 2 * kTileM * 4;
  // q_full, k_full[sub], k_empty[sub], v_full[2], v_empty[2], s_full[2], p_full[2], o_full, o_final
  static constexpr uint32_t kNumBars = 1 + 2 * kSubTiles + 4 + 2 * kSBuffers + 2;
  static constexpr uint32_t kSmemTmemPtr = kSmemBar + kNumBars * 8;
  static constexpr uint32_t kSmemBytes = kSmemTmemPtr + 16 + 1024;  // + slack for manual 1024 B alignment
  static_assert(kSmemBytes <= 232448, "shared memory over budget");
  static_assert(8 * 4096 <= kTileBytes, "epilogue scratch does not fit the K tile");
  static constexpr uint32_t kTmemO = kSBuffers * kBlockN;  // O follows the two S buffers
  static constexpr uint32_t kTmemCols = 512;
  static_assert(kTmemO + DPAD <= kTmemCols, "tile does not fit TMEM");
};

// kTrace: debug instantiation that records clock64() at the pipeline hand-off points of CTA (0,0)
// (scripts/trace_forward_d256.py); the production instantiation compiles all of it away.
constexpr uint32_t kTraceSlots = 8;    // per (role, iteration)
constexpr uint32_t kTraceIters = 128;  // iterations recorded per role
#define MFA_TRACE(role, iter, slot)                                                                   \
  do {                                                                                                \
    if (kTrace && trace != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && lane == 0 &&             \
        (iter) < kTraceIters)                                                                         \
      trace[((role) * kTraceIters + (iter)) * kTraceSlots + (slot)] = clock64();                      \
  } while (0)

// kGeneric: the layout-generic instantiation, which also serves TRANSPOSED operands (stored [D][seq], leading dimension
// = sequence length: AttentionKernel.swift:189-195) for any D <= 256.  `tmask` bit 0/1/2/3 = Q/K/V/O transposed.  A
// transposed operand is fetched through a tensor map of the transposed view (inner dimension = sequence) and consumed
// through the other UMMA major-ness: Q^T and K^T tiles are MN-major operands of S = Q K^T, V^T is a K-major operand of
// O += P V; a transposed O is stored straight from registers (a warp's 32 rows are contiguous in memory then).
template <uint32_t DPAD, bool kBF16, bool kTrace = false, bool kGeneric = false>
__global__ void __launch_bounds__(kThreads, 1)
    attention_forward_d256_tcgen05(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                              const __grid_constant__ CUtensorMap mapV, float *__restrict__ O, void *__restrict__ L,
                              uint32_t R, uint32_t C, uint32_t D, float scale_log2, int l_is_fp16, uint32_t tmask,
                              long long *__restrict__ trace) {
  using Cfg = Config<DPAD>;
  const bool transQ = kGeneric && (tmask & 1u), transK = kGeneric && (tmask & 2u), transV = kGeneric && (tmask & 4u),
             transO = kGeneric && (tmask & 8u);
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t head = blockIdx.y;
  const uint32_t q_row0 = blockIdx.x * kTileM;
  const uint32_t num_blocks = (C + kBlockN - 1) / kBlockN;

  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::kSmemBar);
  uint64_t *q_full = bars;
  uint64_t *k_full = q_full + 1;                 // [sub-tile]  one phase per key block
  uint64_t *k_empty = k_full + Cfg::kSubTiles;   // [sub-tile]
  uint64_t *v_full = k_empty + Cfg::kSubTiles;   // [key half]
  uint64_t *v_empty = v_full + 2;                // [key half]
  uint64_t *s_full = v_empty + 2;                // [buffer]
  uint64_t *p_full = s_full + kSBuffers;         // [buffer] (256 arrivals)
  uint64_t *o_full = p_full + kSBuffers;         // one phase per key block
  uint64_t *o_final = o_full + 1;                // completes once, after the last O += P V
  uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(smem + Cfg::kSmemTmemPtr);

  // ---------------- one-time setup ----------------
  if (threadIdx.x == 0) {
    mbar_init(q_full, 1);
    for (uint32_t s = 0; s < Cfg::kSubTiles; ++s) {
      mbar_init(&k_full[s], 1);
      mbar_init(&k_empty[s], 1);
    }
    for (uint32_t s = 0; s < 2; ++s) {
      mbar_init(&v_full[s], 1);
      mbar_init(&v_empty[s], 1);
    }
    for (uint32_t bf = 0; bf < kSBuffers; ++bf) {
      mbar_init(&s_full[bf], 1);
      mbar_init(&p_full[bf], 2 * kTileM);
    }
    mbar_init(o_full, 1);
    mbar_init(o_final, 1);
    fence_barrier_init();
  }
  if (warp == 8) {
    tmem_alloc(tmem_ptr_smem, Cfg::kTmemCols);
    tmem_relinquish();
  }
  if (warp == 9 && lane == 0) {
    prefetch_tensormap(&mapQ);
    prefetch_tensormap(&mapK);
    prefetch_tensormap(&mapV);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  if (warp < 8) {
    // =====================================================================================
    // softmax warps: thread <-> (query row, half of the block's 128 key columns).  Warpgroup h = warp / 4 owns columns
    // [64 h, 64 h + 64); warps w and w + 4 share the 32 rows of TMEM lane quarter w and take their joint decisions
    // (lazy rescale) through a 64-thread named barrier with an OR reduction.
    // =====================================================================================
    setmaxnreg_inc<kSoftmaxRegs>();
    constexpr uint32_t kCols = kBlockN / 2;  // columns per thread and block
    const uint32_t h = warp >> 2, quarter = warp & 3;
    const uint32_t row_in_tile = quarter * 32 + lane;
    const uint32_t tTile = tmem_base + ((quarter * 32) << 16);
    const uint32_t tO = tTile + Cfg::kTmemO;
    const uint32_t pair_bar = 2 + quarter;  // named barrier of the two warps that share these rows
    const uint32_t trace_role = warp == 0 ? 0 : (warp == 4 ? 1 : 3);
    float *xch = reinterpret_cast<float *>(smem + Cfg::kSmemXch);  // [2][128] row-max / row-sum exchange

    float m = -FLT_MAX;  // running max, log2 domain (AttentionKernel+Caching.swift:310); identical in both threads of a row
    float l = 0.f;       // running sum over this thread's columns
    const uint32_t tail_cols = C - (num_blocks - 1) * kBlockN;  // valid columns in the last block

    for (uint32_t i = 0; i < num_blocks; ++i) {
      const uint32_t bf = i & 1, ph = (i >> 1) & 1;
      const uint32_t tS = tTile + bf * kBlockN;
      mbar_wait(&s_full[bf], ph);
      tc_fence_after();
      MFA_TRACE(trace_role, i, 0);

      float s[kCols];
#pragma unroll
      for (uint32_t c = 0; c < kCols; c += 32) tmem_ld32(tS + h * kCols + c, *reinterpret_cast<uint32_t(*)[32]>(&s[c]));
      tc_wait_ld();
      MFA_TRACE(trace_role, i, 1);

      // edge mask (maskAttentionMatrixEdge, AttentionKernel+Softmax.swift:228-260)
      if (i == num_blocks - 1 && tail_cols < kBlockN) {
#pragma unroll
        for (uint32_t c = 0; c < kCols; ++c)
          if (h * kCols + c >= tail_cols) s[c] = -INFINITY;
      }

      // Lazy running max, as in tcgen05_forward.cu: P is computed against the current (possibly stale) m straight away;
      // only if some half-row of P sums to more than 2^8 -- or m was never set -- do the two warps of these rows fall
      // back to the exact path (joint row max, wait for every issued O += P V, rescale O and l, recompute).
      uint32_t packed[kCols / 2];
      float half_sum;
      if (i == 0) {
        half_sum = INFINITY;
      } else {
        float2 sum2 = make_float2(0.f, 0.f);
        const float2 scale2 = make_float2(scale_log2, scale_log2), negm2 = make_float2(-m, -m);
#pragma unroll
        for (uint32_t k = 0; k < kCols / 2; ++k) {
          const float2 x = ffma2(make_float2(s[2 * k], s[2 * k + 1]), scale2, negm2);
          float2 pr;
          pr.x = ex2_approx(x.x);
          pr.y = ex2_approx(x.y);
          sum2 = fadd2(sum2, pr);
          packed[k] = kBF16 ? pack_bf16x2(pr.x, pr.y) : pack_f16x2(pr.x, pr.y);
        }
        half_sum = sum2.x + sum2.y;
      }
      // (also orders both warps' S loads before either overwrites the buffer with P: warpgroup 1's P columns
      // [32, 64) lie inside warpgroup 0's S columns [0, 64))
      if (bar_red_or(pair_bar, 64, !(half_sum <= kLazySumLimit))) {  // also catches inf / NaN
        // ---- exact path (rare) ----
        float mx0 = s[0], mx1 = s[1], mx2 = s[2], mx3 = s[3];
#pragma unroll
        for (uint32_t c = 4; c < kCols; c += 4) {
          mx0 = fmaxf(mx0, s[c]);
          mx1 = fmaxf(mx1, s[c + 1]);
          mx2 = fmaxf(mx2, s[c + 2]);
          mx3 = fmaxf(mx3, s[c + 3]);
        }
        const float m_loc = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * scale_log2;
        xch[h * kTileM + row_in_tile] = m_loc;
        bar_sync(pair_bar, 64);
        const float m_new = fmaxf(m, fmaxf(m_loc, xch[(1 - h) * kTileM + row_in_tile]));
        if (i > 0) {
          mbar_wait(o_full, (i - 1) & 1);  // O += P V of the previous block has landed (the current one is not issued yet)
          tc_fence_after();
          const float correction = ex2_approx(m - m_new);
#pragma unroll
          for (uint32_t c = 0; c < DPAD / 2; c += 32) {  // each warpgroup rescales its half of the O columns
            uint32_t o[32];
            tmem_ld32(tO + h * (DPAD / 2) + c, o);
            tc_wait_ld();
#pragma unroll
            for (uint32_t k = 0; k < 32; ++k) o[k] = __float_as_uint(__uint_as_float(o[k]) * correction);
            tmem_st32(tO + h * (DPAD / 2) + c, o);
          }
          l *= correction;
        }
        m = m_new;
        float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
        for (uint32_t k = 0; k < kCols / 2; ++k) {
          const float p0 = ex2_approx(fmaf(s[2 * k], scale_log2, -m));
          const float p1 = ex2_approx(fmaf(s[2 * k + 1], scale_log2, -m));
          sum0 += p0;
          sum1 += p1;
          packed[k] = kBF16 ? pack_bf16x2(p0, p1) : pack_f16x2(p0, p1);
        }
        half_sum = sum0 + sum1;
        bar_sync(pair_bar, 64);  // the exchange slots may be rewritten in a later block only after both have read them
      }
      l += half_sum;
      MFA_TRACE(trace_role, i, 2);
      // P (16-bit) over S: keys [64 h, 64 h + 64) -> columns [32 h, 32 h + 32)
      tmem_st32(tS + h * (kCols / 2), packed);
      MFA_TRACE(trace_role, i, 3);
      tc_wait_st();
      tc_fence_before();
      mbar_arrive(&p_full[bf]);
      MFA_TRACE(trace_role, i, 4);
    }

    // ---------------- epilogue: O / l -> global (FP32), L = m + log2(l) ----------------
    // (o_full may be up to two phases behind here, which a parity wait cannot tell apart; o_final is one-shot)
    xch[h * kTileM + row_in_tile] = l;
    bar_sync(pair_bar, 64);
    l += xch[(1 - h) * kTileM + row_in_tile];
    mbar_wait(o_final, 0);
    tc_fence_after();
    const uint32_t row = q_row0 + row_in_tile;
    const float inv_l = 1.0f / l;
    if (transO) {
      // O stored [D][R]: for a fixed column the warp's 32 rows are 32 consecutive floats -- one 128 B line per store
      float *o_col = O + static_cast<size_t>(head) * D * R + row;
#pragma unroll 1
      for (uint32_t cc = 0; cc < DPAD / 2; cc += 32) {
        const uint32_t c = h * (DPAD / 2) + cc;
        uint32_t o[32];
        tmem_ld32(tO + c, o);
        tc_wait_ld();
        if (row < R) {
#pragma unroll
          for (uint32_t k = 0; k < 32; ++k)
            if (c + k < D) o_col[static_cast<size_t>(c + k) * R] = __uint_as_float(o[k]) * inv_l;
        }
      }
    } else {
      // Warpgroup h stores columns [h DPAD/2, (h+1) DPAD/2).  TMEM hands every thread one row; each warp transposes
      // 32 x 32 chunks through a private XOR-swizzled scratch tile (overlaying the K tile, dead after the last MMA)
      // so that every global store instruction writes four full 128 B lines (see tcgen05_forward.cu).
      float4 *scratch = reinterpret_cast<float4 *>(smem + Cfg::kSmemK) + warp * 256;
      const uint32_t warp_row0 = q_row0 + quarter * 32;
      float *o_base = O + (static_cast<size_t>(head) * R + warp_row0) * D;
      const uint32_t sub_row = lane >> 3, quad = lane & 7;
#pragma unroll 1
      for (uint32_t cc = 0; cc < DPAD / 2; cc += 32) {
        const uint32_t c = h * (DPAD / 2) + cc;
        uint32_t o[32];
        tmem_ld32(tO + c, o);
        tc_wait_ld();
#pragma unroll
        for (uint32_t j = 0; j < 8; ++j)
          scratch[lane * 8 + (j ^ (lane & 7))] =
              make_float4(__uint_as_float(o[4 * j]) * inv_l, __uint_as_float(o[4 * j + 1]) * inv_l,
                          __uint_as_float(o[4 * j + 2]) * inv_l, __uint_as_float(o[4 * j + 3]) * inv_l);
        __syncwarp();
        float4 v[8];
#pragma unroll
        for (uint32_t k = 0; k < 8; ++k) {
          const uint32_t r = 4 * k + sub_row;
          v[k] = scratch[r * 8 + (quad ^ (r & 7))];
        }
        if (c + 4 * quad < D) {  // D % 8 == 0: a float4 is either fully inside or fully outside
#pragma unroll
          for (uint32_t k = 0; k < 8; ++k) {
            const uint32_t r = 4 * k + sub_row;
            if (warp_row0 + r < R) *reinterpret_cast<float4 *>(o_base + static_cast<size_t>(r) * D + c + 4 * quad) = v[k];
          }
        }
        __syncwarp();
      }
    }
    if (h == 0 && row < R && L != nullptr) {
      const float lse2 = m + log2f(l);  // AttentionKernel+Caching.swift:373-377
      const size_t idx = static_cast<size_t>(head) * R + row;
      if (l_is_fp16)
        reinterpret_cast<__half *>(L)[idx] = __float2half_rn(lse2);
      else
        reinterpret_cast<float *>(L)[idx] = lse2;
    }
  } else {
    setmaxnreg_dec<kOtherRegs>();
    // The producer warps run their control flow warp-wide and hand exactly one elected lane to the
    // TMA / tcgen05 instructions: operands stay in uniform registers and the issue loops are branch-free.
    if (warp == 9) {
      // ===================================================================================
      // TMA producer: Q once, then K -- one sub-tile ([128 keys][64 columns of D]) at a time, each reloaded as soon
      // as the S MMAs that read it have retired
      // ===================================================================================
      if (elect_one()) {
        mbar_arrive_expect_tx(q_full, Cfg::kTileBytes);
        if (transQ) {  // two boxes of [DPAD rows of D][64 query rows]: the 64-row halves of the M tile
          tma_load_3d(smem + Cfg::kSmemQ, &mapQ, q_full, q_row0, 0, head);
          tma_load_3d(smem + Cfg::kSmemQ + DPAD * 128, &mapQ, q_full, q_row0 + 64, 0, head);
        } else {
#pragma unroll
          for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
            tma_load_3d(smem + Cfg::kSmemQ + ds * kSubTileBytes, &mapQ, q_full, ds * 64, q_row0, head);
        }
      }
      for (uint32_t i = 0; i < num_blocks; ++i) {
        MFA_TRACE(4, i, 0);
#pragma unroll
        for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds) {
          mbar_wait(&k_empty[ds], (i & 1) ^ 1);
          if (ds == 0) MFA_TRACE(4, i, 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(&k_full[ds], kSubTileBytes);
            if (transK) {  // two boxes of [64 rows of D][64 keys]: the key halves of this 64-column group of D
              tma_load_3d(smem + Cfg::kSmemK + ds * kSubTileBytes, &mapK, &k_full[ds], i * kBlockN, ds * 64, head);
              tma_load_3d(smem + Cfg::kSmemK + ds * kSubTileBytes + kVHalfBytes, &mapK, &k_full[ds], i * kBlockN + 64,
                          ds * 64, head);
            } else {
              tma_load_3d(smem + Cfg::kSmemK + ds * kSubTileBytes, &mapK, &k_full[ds], ds * 64, i * kBlockN, head);
            }
          }
        }
      }
    } else if (warp == 10) {
      // ===================================================================================
      // TMA producer for V, one 64-key half at a time (a separate warp: K reloads must not queue behind V's)
      // ===================================================================================
      for (uint32_t i = 0; i < num_blocks; ++i) {
#pragma unroll
        for (uint32_t half = 0; half < 2; ++half) {
          mbar_wait(&v_empty[half], (i & 1) ^ 1);
          if (half == 0) MFA_TRACE(4, i, 2);
          if (elect_one()) {
            mbar_arrive_expect_tx(&v_full[half], Cfg::kSubTiles * kVHalfBytes);
            if (transV) {  // one box of [DPAD rows of D][64 keys] per key half
              tma_load_3d(smem + Cfg::kSmemV + half * (DPAD * 128), &mapV, &v_full[half], i * kBlockN + half * 64, 0, head);
            } else {
#pragma unroll
              for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
                tma_load_3d(smem + Cfg::kSmemV + ds * kSubTileBytes + half * kVHalfBytes, &mapV, &v_full[half], ds * 64,
                            i * kBlockN + half * 64, head);
            }
          }
        }
      }
    } else if (warp == 8) {
      // ===================================================================================
      // MMA issuer
      // ===================================================================================
      constexpr uint32_t kFormat = kBF16 ? 1u : 0u;
      // S[128 x 128] = Q[128 x D] . K[128 x D]^T : A and B both K-major
      // (a transposed Q or K tile is an MN-major operand: rows = D, 64 sequence elements per 128 B swizzle row)
      const uint32_t idescS = make_idesc_f16(kTileM, kBlockN, kFormat, transQ ? 1u : 0u, transK ? 1u : 0u);
      // O[128 x DPAD] += P[128 x 128] . V[128 x DPAD] : A from TMEM, B (= V, [key][d]) is MN-major; a transposed V
      // ([d][key]) is K-major
      const uint32_t idescO = make_idesc_f16(kTileM, DPAD, kFormat, 0, transV ? 0u : 1u);
      // Descriptors differ only in the 14-bit start-address field; build each once and add (bytes >> 4).
      // MN-major: LBO = distance between the 64-element blocks along M / N, SBO = 1024 between 8-row groups along K.
      const uint64_t descQ = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemQ), transQ ? DPAD * 128 : 16, 1024);
      const uint64_t descK = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemK), transK ? kVHalfBytes : 16, 1024);
      const uint64_t descV = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemV), transV ? 16 : kSubTileBytes, 1024);

      // S(block) into buffer bf: per 64-column sub-tile of D, wait for K's sub-tile, four k-steps, release it
      auto issue_S = [&](uint32_t block, uint32_t bf) {
        const uint32_t d_tmem = tmem_base + bf * kBlockN;
#pragma unroll
        for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds) {
          mbar_wait(&k_full[ds], block & 1);
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (uint32_t kk = 0; kk < 4; ++kk) {
              // K-major: 16 elements = 32 B inside the 128 B swizzle row, 4 k-steps per 64-element sub-tile;
              // MN-major: 16 rows of D = 2048 B
              const uint32_t k_major_off = ds * kSubTileBytes + kk * 32;
              const uint32_t a_off = transQ ? (ds * 4 + kk) * 2048 : k_major_off;
              const uint32_t b_off = transK ? ds * kSubTileBytes + kk * 2048 : k_major_off;
              umma_ss(d_tmem, descQ + (a_off >> 4), descK + (b_off >> 4), idescS, (ds | kk) != 0);
            }
            umma_commit(&k_empty[ds]);
            if (ds == Cfg::kSubTiles - 1) umma_commit(&s_full[bf]);
          }
          __syncwarp();
        }
      };
      // O += P(block) V(block): two 64-key halves, each released as soon as its four k-steps have retired
      auto issue_PV = [&](uint32_t block, uint32_t bf) {
        const uint32_t d_tmem = tmem_base + Cfg::kTmemO;
        const uint32_t a_tmem = tmem_base + bf * kBlockN;
#pragma unroll
        for (uint32_t half = 0; half < 2; ++half) {
          mbar_wait(&v_full[half], block & 1);
          tc_fence_after();
          if (elect_one()) {
#pragma unroll
            for (uint32_t kk = 0; kk < 4; ++kk) {
              const uint32_t k = half * 4 + kk;
              // MN-major V: 16 keys = two 8-row groups of 1024 B, 64-wide column blocks kSubTileBytes apart (LBO);
              // K-major V^T: 16 keys = 32 B inside the swizzle row of this key half
              const uint32_t b_off = transV ? half * (DPAD * 128) + kk * 32 : k * 2048;
              umma_ts(d_tmem, a_tmem + k * 8, descV + (b_off >> 4), idescO, (block | k) != 0 ? 1u : 0u);
            }
            umma_commit(&v_empty[half]);
            if (half == 1) {
              umma_commit(o_full);
              if (block == num_blocks - 1) umma_commit(o_final);
            }
          }
          __syncwarp();
        }
      };

      // prologue: S(0) and S(1)
      mbar_wait(q_full, 0);
      for (uint32_t i = 0; i < kSBuffers && i < num_blocks; ++i) issue_S(i, i);

      for (uint32_t i = 0; i < num_blocks; ++i) {
        const uint32_t bf = i & 1, ph = (i >> 1) & 1;
        MFA_TRACE(2, i, 0);
        mbar_wait(&p_full[bf], ph);
        tc_fence_after();
        MFA_TRACE(2, i, 1);
        issue_PV(i, bf);
        // S(i+2) overwrites P(i) only after O += P V (i): the tensor pipe runs in order
        if (i + kSBuffers < num_blocks) issue_S(i + kSBuffers, bf);
        MFA_TRACE(2, i, 2);
      }
    }
  }

  // ---------------- teardown ----------------
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <uint32_t DPAD, bool kBF16, bool kTrace = false, bool kGeneric = false>
cudaError_t launch(const AttentionParams &p, cudaStream_t stream, long long *trace = nullptr) {
  using Cfg = Config<DPAD>;
  auto kernel = attention_forward_d256_tcgen05<DPAD, kBF16, kTrace, kGeneric>;
  cudaError_t e;
  if ((e = ensure_max_dynamic_smem(reinterpret_cast<const void *>(kernel), Cfg::kSmemBytes, current_device())) != cudaSuccess)
    return e;

  CUtensorMap mapQ, mapK, mapV;
  const bool tQ = kGeneric && p.transposed[sQ], tK = kGeneric && p.transposed[sK], tV = kGeneric && p.transposed[sV];
  e = tQ ? make_tensor_map_16bit_transposed(&mapQ, p.buf[sQ], p.R, p.D, p.batch, DPAD)
         : make_tensor_map_16bit(&mapQ, p.buf[sQ], p.R, p.D, p.batch, kTileM);
  if (e != cudaSuccess) return e;
  e = tK ? make_tensor_map_16bit_transposed(&mapK, p.buf[sK], p.C, p.D, p.batch, 64)
         : make_tensor_map_16bit(&mapK, p.buf[sK], p.C, p.D, p.batch, kBlockN);
  if (e != cudaSuccess) return e;
  e = tV ? make_tensor_map_16bit_transposed(&mapV, p.buf[sV], p.C, p.D, p.batch, DPAD)
         : make_tensor_map_16bit(&mapV, p.buf[sV], p.C, p.D, p.batch, 64);
  if (e != cudaSuccess) return e;
  const uint32_t tmask = (tQ ? 1u : 0u) | (tK ? 2u : 0u) | (tV ? 4u : 0u) | ((kGeneric && p.transposed[sO]) ? 8u : 0u);

  dim3 grid((p.R + kTileM - 1) / kTileM, p.batch);
  kernel<<<grid, kThreads, Cfg::kSmemBytes, stream>>>(mapQ, mapK, mapV, static_cast<float *>(p.buf[sO]), p.buf[sL],
                                                      p.R, p.C, p.D, p.scale_log2, p.prec[sL] == FP16 ? 1 : 0, tmask,
                                                      trace);
  return cudaGetLastError();
}

}  // namespace fwd256

// Debug entry (not in include/mfa_b200.h): the D <= 256 bf16 kernel with pipeline timestamps of CTA (0,0)
// (5 roles x 128 iterations x 8 slots of clock64()).  Used by scripts/trace_forward_d256.py.
cudaError_t launch_tcgen05_forward_d256_trace(const AttentionParams &p, cudaStream_t stream, long long *trace) {
  return fwd256::launch<256, true, true>(p, stream, trace);
}

// Forward with transposed operands (any D <= 256, D % 8 == 0): the layout-generic instantiations.
cudaError_t launch_tcgen05_forward_generic(const AttentionParams &p, cudaStream_t stream) {
  const bool bf16 = p.prec[sQ] == BF16;
  if (p.D <= 128)
    return bf16 ? fwd256::launch<128, true, false, true>(p, stream) : fwd256::launch<128, false, false, true>(p, stream);
  return bf16 ? fwd256::launch<256, true, false, true>(p, stream) : fwd256::launch<256, false, false, true>(p, stream);
}

void tcgen05_forward_generic_geometry(uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par, uint32_t *trav,
                                      uint32_t *head) {
  *threads = fwd256::kThreads;
  *smem_bytes = D <= 128 ? fwd256::Config<128>::kSmemBytes : fwd256::Config<256>::kSmemBytes;
  *par = fwd256::kTileM;
  *trav = fwd256::kBlockN;
  const uint32_t padded = (D + 7) / 8 * 8, block = D <= 128 ? 128u : 256u;
  *head = block < padded ? block : padded;
}

cudaError_t launch_tcgen05_forward_d256(const AttentionParams &p, cudaStream_t stream) {
  return p.prec[sQ] == BF16 ? fwd256::launch<256, true>(p, stream) : fwd256::launch<256, false>(p, stream);
}

}  // namespace mfa

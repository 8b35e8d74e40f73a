// FlashAttention forward for sm_100a: TMA -> shared memory -> tcgen05.mma -> TMEM.
//
// Replaces the reference's generated forward kernel (loopForward, AttentionKernel+Source.swift:158-200;
// outer product S = Q K^T, +OuterProduct.swift:18-487; online softmax, +Softmax.swift:228-324,334-505;
// accumulate O += P V, +Accumulate.swift:24-582) for 16-bit row-major operands.
//
// One CTA owns 256 query rows (two 128-row tcgen05 M-tiles that ping-pong on the tensor pipe) and
// walks the keys in blocks of 128.  Warp roles (384 threads):
//   warps 0-3   softmax for tile 0  (thread = one query row = one TMEM lane)
//   warps 4-7   softmax for tile 1
//   warp  8     MMA issuer (one elected thread issues every tcgen05.mma / commit); owns TMEM alloc
//   warp  9     TMA producer (Q once, then K and V stages)
//   warps 10-11 idle (they donate their registers via setmaxnreg)
// On-chip residency (the reference's "cache Q, O" rows, AttentionDescriptor+Parameters.swift:109-120,
// re-expressed for B200): Q tiles stay in SMEM for the whole traversal, O accumulators stay in TMEM,
// S lives in TMEM and is overwritten in place by P (16-bit) which feeds the second MMA straight from TMEM.
//   TMEM columns: [0,128) S0/P0  [128,256) S1/P1  [256,256+D) O0  [256+D,256+2D) O1
// Softmax bookkeeping follows Appendix A of SURVEY.md (log2 domain, L = m + log2 l) with one B200-specific
// change: the running max is only refreshed when it grows by more than 2^8 ("lazy rescale"), so the
// O *= correction pass over TMEM is rare; results are mathematically identical.
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
// Split-KV takes two launches: normalised partials in the library's workspace, then the combine_splits kernel, launched
// with programmatic stream serialisation so that it is resident when the attention kernel drains.  A one-launch form
// (every split CTA left its raw partial in the workspace, waited on a per-tile-pair arrival counter for its siblings
// and merged a slice of the rows; cooperative launch) measured slower on B200, one N = 4096, D = 128 bf16 head
// (profiles/r2_single_head_latency.jsonl), eager / CUDA graph: two launches 20.5 / 18.3 us, one launch 22.6 / 20.5 us --
// the merge is the same L2 traffic either way, and the second launch (hidden behind the first by programmatic stream
// serialisation) costs less than the cooperative launch plus the arrive-and-spin round trip.  It was removed, as was a
// form that reduced through distributed shared memory inside a thread-block cluster (37 us in round 1: only 15
// clusters of 8 CTAs are co-resident, DSMEM pulls at ~6 B/clk/SM).

namespace fwd {

using namespace ptx;

constexpr uint32_t kTileM = 128;         // rows per tcgen05 M-tile
constexpr uint32_t kTilesPerCta = 2;     // ping-pong tiles
constexpr uint32_t kBlockN = 128;        // keys per traversal block
constexpr uint32_t kSubTileBytes = 128 * 128;  // [128 rows][64 x 16-bit] = one 128B-swizzled TMA box
constexpr uint32_t kThreads = 384;
// setmaxnreg budget: the CTA is launched with floor(65536 / 384 / 8) * 8 = 168 registers per thread; the two
// softmax warpgroups grow to kSoftmaxRegs after the producer warpgroup has shrunk to kOtherRegs.  The sum
// must not exceed the launch allocation or the second setmaxnreg.inc never returns.
constexpr uint32_t kLaunchRegs = 168, kSoftmaxRegs = 208, kOtherRegs = 88;
static_assert(kSoftmaxRegs * 256 + kOtherRegs * 128 <= kLaunchRegs * kThreads, "setmaxnreg over-subscribed");
// kPoly (template parameter, from the parameter-table row the kernel was created from): of every 4 element pairs, how
// many take exp2 on the FMA pipe (exp2_poly2) instead of the MUFU pipe.  Swept on B200 (TFLOP/s at N = 4096, 64 heads;
// scripts/sweep.py repeats it):  D=128: 0 -> 1258, 1 -> 1241, 2 -> 1183;  D=64: 0 -> 729, 1 -> 765, 2 -> 737.  At D = 64
// the tensor pipe needs half as long per block, the MUFU pipe (16 ex2 / clk / SM) just as long, so taking a quarter of the
// exponentials off it pays; at D = 128 it only costs issue slots.
constexpr float kLazySumLimit = 256.0f;  // a half-row of P summing to <= 2^8 proves every element is <= 2^8

template <uint32_t DPAD>
struct Config {
  static constexpr uint32_t kSubTiles = DPAD / 64;                 // 64-element sub-tiles along D
  static constexpr uint32_t kTileBytes = kSubTiles * kSubTileBytes;  // one 128 x DPAD operand tile
  // K / V ring depth.  At D <= 64, A/B on one box (profiles/r2_sweep_fwd_stages_d64.jsonl, TFLOP/s, 4 | 3 | 2 stages):
  // N=4096 757 | 767 | 757, N=2048 714 | 716 | 713, N=512 532 | 541 | 530: depth barely matters (the softmax warps set the
  // pace), three stages are never worse and free 32 KB of shared memory.
  static constexpr uint32_t kStages = DPAD <= 64 ? 3 : 2;
  static constexpr uint32_t kSmemQ = 0;
  static constexpr uint32_t kSmemK = kSmemQ + kTilesPerCta * kTileBytes;
  static constexpr uint32_t kSmemV = kSmemK + kStages * kTileBytes;
  static constexpr uint32_t kSmemScratch = kSmemV + kStages * kTileBytes;  // epilogue transpose: 8 warps x 32 x 32 floats
  static constexpr uint32_t kSmemBar = kSmemScratch + 8 * 32 * 32 * 4;
  static constexpr uint32_t kNumBars = 2 + 4 * kStages + 6 * kTilesPerCta;
  static constexpr uint32_t kSmemTmemPtr = kSmemBar + kNumBars * 8;
  static constexpr uint32_t kSmemBytes = kSmemTmemPtr + 16 + 1024;  // + slack for manual 1024 B alignment
  static_assert(kSmemBytes <= 232448, "shared memory over budget");
  static constexpr uint32_t kTmemS = 0;
  static constexpr uint32_t kTmemO = 256;
  static constexpr uint32_t kTmemCols = 512;
};

struct Barriers {
  uint64_t *q_full, *q_empty, *k_full, *k_empty, *v_full, *v_empty, *s_full, *p_full, *o_full, *o_free, *pv_half;
};

// kTrace: debug instantiation that records clock64() at the pipeline hand-off points of CTA (0,0)
// (scripts/trace_forward.py); the production instantiation compiles all of it away.
constexpr uint32_t kTraceSlots = 8;  // per (role, iteration)
#define MFA_TRACE(role, iter, slot)                                                                   \
  do {                                                                                                \
    if (kTrace && trace != nullptr && blockIdx.x == 0 && lane == 0)                \
      trace[((role) * 64 + ((iter) & 63)) * kTraceSlots + (slot)] = clock64();                        \
  } while (0)

// item-level probes: roles 4 (tile 0 softmax), 5 (tile 1 softmax), 6 (MMA), indexed by the CTA's item counter
#define MFA_TRACE_ITEM(role, it, slot) MFA_TRACE(role, it, slot)

template <uint32_t DPAD, bool kBF16, uint32_t kPolyPairs, bool kTrace = false, bool kTmaStoreO = false>
__global__ void __launch_bounds__(kThreads, 1)
    attention_forward_tcgen05(const __grid_constant__ CUtensorMap mapQ, const __grid_constant__ CUtensorMap mapK,
                              const __grid_constant__ CUtensorMap mapV, const __grid_constant__ CUtensorMap mapO,
                              float *__restrict__ O, void *__restrict__ L,
                              uint32_t R, uint32_t C, uint32_t D, float scale_log2, int l_is_fp16,
                              uint32_t num_items, uint32_t pairs_per_head, uint32_t num_splits, uint32_t batch,
                              long long *__restrict__ trace) {
  // Persistent CTAs: one per SM, each walking the work items (head, 256-row tile pair) blockIdx.x,
  // blockIdx.x + gridDim.x, ...  Barrier phases are carried across items, so the producers (TMA, MMA) run ahead
  // into the next item while the softmax warps drain the current one; TMEM alloc, barrier init and descriptor
  // prefetch are paid once per SM instead of once per tile.
  using Cfg = Config<DPAD>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // Split-KV: when there are fewer (head, tile pair) items than SMs, the key axis of every item is cut into
  // num_splits equal ranges that become separate work items.  Each writes a normalised partial O and its L as if it
  // were a whole problem (O and L then point at scratch laid out [split][head][row]) and the combine_splits kernel
  // merges them.
  const uint32_t total_blocks = (C + kBlockN - 1) / kBlockN;
  const uint32_t num_blocks = total_blocks / num_splits;  // key blocks per work item (host guarantees divisibility)

  uint64_t *bars = reinterpret_cast<uint64_t *>(smem + Cfg::kSmemBar);
  Barriers b;
  b.q_full = bars;
  b.q_empty = bars + 1;                    // every S MMA of the current item has read Q
  b.k_full = bars + 2;
  b.k_empty = b.k_full + Cfg::kStages;
  b.v_full = b.k_empty + Cfg::kStages;
  b.v_empty = b.v_full + Cfg::kStages;
  b.s_full = b.v_empty + Cfg::kStages;
  b.p_full = b.s_full + kTilesPerCta;      // [tile][column half]: P columns 0-63 / 64-127 written
  b.o_full = b.p_full + 2 * kTilesPerCta;
  b.o_free = b.o_full + kTilesPerCta;      // [tile] the epilogue has read O out of TMEM (128 arrivals)
  b.pv_half = b.o_free + kTilesPerCta;     // [tile] O += P V over the first 64 keys of the block is done
  uint32_t *tmem_ptr_smem = reinterpret_cast<uint32_t *>(smem + Cfg::kSmemTmemPtr);

  // ---------------- one-time setup ----------------
  if (threadIdx.x == 0) {
    mbar_init(b.q_full, 1);
    mbar_init(b.q_empty, 1);
    for (uint32_t s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&b.k_full[s], 1);
      mbar_init(&b.k_empty[s], 1);
      mbar_init(&b.v_full[s], 1);
      mbar_init(&b.v_empty[s], 1);
    }
    for (uint32_t t = 0; t < kTilesPerCta; ++t) {
      mbar_init(&b.s_full[t], 1);
      mbar_init(&b.p_full[2 * t], kTileM);
      mbar_init(&b.p_full[2 * t + 1], kTileM);
      mbar_init(&b.o_full[t], 1);
      mbar_init(&b.o_free[t], kTileM);
      mbar_init(&b.pv_half[t], 1);
    }
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
  // split-KV: let the combine kernel (launched with programmatic stream serialisation) be set up now; its
  // griddepcontrol.wait still holds it until this grid has completed and flushed
  if (num_splits > 1) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp < 8) {
    // =====================================================================================
    // softmax warps: thread <-> query row <-> TMEM lane
    // =====================================================================================
    setmaxnreg_inc<kSoftmaxRegs>();
    const uint32_t t = warp >> 2;                      // tile
    const uint32_t row_in_tile = (warp & 3) * 32 + lane;
    const uint32_t lane_addr = ((warp & 3) * 32) << 16;  // this warp's TMEM lane quarter
    const uint32_t tS = tmem_base + lane_addr + Cfg::kTmemS + t * kBlockN;
    const uint32_t tO = tmem_base + lane_addr + Cfg::kTmemO + t * DPAD;

    const uint32_t tail_cols = C - (total_blocks - 1) * kBlockN;  // valid columns in the last key block

    for (uint32_t item = blockIdx.x, it = 0; item < num_items; item += gridDim.x, ++it) {
    const uint32_t split = item % num_splits;
    // output slot; split-KV lays partials out as [split][head]
    const uint32_t head = (item / num_splits) / pairs_per_head + split * batch;
    const uint32_t q_row0 = ((item / num_splits) % pairs_per_head) * (kTileM * kTilesPerCta);
    const uint32_t key_block0 = split * num_blocks;
    const uint32_t g0 = it * num_blocks;  // key blocks this CTA has processed before this item (barrier phases)
    float m = -FLT_MAX;  // running max, log2 domain   (AttentionKernel+Caching.swift:310)
    float l = 0.f;       // running sum
    MFA_TRACE_ITEM(warp == 0 ? 4 : (warp == 4 ? 5 : 7), it, 0);

    for (uint32_t j = 0; j < num_blocks; ++j) {
      mbar_wait(&b.s_full[t], (g0 + j) & 1);
      tc_fence_after();
      MFA_TRACE(warp == 0 ? 0 : (warp == 4 ? 1 : 5), j, 0);

      float s[kBlockN];
#pragma unroll
      for (uint32_t c = 0; c < kBlockN; c += 32) tmem_ld32(tS + c, *reinterpret_cast<uint32_t(*)[32]>(&s[c]));
      tc_wait_ld();
      MFA_TRACE(warp == 0 ? 0 : (warp == 4 ? 1 : 5), j, 1);

      // edge mask (maskAttentionMatrixEdge, AttentionKernel+Softmax.swift:228-260)
      if (key_block0 + j == total_blocks - 1 && tail_cols < kBlockN) {
#pragma unroll
        for (uint32_t c = 0; c < kBlockN; ++c)
          if (c >= tail_cols) s[c] = -INFINITY;
      }

      // The reference tracks the exact running row max every block (onlineReduceMaximum / onlineCorrectO,
      // +Softmax.swift:267-301).  Here the max is refreshed lazily: P is computed against the current (possibly
      // stale) m straight away, and only if a half-row of P sums to more than 2^8 -- i.e. some element could
      // exceed 2^8, or m was never set -- does the thread group fall back to the exact path: reduce the row max of
      // that half, wait for every O += P V issued so far, rescale O and l, and recompute the half.  With m lagging
      // the true max by at most 8 (log2), P <= 2^8 keeps full FP32 / 16-bit accuracy, and the 128-element max
      // reduction disappears from the common path; the result is mathematically identical.
#pragma unroll
      for (uint32_t half = 0; half < 2; ++half) {
        const uint32_t c0 = half * (kBlockN / 2);
        uint32_t packed[32];
        // The MUFU pipe (16 ex2 / clk / SM) needs as long for a 128 x 128 block as the tensor pipe needs for its two
        // GEMMs, so kPolyPairs of every 4 element pairs take exp2 on the FMA pipe instead (exp2_poly2).
        float half_sum;
        if (half == 0 && j == 0) {
          half_sum = INFINITY;  // m is not set yet: the item's very first half goes straight to the exact path
        } else {
          float2 sum2 = make_float2(0.f, 0.f);
          const float2 scale2 = make_float2(scale_log2, scale_log2), negm2 = make_float2(-m, -m);
#pragma unroll
          for (uint32_t i = 0; i < 32; ++i) {
            const float2 x = ffma2(make_float2(s[c0 + 2 * i], s[c0 + 2 * i + 1]), scale2, negm2);
            float2 pr;
            if (kPolyPairs > 0 && (i & 3) < kPolyPairs) {
              pr = exp2_poly2(x);
            } else {
              pr.x = ex2_approx(x.x);
              pr.y = ex2_approx(x.y);
            }
            packed[i] = kBF16 ? pack_bf16x2(pr.x, pr.y) : pack_f16x2(pr.x, pr.y);
            sum2 = fadd2(sum2, pr);
          }
          half_sum = sum2.x + sum2.y;
        }
        if (__any_sync(0xffffffffu, !(half_sum <= kLazySumLimit))) {  // also catches inf / NaN
          // ---- exact path (rare) ----
          float mx0 = s[c0], mx1 = s[c0 + 1], mx2 = s[c0 + 2], mx3 = s[c0 + 3];
#pragma unroll
          for (uint32_t c = 4; c < kBlockN / 2; c += 4) {
            mx0 = fmaxf(mx0, s[c0 + c]);
            mx1 = fmaxf(mx1, s[c0 + c + 1]);
            mx2 = fmaxf(mx2, s[c0 + c + 2]);
            mx3 = fmaxf(mx3, s[c0 + c + 3]);
          }
          const float m_new = fmaxf(m, fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3)) * scale_log2);
          if (j > 0 || half > 0) {
            // everything already handed to the MMA warp must have been accumulated before O is rescaled:
            // the first half of this block (pv_half) or the whole previous block (o_full)
            if (half > 0)
              mbar_wait(&b.pv_half[t], (g0 + j) & 1);
            else
              mbar_wait(&b.o_full[t], (g0 + j - 1) & 1);
            tc_fence_after();
            const float correction = ex2_approx(m - m_new);
#pragma unroll
            for (uint32_t c = 0; c < DPAD; c += 32) {
              uint32_t o[32];
              tmem_ld32(tO + c, o);
              tc_wait_ld();
#pragma unroll
              for (uint32_t i = 0; i < 32; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * correction);
              tmem_st32(tO + c, o);
            }
            l *= correction;
          }
          m = m_new;
          float sum0 = 0.f, sum1 = 0.f;
#pragma unroll
          for (uint32_t i = 0; i < 32; ++i) {
            const float p0 = ex2_approx(fmaf(s[c0 + 2 * i], scale_log2, -m));
            const float p1 = ex2_approx(fmaf(s[c0 + 2 * i + 1], scale_log2, -m));
            packed[i] = kBF16 ? pack_bf16x2(p0, p1) : pack_f16x2(p0, p1);
            sum0 += p0;
            sum1 += p1;
          }
          half_sum = sum0 + sum1;
        }
        l += half_sum;
        // P (16-bit) over S: keys [64 half, 64 half + 64) -> columns [32 half, 32 half + 32)
        tmem_st32(tS + half * 32, packed);
        tc_wait_st();
        tc_fence_before();
        // the first 64 columns of P are released on their own so that the MMA warp starts O += P V on them while
        // the MUFU pipe works through the other half
        mbar_arrive(&b.p_full[2 * t + half]);
        MFA_TRACE(warp == 0 ? 0 : (warp == 4 ? 1 : 5), j, 2 + half);
      }
      MFA_TRACE(warp == 0 ? 0 : (warp == 4 ? 1 : 5), j, 4);
    }

    {
      // ---------------- epilogue: O / l -> global (FP32), L = m + log2(l) ----------------
      MFA_TRACE_ITEM(warp == 0 ? 4 : (warp == 4 ? 5 : 7), it, 1);
      mbar_wait(&b.o_full[t], (g0 + num_blocks - 1) & 1);
      tc_fence_after();
      MFA_TRACE_ITEM(warp == 0 ? 4 : (warp == 4 ? 5 : 7), it, 2);
      const uint32_t row = q_row0 + t * kTileM + row_in_tile;
      const float out_scale = 1.0f / l;
      // TMEM hands every thread one row; storing rows straight from registers would touch 32 different cache
      // lines per warp store.  Each warp therefore transposes 32 x 32 chunks through a private XOR-swizzled scratch
      // tile in shared memory (128-bit accesses, conflict-free both ways) and writes four full 128 B lines per store.
      const uint32_t scratch = smem_u32(smem + Cfg::kSmemScratch) + warp * (32 * 8 * 16);  // this warp's 4 KB tile
      const uint32_t warp_row0 = q_row0 + t * kTileM + (warp & 3) * 32;
      float *o_base = O + (static_cast<size_t>(head) * R + warp_row0) * D;
      const uint32_t sub_row = lane >> 3, quad = lane & 7;  // transposed view: 4 rows x 8 float4 per warp access
      // Short items: the transposed chunk leaves through the TMA (cp.async.bulk.tensor store from the scratch tile,
      // whose XOR pattern IS the 128-byte swizzle of a [32 rows][32 floats] box): the warp does not wait for the global
      // writes -- it only waits, before rewriting the scratch tile, until the previous chunk's store has READ it.  Rows past
      // R and columns past D are clipped by the tensor map.  (Generic-proxy stores from registers, the other instantiation,
      // hold the warp until every line has left the SM.)  With one scratch tile per warp the wait for the previous chunk's
      // read is partly exposed, and at 32 blocks per item the epilogue is too small a share to matter, so the launcher picks
      // this instantiation for short items only (A/B on one box, TFLOP/s, this build | register stores: N=512 D=64 525 | 501,
      // N=1024 D=128 833 | 780, N=2048 D=64 FP16 712 | 702; N=4096 D=128 equal: profiles/r2_sweep_fwd_tma_store.jsonl).
      // (A second scratch tile per warp at D <= 64, so that the two chunks never wait for each other, measured the same
      // within 0.5 %: profiles/r2_sweep_fwd_two_tiles.jsonl -- not kept.)
      constexpr bool kTmaStore = kTmaStoreO;  // (its own instantiation: as a run-time branch it cost the long-item case 1.8 %)
  #pragma unroll
      for (uint32_t c = 0; c < DPAD; c += 32) {
        uint32_t o[32];
        tmem_ld32(tO + c, o);
        tc_wait_ld();
        if constexpr (kTmaStore) {
          if (lane == 0) tma_store_wait_read_all();  // (also covers the previous item's last chunk)
          __syncwarp();
        }
  #pragma unroll
        for (uint32_t j = 0; j < 8; ++j)
          sts_f32x4(scratch + (lane * 8 + (j ^ (lane & 7))) * 16,
                    make_float4(__uint_as_float(o[4 * j]) * out_scale, __uint_as_float(o[4 * j + 1]) * out_scale,
                                __uint_as_float(o[4 * j + 2]) * out_scale, __uint_as_float(o[4 * j + 3]) * out_scale));
        if constexpr (kTmaStore) {
          fence_proxy_async_smem();  // this lane's writes -> visible to the async proxy
          __syncwarp();
          if (lane == 0 && c < D) {
            tma_store_3d(&mapO, scratch, static_cast<int32_t>(c), static_cast<int32_t>(warp_row0), static_cast<int32_t>(head));
            tma_store_commit();
          }
        } else {
          __syncwarp();
          // read the whole transposed chunk into distinct registers BEFORE the first store: a store keeps its source
          // registers busy until the data has left the SM, so reusing a handful of registers would serialise the
          // stores on memory latency (measured: 11k cycles per tile epilogue)
          float4 v[8];
  #pragma unroll
          for (uint32_t i = 0; i < 8; ++i) {
            const uint32_t r = 4 * i + sub_row;
            v[i] = lds_f32x4(scratch + (r * 8 + (quad ^ (r & 7))) * 16);
          }
          if (c + 4 * quad < D) {  // D % 8 == 0: a float4 is either fully inside or fully outside
  #pragma unroll
            for (uint32_t i = 0; i < 8; ++i) {
              const uint32_t r = 4 * i + sub_row;
              if (warp_row0 + r < R) *reinterpret_cast<float4 *>(o_base + static_cast<size_t>(r) * D + c + 4 * quad) = v[i];
            }
          }
          __syncwarp();
        }
      }
      if (row < R && L != nullptr) {
        const float lse2 = m + log2f(l);  // AttentionKernel+Caching.swift:373-377
        const size_t idx = static_cast<size_t>(head) * R + row;
        if (l_is_fp16)
          reinterpret_cast<__half *>(L)[idx] = __float2half_rn(lse2);
        else
          reinterpret_cast<float *>(L)[idx] = lse2;
      }
    }
    // O of this tile is out of TMEM: the next item's first O = P V (accumulate off) may overwrite it
    tc_fence_before();
    mbar_arrive(&b.o_free[t]);
    MFA_TRACE_ITEM(warp == 0 ? 4 : (warp == 4 ? 5 : 7), it, 3);
    }  // work items
    if (kTmaStoreO && lane == 0) tma_store_wait_all();  // the CTA's shared memory outlives its stores
  } else {
    setmaxnreg_dec<kOtherRegs>();
    // Both producer warps run their control flow warp-wide and hand exactly one elected lane to the
    // TMA / tcgen05 instructions: operands stay in uniform registers and the issue loops are branch-free.
    if (warp == 9) {
      // ===================================================================================
      // TMA producer
      // ===================================================================================
      for (uint32_t item = blockIdx.x, it = 0; item < num_items; item += gridDim.x, ++it) {
      const uint32_t head = (item / num_splits) / pairs_per_head;
      const uint32_t q_row0 = ((item / num_splits) % pairs_per_head) * (kTileM * kTilesPerCta);
      const uint32_t key_block0 = (item % num_splits) * num_blocks;
      const uint32_t g0 = it * num_blocks;
      mbar_wait(b.q_empty, (it & 1) ^ 1);  // the previous item's S MMAs are done with the Q tiles
      if (elect_one()) {
        mbar_arrive_expect_tx(b.q_full, kTilesPerCta * Cfg::kTileBytes);
#pragma unroll
        for (uint32_t t = 0; t < kTilesPerCta; ++t)
#pragma unroll
          for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
            tma_load_3d(smem + Cfg::kSmemQ + t * Cfg::kTileBytes + ds * kSubTileBytes, &mapQ, b.q_full, ds * 64,
                        q_row0 + t * kTileM, head);
      }
      for (uint32_t j = 0; j < num_blocks; ++j) {
        const uint32_t stage = (g0 + j) % Cfg::kStages, phase = ((g0 + j) / Cfg::kStages) & 1;
        MFA_TRACE(3, j, 0);
        mbar_wait(&b.k_empty[stage], phase ^ 1);
        MFA_TRACE(3, j, 1);
        if (elect_one()) {
          mbar_arrive_expect_tx(&b.k_full[stage], Cfg::kTileBytes);
#pragma unroll
          for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
            tma_load_3d(smem + Cfg::kSmemK + stage * Cfg::kTileBytes + ds * kSubTileBytes, &mapK, &b.k_full[stage],
                        ds * 64, (key_block0 + j) * kBlockN, head);
        }
        mbar_wait(&b.v_empty[stage], phase ^ 1);
        MFA_TRACE(3, j, 2);
        if (elect_one()) {
          mbar_arrive_expect_tx(&b.v_full[stage], Cfg::kTileBytes);
#pragma unroll
          for (uint32_t ds = 0; ds < Cfg::kSubTiles; ++ds)
            tma_load_3d(smem + Cfg::kSmemV + stage * Cfg::kTileBytes + ds * kSubTileBytes, &mapV, &b.v_full[stage],
                        ds * 64, (key_block0 + j) * kBlockN, head);
        }
      }
      }  // work items
    } else if (warp == 8) {
      // ===================================================================================
      // MMA issuer
      // ===================================================================================
      constexpr uint32_t kFormat = kBF16 ? 1u : 0u;
      // S[128 x 128] = Q[128 x D] . K[128 x D]^T : A and B both K-major
      constexpr uint32_t idescS = make_idesc_f16(kTileM, kBlockN, kFormat, 0, 0);
      // O[128 x DPAD] += P[128 x 128] . V[128 x DPAD] : A from TMEM, B (= V, [key][d]) is MN-major
      constexpr uint32_t idescO = make_idesc_f16(kTileM, DPAD, kFormat, 0, 1);
      // Descriptors differ only in the 14-bit start-address field; build each once and add (bytes >> 4).
      const uint64_t descQ = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemQ), 16, 1024);
      const uint64_t descK = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemK), 16, 1024);
      const uint64_t descV = make_smem_desc_sw128(smem_u32(smem + Cfg::kSmemV), kSubTileBytes, 1024);

      // every tcgen05.mma / commit below is issued by the one elected lane
      auto issue_S = [&](uint32_t t, uint32_t stage) {
        const uint32_t d_tmem = tmem_base + Cfg::kTmemS + t * kBlockN;
        const uint64_t a0 = descQ + ((t * Cfg::kTileBytes) >> 4);
        const uint64_t b0 = descK + ((stage * Cfg::kTileBytes) >> 4);
#pragma unroll
        for (uint32_t k = 0; k < DPAD / 16; ++k) {
          // 16 elements = 32 B inside the 128 B swizzle row; 4 k-steps per 64-element sub-tile
          const uint32_t off = ((k >> 2) * kSubTileBytes + (k & 3) * 32) >> 4;
          umma_ss(d_tmem, a0 + off, b0 + off, idescS, k > 0);
        }
      };
      // half 0: keys 0-63 of the block (P columns 0-63), half 1: keys 64-127
      auto issue_PV = [&](uint32_t t, uint32_t half, uint32_t stage, uint32_t accumulate) {
        const uint32_t d_tmem = tmem_base + Cfg::kTmemO + t * DPAD;
        const uint32_t a_tmem = tmem_base + Cfg::kTmemS + t * kBlockN;
        const uint64_t b0 = descV + ((stage * Cfg::kTileBytes) >> 4);
#pragma unroll
        for (uint32_t kk = 0; kk < kBlockN / 32; ++kk) {
          const uint32_t k = half * (kBlockN / 32) + kk;
          // 16 keys = two 8-row groups of 1024 B; 64-wide column blocks are kSubTileBytes apart (LBO)
          umma_ts(d_tmem, a_tmem + k * 8, b0 + ((k * 2048) >> 4), idescO, k > 0 ? 1u : accumulate);
        }
      };

      for (uint32_t item = blockIdx.x, it = 0; item < num_items; item += gridDim.x, ++it) {
      const uint32_t g0 = it * num_blocks;
      {
        // first S of the item: overlaps the softmax warps' epilogue of the previous item (S/P regions are free
        // once the previous item's last O += P V has been issued: the tensor pipe runs in order)
        const uint32_t stage0 = g0 % Cfg::kStages, phase0 = (g0 / Cfg::kStages) & 1;
        MFA_TRACE_ITEM(6, it, 0);
        mbar_wait(b.q_full, it & 1);
        mbar_wait(&b.k_full[stage0], phase0);
        tc_fence_after();
        if (elect_one()) {
          issue_S(0, stage0);
          umma_commit(&b.s_full[0]);
          issue_S(1, stage0);
          umma_commit(&b.s_full[1]);
          umma_commit(&b.k_empty[stage0]);
          if (num_blocks == 1) umma_commit(b.q_empty);
        }
        __syncwarp();
        MFA_TRACE_ITEM(6, it, 1);
      }

      for (uint32_t j = 0; j < num_blocks; ++j) {
        const uint32_t g = g0 + j;
        const uint32_t stage = g % Cfg::kStages, phase = (g / Cfg::kStages) & 1;
        const uint32_t nstage = (g + 1) % Cfg::kStages, nphase = ((g + 1) / Cfg::kStages) & 1;
        const bool has_next = j + 1 < num_blocks;
        mbar_wait(&b.v_full[stage], phase);
        MFA_TRACE(2, j, 0);
#pragma unroll
        for (uint32_t t = 0; t < kTilesPerCta; ++t) {
          mbar_wait(&b.p_full[2 * t], g & 1);
          // the previous item's epilogue must have read O out before accumulate-off overwrites it
          if (j == 0 && it > 0) mbar_wait(&b.o_free[t], (it - 1) & 1);
          tc_fence_after();
          if (elect_one()) {
            issue_PV(t, 0, stage, j > 0 ? 1u : 0u);
            umma_commit(&b.pv_half[t]);
          }
          __syncwarp();
          mbar_wait(&b.p_full[2 * t + 1], g & 1);
          if (t == 0) MFA_TRACE(2, j, 2);
          if (t == 0 && has_next) mbar_wait(&b.k_full[nstage], nphase);
          tc_fence_after();
          MFA_TRACE(2, j, 1 + 3 * t);
          if (elect_one()) {
            issue_PV(t, 1, stage, 1u);
            umma_commit(&b.o_full[t]);
            if (t == kTilesPerCta - 1) umma_commit(&b.v_empty[stage]);
            if (has_next) {
              issue_S(t, nstage);
              umma_commit(&b.s_full[t]);
              if (t == kTilesPerCta - 1) {
                umma_commit(&b.k_empty[nstage]);
                if (j + 2 == num_blocks) umma_commit(b.q_empty);  // that was the item's last read of Q
              }
            }
          }
          __syncwarp();
          MFA_TRACE(2, j, 3 + 3 * t);
        }
      }
      MFA_TRACE_ITEM(6, it, 2);
      }  // work items
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

// Merges the num_splits partial results of split-KV: L = log2 sum_s 2^L_s,  O = sum_s 2^(L_s - L) O_s.
// One thread per (row, 4 columns); partials are [split][head][row][D] FP32 and [split][head][row] FP32.  Every load of
// a thread is issued before the first use (the partials sit in L2; a dependent chain of num_splits round trips was
// 3x slower).  Launched with programmatic stream serialisation: the grid is set up while the attention kernel drains
// and griddepcontrol.wait holds it until that kernel's writes are visible.
template <uint32_t kMaxSplits>
__global__ void __launch_bounds__(128)
    combine_splits(const float *__restrict__ O_part, const float *__restrict__ L_part, float *__restrict__ O,
                   void *__restrict__ L, uint32_t rows_total, uint32_t D, uint32_t num_splits, int l_is_fp16) {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  const uint32_t quads_per_row = D / 4;
  const uint64_t idx = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const uint64_t row = idx / quads_per_row;
  const uint32_t quad = static_cast<uint32_t>(idx % quads_per_row);
  if (row >= rows_total) return;
  float ls[kMaxSplits];
  float4 v[kMaxSplits];
#pragma unroll
  for (uint32_t s = 0; s < kMaxSplits; ++s) {
    ls[s] = -INFINITY;
    v[s] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (s < num_splits) {
      ls[s] = __ldcg(L_part + static_cast<uint64_t>(s) * rows_total + row);
      v[s] = __ldcg(reinterpret_cast<const float4 *>(O_part + (static_cast<uint64_t>(s) * rows_total + row) * D) + quad);
    }
  }
  float lmax = ls[0];
#pragma unroll
  for (uint32_t s = 1; s < kMaxSplits; ++s) lmax = fmaxf(lmax, ls[s]);
  float denom = 0.f;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (uint32_t s = 0; s < kMaxSplits; ++s) {
    const float w = exp2f(ls[s] - lmax);  // 0 for the unused slots
    denom += w;
    acc.x = fmaf(w, v[s].x, acc.x);
    acc.y = fmaf(w, v[s].y, acc.y);
    acc.z = fmaf(w, v[s].z, acc.z);
    acc.w = fmaf(w, v[s].w, acc.w);
  }
  const float inv = 1.0f / denom;
  *reinterpret_cast<float4 *>(O + row * D + 4 * quad) = make_float4(acc.x * inv, acc.y * inv, acc.z * inv, acc.w * inv);
  if (quad == 0 && L != nullptr) {
    const float lse = lmax + log2f(denom);
    if (l_is_fp16)
      reinterpret_cast<__half *>(L)[row] = __float2half_rn(lse);
    else
      reinterpret_cast<float *>(L)[row] = lse;
  }
}

// how many key ranges to cut every item into: only when the SMs would otherwise idle, only into equal ranges of at
// least four key blocks (shorter ranges are dominated by the per-item prologue / epilogue)
// (min_blocks and max_splits are the row's tuning columns; min_blocks = 0 turns splitting off)
static uint32_t choose_splits(uint32_t items, uint32_t total_blocks, uint32_t sm_count, uint32_t min_blocks,
                              uint32_t max_splits) {
  if (items * 2 > sm_count || min_blocks == 0) return 1;
  if (max_splits > 16) max_splits = 16;
  const uint32_t target = sm_count / items;
  uint32_t best = 1;
  for (uint32_t s = 2; s <= target && s <= max_splits; ++s)
    if (total_blocks % s == 0 && total_blocks / s >= min_blocks) best = s;
  return best;
}

template <uint32_t DPAD, bool kBF16, uint32_t kPoly, bool kTrace = false>
cudaError_t launch(const AttentionParams &p, cudaStream_t stream, long long *trace = nullptr) {
  using Cfg = Config<DPAD>;
  auto kernel = attention_forward_tcgen05<DPAD, kBF16, kPoly, kTrace, false>;
  const int device = current_device();
  cudaError_t e;
  if ((e = ensure_max_dynamic_smem(reinterpret_cast<const void *>(kernel), Cfg::kSmemBytes, device)) != cudaSuccess) return e;

  CUtensorMap mapQ, mapK, mapV, mapO;  // mapO: FP32 [heads][R][D] in boxes of 32 columns x 32 rows (the epilogue's stores)
  if ((e = make_tensor_map_16bit(&mapQ, p.buf[sQ], p.R, p.D, p.batch, kTileM)) != cudaSuccess) return e;
  if ((e = make_tensor_map_16bit(&mapK, p.buf[sK], p.C, p.D, p.batch, kBlockN)) != cudaSuccess) return e;
  if ((e = make_tensor_map_16bit(&mapV, p.buf[sV], p.C, p.D, p.batch, kBlockN)) != cudaSuccess) return e;

  const uint32_t pairs_per_head = (p.R + kTileM * kTilesPerCta - 1) / (kTileM * kTilesPerCta);
  const uint32_t num_items = pairs_per_head * p.batch;
  const uint32_t sm_count = device_sm_count(device);
  const uint32_t total_blocks = (p.C + kBlockN - 1) / kBlockN;
  const int l_is_fp16 = p.prec[sL] == FP16 ? 1 : 0;

  const uint32_t splits = choose_splits(num_items, total_blocks, sm_count, p.split_min_blocks, p.split_max);
  // short items (many epilogues per unit of work): O leaves through TMA stores; long items keep the register stores
  // (split single heads measured 1-2 % slower with it: one item per CTA, nothing to overlap the store with)
  if constexpr (!kTrace) {
    if (splits == 1 && total_blocks <= 16) {
    kernel = attention_forward_tcgen05<DPAD, kBF16, kPoly, kTrace, true>;
    if ((e = ensure_max_dynamic_smem(reinterpret_cast<const void *>(kernel), Cfg::kSmemBytes, device)) != cudaSuccess) return e;
    }
  }
  if (splits == 1) {
    if ((e = make_tensor_map_f32(&mapO, p.buf[sO], p.R, p.D, p.batch, 32)) != cudaSuccess) return e;
    const uint32_t grid = num_items < sm_count ? num_items : sm_count;
    kernel<<<grid, kThreads, Cfg::kSmemBytes, stream>>>(mapQ, mapK, mapV, mapO, static_cast<float *>(p.buf[sO]), p.buf[sL],
                                                        p.R, p.C, p.D, p.scale_log2, l_is_fp16, num_items,
                                                        pairs_per_head, 1u, p.batch, trace);
    return cudaGetLastError();
  }

  // ---- split-KV: normalised partial O / L per split ([split][head][row]) in the library's per-(device, stream)
  // workspace, then the combine kernel
  const uint32_t split_items = num_items * splits;  // <= sm_count by construction of choose_splits
  const uint64_t rows_total = static_cast<uint64_t>(p.batch) * p.R;
  const size_t o_bytes = static_cast<size_t>(splits) * rows_total * p.D * sizeof(float);
  const size_t l_bytes = static_cast<size_t>(splits) * rows_total * sizeof(float);
  void *ws = nullptr;
  if ((e = workspace_for(device, stream, o_bytes + l_bytes, &ws)) != cudaSuccess) return e;
  float *scratch = static_cast<float *>(ws);
  float *L_part = scratch + static_cast<size_t>(splits) * rows_total * p.D;
  // partials are laid out [split][head][row][D]: one tensor map over splits x batch "heads"
  if ((e = make_tensor_map_f32(&mapO, scratch, p.R, p.D, p.batch * splits, 32)) != cudaSuccess) return e;
  const uint32_t grid = split_items < sm_count ? split_items : sm_count;
  kernel<<<grid, kThreads, Cfg::kSmemBytes, stream>>>(mapQ, mapK, mapV, mapO, scratch, L_part, p.R, p.C, p.D, p.scale_log2,
                                                      0, split_items, pairs_per_head, splits, p.batch, trace);
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  const uint64_t threads = rows_total * (p.D / 4);
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cudaLaunchConfig_t config = {};
  config.gridDim = dim3(static_cast<uint32_t>((threads + 127) / 128), 1, 1);
  config.blockDim = dim3(128, 1, 1);
  config.stream = stream;
  config.attrs = &attr;
  config.numAttrs = 1;
  auto combine = splits <= 4 ? combine_splits<4> : (splits <= 8 ? combine_splits<8> : combine_splits<16>);
  e = cudaLaunchKernelEx(&config, combine, static_cast<const float *>(scratch), static_cast<const float *>(L_part),
                         static_cast<float *>(p.buf[sO]), p.buf[sL], static_cast<uint32_t>(rows_total), p.D, splits,
                         l_is_fp16);
  return e == cudaSuccess ? cudaGetLastError() : e;
}

}  // namespace fwd

uint32_t tcgen05_forward_max_head() { return 256; }

// Transposed operands are served by the layout-generic kernel (tcgen05_forward_d256.cu) when TMA can address them: a
// transposed operand's row pitch is its sequence length, which must then be a multiple of 8 elements (16 bytes).
bool tcgen05_forward_transposes_ok(uint32_t R, uint32_t C, bool tQ, bool tK, bool tV) {
  return (!tQ || R % 8 == 0) && (!tK || C % 8 == 0) && (!tV || C % 8 == 0);
}

bool tcgen05_forward_supported(const AttentionParams &p) {
  return (p.prec[sQ] == FP16 || p.prec[sQ] == BF16) && p.prec[sK] == p.prec[sQ] && p.prec[sV] == p.prec[sQ] &&
         p.prec[sO] == FP32 && p.D % 8 == 0 && p.D <= tcgen05_forward_max_head() &&
         tcgen05_forward_transposes_ok(p.R, p.C, p.transposed[sQ], p.transposed[sK], p.transposed[sV]);
}

cudaError_t launch_tcgen05_forward(const AttentionParams &p, cudaStream_t stream) {
  const bool bf16 = p.prec[sQ] == BF16;
  // the row's exp2 column selects the instantiation (kernel creation has checked the range)
#define MFA_FWD_DISPATCH(DPAD_)                                                                              \
  switch (p.exp2_fma_quarters) {                                                                             \
    case 0: return bf16 ? fwd::launch<DPAD_, true, 0>(p, stream) : fwd::launch<DPAD_, false, 0>(p, stream);  \
    case 1: return bf16 ? fwd::launch<DPAD_, true, 1>(p, stream) : fwd::launch<DPAD_, false, 1>(p, stream);  \
    default: return bf16 ? fwd::launch<DPAD_, true, 2>(p, stream) : fwd::launch<DPAD_, false, 2>(p, stream); \
  }
  if (p.D <= 64) {
    MFA_FWD_DISPATCH(64)
  }
  MFA_FWD_DISPATCH(128)
#undef MFA_FWD_DISPATCH
}

// Debug entry (not in include/mfa_b200.h): the D=128 bf16 forward with pipeline timestamps of CTA (0,0)
// written to `trace` (3 roles x 64 iterations x 8 slots of clock64()).  Used by scripts/trace_forward.py.
cudaError_t launch_tcgen05_forward_trace(const AttentionParams &p, cudaStream_t stream, long long *trace) {
  return fwd::launch<128, true, 0, true>(p, stream, trace);
}

// 1 launch, or 2 (attention + combine) when split-KV engages for this problem size
uint32_t tcgen05_forward_launch_count(uint32_t R, uint32_t C, uint32_t batch, uint32_t min_blocks, uint32_t max_splits) {
  const uint32_t sm_count = device_sm_count(current_device());
  const uint32_t pairs = (R + fwd::kTileM * fwd::kTilesPerCta - 1) / (fwd::kTileM * fwd::kTilesPerCta);
  const uint32_t blocks = (C + fwd::kBlockN - 1) / fwd::kBlockN;
  return fwd::choose_splits(pairs * batch, blocks, sm_count, min_blocks, max_splits) == 1 ? 1 : 2;
}

void tcgen05_forward_geometry(uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par, uint32_t *trav,
                              uint32_t *head) {
  *threads = fwd::kThreads;
  *smem_bytes = D <= 64 ? fwd::Config<64>::kSmemBytes : fwd::Config<128>::kSmemBytes;
  *par = fwd::kTileM * fwd::kTilesPerCta;
  *trav = fwd::kBlockN;
  *head = D <= 64 ? 64 : 128;
  const uint32_t padded = (D + 7) / 8 * 8;
  if (*head > padded) *head = padded;
}

}  // namespace mfa

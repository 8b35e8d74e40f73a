// Tensor-core GEMM for sm_100a: C (+)= A . B with A and B both FP16 or both BF16 and C in FP32, FP16 or BF16.
//
// A persistent, warp-specialised kernel, one CTA per SM:
//   warps 0-3  epilogue: tcgen05.ld the FP32 accumulator (warp w reads TMEM lanes 32w..32w+31, i.e. rows of the tile),
//              add the previous C when asked, convert, and store with plain st.global (masked at the M / N edges; any
//              ldc; in place for loadPreviousC)
//   warp 4     TMA producer: fills a 4-stage ring of [128 x 64] A and [64 x 256] B tiles (48 KB a stage)
//   warp 5     MMA issuer: tcgen05.mma.cta_group::1.kind::f16, 128 x 256 x 16, into one of two TMEM accumulators
// The two accumulators (2 x 256 of the 512 TMEM columns) let the epilogue of one tile overlap the main loop of the next.
// The 197 KB of shared memory keep a second CTA off the SM, which the 512-column TMEM allocation requires.
//
// Layouts (128-byte swizzle everywhere; see sm100_ptx.cuh for the descriptor fields):
//   A row-major  (M x K, K contiguous):  K-major,  one box of 64 (K) x 128 (M) rows
//   A transposed (K x M, M contiguous):  MN-major, two boxes of 64 (M) x 64 (K), 8 KB apart (LBO)
//   B row-major  (K x N, N contiguous):  MN-major, four boxes of 64 (N) x 64 (K), 8 KB apart (LBO)
//   B transposed (N x K, K contiguous):  K-major,  one box of 64 (K) x 256 (N) rows
// The batch is the third tensor-map dimension.  TMA reads out-of-bounds elements (beyond M, N or K) as zero, so edge
// tiles need no special path in the main loop.
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "device_state.h"
#include "gemm_params.h"
#include "sm100_ptx.cuh"
#include "tma_host.h"

namespace mfa {
namespace {
using namespace ptx;

constexpr uint32_t BM = kTcGemmBlockM, BN = kTcGemmBlockN, BK = kTcGemmBlockK;
constexpr uint32_t kStages = 4;
constexpr uint32_t kABytes = BM * BK * 2, kBBytes = BN * BK * 2, kStageBytes = kABytes + kBBytes;
constexpr uint32_t kBarrierBytes = 256;
constexpr uint32_t kSmemBytes = 1024 /* alignment slack */ + kStages * kStageBytes + kBarrierBytes;
constexpr uint32_t kTmemCols = 2 * BN;
// tiles are walked in groups of this many M-tiles, M fastest, so the CTAs of one wave share A rows and B columns in L2
constexpr uint32_t kGroupM = 16;

struct TcGemmArgs {
  void *C;
  uint32_t M, N, ldc;
  uint32_t tiles_m, tiles_n, num_tiles, num_kb;
  uint8_t precC, load_previous_C;
};

__device__ __forceinline__ void tile_coords(const TcGemmArgs &a, uint32_t t, uint32_t &m0, uint32_t &n0, uint32_t &b) {
  const uint32_t per_batch = a.tiles_m * a.tiles_n;
  b = t / per_batch;
  const uint32_t r = t - b * per_batch;
  const uint32_t first_m = (r / (kGroupM * a.tiles_n)) * kGroupM;
  const uint32_t group = min(a.tiles_m - first_m, kGroupM);
  const uint32_t local = r - first_m * a.tiles_n;
  m0 = (first_m + local % group) * BM;
  n0 = (local / group) * BN;
}

// 32 consecutive accumulator columns of one row -> C (row pointer `row`, columns [n, n + 32) clipped to N)
template <uint32_t kPrec>
__device__ __forceinline__ void store_chunk(void *row, uint32_t n, uint32_t N, const uint32_t (&r)[32], bool add) {
  constexpr uint32_t kElem = kPrec == 0 ? 4 : 2;
  char *p = static_cast<char *>(row) + static_cast<size_t>(n) * kElem;
  float v[32];
#pragma unroll
  for (uint32_t j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
  if (n + 32 <= N && (reinterpret_cast<uintptr_t>(p) & 15) == 0) {
    if (kPrec == 0) {
      float4 *q = reinterpret_cast<float4 *>(p);
#pragma unroll
      for (uint32_t j = 0; j < 8; ++j) {
        float4 o = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
        if (add) {
          const float4 c = q[j];
          o.x += c.x; o.y += c.y; o.z += c.z; o.w += c.w;
        }
        q[j] = o;
      }
    } else {
      uint4 *q = reinterpret_cast<uint4 *>(p);
#pragma unroll
      for (uint32_t j = 0; j < 4; ++j) {
        float *w = v + 8 * j;
        if (add) {
          const uint4 c = q[j];
          const uint32_t cw[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
          for (uint32_t h = 0; h < 4; ++h) {
            const float2 f = kPrec == 1 ? unpack_f16x2(cw[h]) : unpack_bf16x2(cw[h]);
            w[2 * h] += f.x;
            w[2 * h + 1] += f.y;
          }
        }
        uint32_t o[4];
#pragma unroll
        for (uint32_t h = 0; h < 4; ++h)
          o[h] = kPrec == 1 ? pack_f16x2(w[2 * h], w[2 * h + 1]) : pack_bf16x2(w[2 * h], w[2 * h + 1]);
        q[j] = make_uint4(o[0], o[1], o[2], o[3]);
      }
    }
    return;
  }
#pragma unroll
  for (uint32_t j = 0; j < 32; ++j) {
    if (n + j >= N) break;
    if (kPrec == 0) {
      float *q = reinterpret_cast<float *>(p) + j;
      *q = add ? v[j] + *q : v[j];
    } else {
      uint16_t *q = reinterpret_cast<uint16_t *>(p) + j;
      float x = v[j];
      if (add) {
        const uint32_t c = *q;
        x += kPrec == 1 ? unpack_f16x2(c).x : __uint_as_float(c << 16);
      }
      *q = static_cast<uint16_t>((kPrec == 1 ? pack_f16x2(x, 0.f) : pack_bf16x2(x, 0.f)) & 0xFFFFu);
    }
  }
}

template <bool kTransA, bool kTransB, bool kBF16>
__global__ void __launch_bounds__(kTcGemmThreads, 1)
    tcgen05_gemm(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB, TcGemmArgs a) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t *full = reinterpret_cast<uint64_t *>(smem + kStages * kStageBytes);
  uint64_t *empty = full + kStages;
  uint64_t *acc_full = empty + kStages;
  uint64_t *acc_empty = acc_full + 2;
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(acc_empty + 2);
  const uint32_t warp = threadIdx.x / 32, lane = threadIdx.x % 32;

  if (threadIdx.x == 128) {
    for (uint32_t s = 0; s < kStages; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (uint32_t s = 0; s < 2; ++s) {
      mbar_init(&acc_full[s], 1);
      mbar_init(&acc_empty[s], 4);  // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 4) {
    // ---------------- TMA producer ----------------
    if (lane == 0) {
      prefetch_tensormap(&mapA);
      prefetch_tensormap(&mapB);
      uint32_t it = 0;
      for (uint32_t t = blockIdx.x; t < a.num_tiles; t += gridDim.x) {
        uint32_t m0, n0, b;
        tile_coords(a, t, m0, n0, b);
        for (uint32_t kb = 0; kb < a.num_kb; ++kb, ++it) {
          const uint32_t st = it % kStages, ph = (it / kStages) & 1;
          mbar_wait(&empty[st], ph ^ 1);
          mbar_arrive_expect_tx(&full[st], kStageBytes);
          uint8_t *sa = smem + st * kStageBytes, *sb = sa + kABytes;
          const int32_t k0 = static_cast<int32_t>(kb * BK);
          if (kTransA) {
            tma_load_3d(sa, &mapA, &full[st], m0, k0, b);
            tma_load_3d(sa + kABytes / 2, &mapA, &full[st], m0 + 64, k0, b);
          } else {
            tma_load_3d(sa, &mapA, &full[st], k0, m0, b);
          }
          if (kTransB) {
            tma_load_3d(sb, &mapB, &full[st], k0, n0, b);
          } else {
#pragma unroll
            for (uint32_t j = 0; j < BN / 64; ++j) tma_load_3d(sb + j * (kBBytes / 4), &mapB, &full[st], n0 + 64 * j, k0, b);
          }
        }
      }
    }
  } else if (warp == 5) {
    // ---------------- MMA issuer ----------------
    constexpr uint32_t idesc = make_idesc_f16(BM, BN, kBF16 ? 1u : 0u, kTransA ? 1u : 0u, kTransB ? 0u : 1u);
    uint32_t it = 0, lt = 0;
    for (uint32_t t = blockIdx.x; t < a.num_tiles; t += gridDim.x, ++lt) {
      const uint32_t buf = lt & 1, use = lt >> 1;
      mbar_wait(&acc_empty[buf], (use & 1) ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + buf * BN;
      for (uint32_t kb = 0; kb < a.num_kb; ++kb, ++it) {
        const uint32_t st = it % kStages, ph = (it / kStages) & 1;
        mbar_wait(&full[st], ph);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + st * kStageBytes), sb = sa + kABytes;
          // K-major: the 16-element K step is 32 B inside the swizzle row; MN-major: 16 K rows = 2048 B
          const uint64_t da = make_smem_desc_sw128(sa, kTransA ? kABytes / 2 : 16, 1024);
          const uint64_t db = make_smem_desc_sw128(sb, kTransB ? 16 : kBBytes / 4, 1024);
#pragma unroll
          for (uint32_t k = 0; k < BK / 16; ++k) {
            const uint32_t ao = kTransA ? k * 2048 : k * 32, bo = kTransB ? k * 32 : k * 2048;
            umma_ss(d_tmem, da + (ao >> 4), db + (bo >> 4), idesc, (kb | k) != 0);
          }
          umma_commit(&empty[st]);
          if (kb + 1 == a.num_kb) umma_commit(&acc_full[buf]);
        }
        __syncwarp();
      }
    }
  } else {
    // ---------------- epilogue: warps 0-3, thread = one row of the tile ----------------
    uint32_t lt = 0;
    for (uint32_t t = blockIdx.x; t < a.num_tiles; t += gridDim.x, ++lt) {
      uint32_t m0, n0, b;
      tile_coords(a, t, m0, n0, b);
      const uint32_t buf = lt & 1, use = lt >> 1;
      mbar_wait(&acc_full[buf], use & 1);
      tc_fence_after();
      const uint32_t row = m0 + warp * 32 + lane;
      const uint32_t elem = a.precC == 0 ? 4 : 2;
      void *crow = static_cast<char *>(a.C) + (static_cast<size_t>(b) * a.M + row) * a.ldc * elem;
      const uint32_t taddr = tmem_base + ((warp * 32) << 16) + buf * BN;
      const bool add = a.load_previous_C != 0;
#pragma unroll 1
      for (uint32_t c = 0; c < BN / 32; ++c) {
        uint32_t r[32];
        tmem_ld32(taddr + c * 32, r);
        tc_wait_ld();
        if (c + 1 == BN / 32) {
          // the whole accumulator is in registers: hand the buffer back to the MMA warp before storing the last chunk
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[buf]);
        }
        const uint32_t n = n0 + c * 32;
        if (row < a.M && n < a.N) {
          if (a.precC == 0)
            store_chunk<0>(crow, n, a.N, r, add);
          else if (a.precC == 1)
            store_chunk<1>(crow, n, a.N, r, add);
          else
            store_chunk<2>(crow, n, a.N, r, add);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// dst[r][c] = c < cols ? src[r * src_ld + c] : 0 for c < dst_ld; one thread per destination element
__global__ void __launch_bounds__(256) stage_rows(const uint16_t *__restrict__ src, uint16_t *__restrict__ dst, uint64_t rows,
                                                  uint32_t cols, uint64_t src_ld, uint32_t dst_ld) {
  const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= rows * dst_ld) return;
  const uint64_t r = i / dst_ld;
  const uint32_t c = static_cast<uint32_t>(i % dst_ld);
  dst[i] = c < cols ? src[r * src_ld + c] : uint16_t(0);
}

bool needs_staging(const void *base, uint32_t ld) { return ld % 8 != 0 || reinterpret_cast<uintptr_t>(base) % 16 != 0; }

typedef void (*GemmKernel)(const CUtensorMap, const CUtensorMap, TcGemmArgs);

template <bool kTransA, bool kTransB>
GemmKernel pick_format(bool bf16) {
  return bf16 ? tcgen05_gemm<kTransA, kTransB, true> : tcgen05_gemm<kTransA, kTransB, false>;
}

}  // namespace

uint32_t tcgen05_gemm_smem_bytes() { return kSmemBytes; }

cudaError_t launch_tcgen05_gemm(const GemmParams &p, cudaStream_t stream) {
  const int device = current_device();
  // stored shape of each operand: rows x cols with leading dimension ld
  const uint32_t rowsA = p.transA ? p.K : p.M, colsA = p.transA ? p.M : p.K;
  const uint32_t rowsB = p.transB ? p.N : p.K, colsB = p.transB ? p.K : p.N;
  const void *A = p.A, *B = p.B;
  uint64_t lda = p.lda, ldb = p.ldb;
  const bool stageA = needs_staging(A, p.lda), stageB = needs_staging(B, p.ldb);
  if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(B)) & 1) {
    set_launch_detail("16-bit operands need 2-byte aligned base pointers");
    return cudaErrorInvalidValue;
  }
  if (stageA || stageB) {
    const uint32_t padA = (colsA + 7) / 8 * 8, padB = (colsB + 7) / 8 * 8;
    const size_t bytesA = stageA ? (static_cast<size_t>(p.batch) * rowsA * padA * 2 + 255) & ~size_t(255) : 0;
    const size_t bytesB = stageB ? (static_cast<size_t>(p.batch) * rowsB * padB * 2 + 255) & ~size_t(255) : 0;
    void *ws = nullptr;
    cudaError_t e = workspace_for(device, stream, bytesA + bytesB, &ws, /*slot=*/3);
    if (e != cudaSuccess) return e;
    auto stage = [&](const void *src, uint64_t src_ld, uint32_t rows, uint32_t cols, uint32_t pad, void *dst) {
      const uint64_t total_rows = static_cast<uint64_t>(p.batch) * rows;
      const uint64_t n = total_rows * pad;
      stage_rows<<<static_cast<uint32_t>((n + 255) / 256), 256, 0, stream>>>(
          static_cast<const uint16_t *>(src), static_cast<uint16_t *>(dst), total_rows, cols, src_ld, pad);
      return cudaGetLastError();
    };
    char *cursor = static_cast<char *>(ws);
    if (stageA) {
      // problems stay back to back: row r of problem b is row b * rowsA + r of the whole buffer at either pitch
      if ((e = stage(A, lda, rowsA, colsA, padA, cursor)) != cudaSuccess) return e;
      A = cursor;
      lda = padA;
      cursor += bytesA;
    }
    if (stageB) {
      if ((e = stage(B, ldb, rowsB, colsB, padB, cursor)) != cudaSuccess) return e;
      B = cursor;
      ldb = padB;
    }
  }
  CUtensorMap mapA, mapB;
  cudaError_t e = make_tensor_map_16bit_strided(&mapA, A, rowsA, colsA, p.batch, lda, lda * rowsA, 64,
                                                p.transA ? 64 : BM);
  if (e != cudaSuccess) return e;
  e = make_tensor_map_16bit_strided(&mapB, B, rowsB, colsB, p.batch, ldb, ldb * rowsB, 64, p.transB ? BN : 64);
  if (e != cudaSuccess) return e;

  TcGemmArgs a;
  a.C = p.C;
  a.M = p.M;
  a.N = p.N;
  a.ldc = p.ldc;
  a.tiles_m = (p.M + BM - 1) / BM;
  a.tiles_n = (p.N + BN - 1) / BN;
  const uint64_t tiles = static_cast<uint64_t>(a.tiles_m) * a.tiles_n * p.batch;
  if (tiles > 0xFFFFFFFFull) {
    set_launch_detail("%llu output tiles exceed the tile index range", (unsigned long long)tiles);
    return cudaErrorInvalidValue;
  }
  a.num_tiles = static_cast<uint32_t>(tiles);
  a.num_kb = (p.K + BK - 1) / BK;
  a.precC = p.precC;
  a.load_previous_C = p.load_previous_C;

  const bool bf16 = p.precA == 2;
  GemmKernel kernel = p.transA ? (p.transB ? pick_format<true, true>(bf16) : pick_format<true, false>(bf16))
                               : (p.transB ? pick_format<false, true>(bf16) : pick_format<false, false>(bf16));
  if ((e = ensure_max_dynamic_smem(reinterpret_cast<const void *>(kernel), kSmemBytes, device)) != cudaSuccess) return e;
  const uint32_t sms = device_sm_count(device);
  const uint32_t grid = a.num_tiles < sms ? a.num_tiles : sms;
  kernel<<<grid, kTcGemmThreads, kSmemBytes, stream>>>(mapA, mapB, a);
  return cudaGetLastError();
}

}  // namespace mfa

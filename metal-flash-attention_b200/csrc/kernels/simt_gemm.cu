// CUDA-core FP32 GEMM: every precision mix, transpose state, leading dimension and loadPreviousC the GEMMDescriptor
// can describe.  It exists for coverage (FP32 operands, FP16 beside BF16), not speed: the 16-bit problems the tensor
// cores can take go to tcgen05_gemm.cu.  One instantiation: operands are converted to FP32 as they are staged in
// shared memory, so the precisions and transposes are run-time arguments.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gemm_params.h"
#include "tma_host.h"

namespace mfa {
namespace {

constexpr uint32_t BM = kSimtGemmBlockM, BN = kSimtGemmBlockN, BK = kSimtGemmBlockK;

__device__ __forceinline__ float load_as_f32(const void *base, size_t i, uint32_t prec) {
  if (prec == 0) return static_cast<const float *>(base)[i];
  const uint16_t bits = static_cast<const uint16_t *>(base)[i];
  if (prec == 1) return __half2float(__ushort_as_half(bits));
  return __uint_as_float(static_cast<uint32_t>(bits) << 16);
}

__device__ __forceinline__ void store_from_f32(void *base, size_t i, uint32_t prec, float v) {
  if (prec == 0)
    static_cast<float *>(base)[i] = v;
  else if (prec == 1)
    static_cast<__half *>(base)[i] = __float2half_rn(v);
  else
    static_cast<__nv_bfloat16 *>(base)[i] = __float2bfloat16_rn(v);
}

// 64 x 64 output tile per CTA, 256 threads with a 4 x 4 patch each (rows ty + 16 i, columns tx + 16 j), K in steps of
// 16.  Each K step's 16 products go into a partial sum that is then added to the accumulator: the running FP32 sum
// takes K / 16 roundings instead of K.
__global__ void __launch_bounds__(kSimtGemmThreads) simt_gemm(GemmParams p) {
  __shared__ float As[BK][BM + 4];  // As[k][m]
  __shared__ float Bs[BK][BN + 4];  // Bs[k][n]
  const uint32_t tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
  const uint32_t n0 = blockIdx.x * BN, m0 = blockIdx.y * BM, b = blockIdx.z;
  const size_t strideA = static_cast<size_t>(p.transA ? p.K : p.M) * p.lda;
  const size_t strideB = static_cast<size_t>(p.transB ? p.N : p.K) * p.ldb;
  const size_t strideC = static_cast<size_t>(p.M) * p.ldc;
  const size_t baseA = b * strideA, baseB = b * strideB;
  float acc[4][4] = {};
  for (uint32_t k0 = 0; k0 < p.K; k0 += BK) {
    // 1024 elements of each tile, 4 per thread; the fastest-varying index follows the stored layout
    for (uint32_t e = tid; e < BM * BK; e += kSimtGemmThreads) {
      uint32_t m, k;
      if (p.transA) { m = e % BM; k = e / BM; } else { k = e % BK; m = e / BK; }
      const uint32_t gm = m0 + m, gk = k0 + k;
      float v = 0.f;
      if (gm < p.M && gk < p.K)
        v = load_as_f32(p.A, baseA + (p.transA ? static_cast<size_t>(gk) * p.lda + gm : static_cast<size_t>(gm) * p.lda + gk),
                        p.precA);
      As[k][m] = v;
    }
    for (uint32_t e = tid; e < BN * BK; e += kSimtGemmThreads) {
      uint32_t n, k;
      if (p.transB) { k = e % BK; n = e / BK; } else { n = e % BN; k = e / BN; }
      const uint32_t gn = n0 + n, gk = k0 + k;
      float v = 0.f;
      if (gn < p.N && gk < p.K)
        v = load_as_f32(p.B, baseB + (p.transB ? static_cast<size_t>(gn) * p.ldb + gk : static_cast<size_t>(gk) * p.ldb + gn),
                        p.precB);
      Bs[k][n] = v;
    }
    __syncthreads();
    float part[4][4] = {};
#pragma unroll
    for (uint32_t k = 0; k < BK; ++k) {
      float a[4], bv[4];
#pragma unroll
      for (uint32_t i = 0; i < 4; ++i) a[i] = As[k][ty + 16 * i];
#pragma unroll
      for (uint32_t j = 0; j < 4; ++j) bv[j] = Bs[k][tx + 16 * j];
#pragma unroll
      for (uint32_t i = 0; i < 4; ++i)
#pragma unroll
        for (uint32_t j = 0; j < 4; ++j) part[i][j] = fmaf(a[i], bv[j], part[i][j]);
    }
#pragma unroll
    for (uint32_t i = 0; i < 4; ++i)
#pragma unroll
      for (uint32_t j = 0; j < 4; ++j) acc[i][j] += part[i][j];
    __syncthreads();
  }
#pragma unroll
  for (uint32_t i = 0; i < 4; ++i) {
    const uint32_t gm = m0 + ty + 16 * i;
    if (gm >= p.M) continue;
#pragma unroll
    for (uint32_t j = 0; j < 4; ++j) {
      const uint32_t gn = n0 + tx + 16 * j;
      if (gn >= p.N) continue;
      const size_t idx = b * strideC + static_cast<size_t>(gm) * p.ldc + gn;
      float v = acc[i][j];
      if (p.load_previous_C) v += load_as_f32(p.C, idx, p.precC);
      store_from_f32(p.C, idx, p.precC, v);
    }
  }
}

}  // namespace

uint32_t simt_gemm_smem_bytes() { return static_cast<uint32_t>(BK * (BM + 4) * 4 + BK * (BN + 4) * 4); }

cudaError_t launch_simt_gemm(const GemmParams &p, cudaStream_t stream) {
  const dim3 grid((p.N + BN - 1) / BN, (p.M + BM - 1) / BM, 1);
  if (grid.y > 65535) {
    set_launch_detail("M = %u exceeds the SIMT GEMM's grid limit", p.M);
    return cudaErrorInvalidValue;
  }
  // the batch rides in gridDim.z (limit 65535): larger batches go out as several launches over slices of it
  constexpr uint32_t kMaxBatch = 65535;
  for (uint32_t b0 = 0; b0 < p.batch; b0 += kMaxBatch) {
    GemmParams q = p;
    q.batch = p.batch - b0 < kMaxBatch ? p.batch - b0 : kMaxBatch;
    const size_t elemA = p.precA == 0 ? 4 : 2, elemB = p.precB == 0 ? 4 : 2, elemC = p.precC == 0 ? 4 : 2;
    q.A = static_cast<const char *>(p.A) + b0 * static_cast<size_t>(p.transA ? p.K : p.M) * p.lda * elemA;
    q.B = static_cast<const char *>(p.B) + b0 * static_cast<size_t>(p.transB ? p.N : p.K) * p.ldb * elemB;
    q.C = static_cast<char *>(p.C) + b0 * static_cast<size_t>(p.M) * p.ldc * elemC;
    dim3 g = grid;
    g.z = q.batch;
    simt_gemm<<<g, kSimtGemmThreads, 0, stream>>>(q);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

}  // namespace mfa

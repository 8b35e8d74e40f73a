// Internal launch interface between csrc/gemm.cpp and the GEMM kernels (simt_gemm.cu, tcgen05_gemm.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mfa {

// One encode() of C = A . B (+ C).  Precisions are GEMMOperandPrecision raw values (FP32 0, FP16 1, BF16 2).
struct GemmParams {
  uint32_t M, N, K;
  uint32_t batch;           // >= 1; problem b of an operand starts at b * trailing * leading elements
  uint32_t lda, ldb, ldc;   // in elements
  const void *A, *B;
  void *C;
  uint8_t precA, precB, precC;
  uint8_t transA, transB;   // A stored K x M / B stored N x K
  uint8_t load_previous_C;
};

// ---- SIMT FP32 family: every precision mix, transpose and leading dimension ----
constexpr uint32_t kSimtGemmBlockM = 64, kSimtGemmBlockN = 64, kSimtGemmBlockK = 16, kSimtGemmThreads = 256;
uint32_t simt_gemm_smem_bytes();
cudaError_t launch_simt_gemm(const GemmParams &p, cudaStream_t stream);

// ---- tcgen05 family: A and B both FP16 or both BF16, C any precision ----
constexpr uint32_t kTcGemmBlockM = 128, kTcGemmBlockN = 256, kTcGemmBlockK = 64, kTcGemmThreads = 192;
uint32_t tcgen05_gemm_smem_bytes();
// Operands whose leading dimension is not a multiple of 8 elements, or whose base is not 16-byte aligned, are first
// copied into a zero-padded staging buffer (TMA needs a 16-byte aligned base and row pitch).
cudaError_t launch_tcgen05_gemm(const GemmParams &p, cudaStream_t stream);

}  // namespace mfa

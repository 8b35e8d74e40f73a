// Internal launch interface between the C-ABI host layer (csrc/*.cpp) and the sm_100a kernels.
// Not part of the public ABI (include/mfa_b200.h is).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mfa {

// Buffer slots = AttentionOperand.bufferBinding
// (/root/reference/Sources/FlashAttention/Attention/AttentionOperand.swift:52-71).
enum Slot { sQ = 0, sK = 1, sV = 2, sO = 3, sL = 4, sD = 5, sdO = 6, sdV = 7, sdK = 8, sdQ = 9, kSlots = 10 };

// Precision raw values = GEMMOperandPrecision (GEMMOperandPrecision.swift:33-37).
enum Prec : uint8_t { FP32 = 0, FP16 = 1, BF16 = 2 };

struct AttentionParams {
  uint32_t R;      // rows of the attention matrix (output sequence length)
  uint32_t C;      // columns (input sequence length)
  uint32_t D;      // head dimension
  uint32_t batch;  // independent single-head problems, >= 1
  void *buf[kSlots];        // device pointers, by slot
  uint8_t prec[kSlots];     // memory precision, by slot
  uint8_t transposed[kSlots];  // 1: stored [D][seq] (leading dim = seq), 0: [seq][D]
  float scale;       // 1/sqrt(D)          (AttentionKernel+Softmax.swift:17-26)
  float scale_log2;  // log2(e)/sqrt(D)
  // tuning columns of the parameter-table row the kernel was created from (tcgen05 family)
  uint8_t exp2_fma_quarters;  // selects the kernel instantiation
  uint8_t split_min_blocks;   // 0 = never split small grids
  uint8_t split_max;
};

// compiled exp2-on-the-FMA-pipe variants (quarters of the element pairs): forward 0..2, backward 0..3
constexpr uint32_t kMaxForwardExp2Quarters = 2, kMaxBackwardExp2Quarters = 3;

// ---- SIMT FP32 family (any shape / layout / precision) -------------------------------------
cudaError_t launch_simt_forward(const AttentionParams &p, cudaStream_t stream);
cudaError_t launch_simt_backward_query(const AttentionParams &p, cudaStream_t stream);
cudaError_t launch_simt_backward_key_value(const AttentionParams &p, cudaStream_t stream);
void simt_geometry(int type, uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par, uint32_t *trav,
                   uint32_t *head);

// ---- tcgen05 / TMA / TMEM family (16-bit inputs, D % 8 == 0) --------------------------------
// kernel.cpp picks the kernel of a descriptor once, at creation; each launcher below serves only its own kernel.
// The *_supported checks validate the encode-time R, C and output precisions against what these kernels handle.
bool tcgen05_forward_supported(const AttentionParams &p);
cudaError_t launch_tcgen05_forward(const AttentionParams &p, cudaStream_t stream);  // row-major, D <= 128
void tcgen05_forward_geometry(uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par, uint32_t *trav,
                              uint32_t *head);
uint32_t tcgen05_forward_launch_count(uint32_t R, uint32_t C, uint32_t batch, uint32_t min_blocks, uint32_t max_splits);
cudaError_t launch_tcgen05_forward_d256(const AttentionParams &p, cudaStream_t stream);  // row-major, 128 < D <= 256
cudaError_t launch_tcgen05_forward_generic(const AttentionParams &p, cudaStream_t stream);  // transposed operands, D <= 256
bool tcgen05_forward_transposes_ok(uint32_t R, uint32_t C, bool tQ, bool tK, bool tV);
// geometry of the kernel template behind both launch_tcgen05_forward_d256 and launch_tcgen05_forward_generic
void tcgen05_forward_generic_geometry(uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par, uint32_t *trav,
                                      uint32_t *head);
bool tcgen05_backward_supported(const AttentionParams &p);
// row-major, D <= 128; key_value: dK and dV, else dQ (and the D term)
cudaError_t launch_tcgen05_backward(const AttentionParams &p, cudaStream_t stream, bool key_value);
uint32_t tcgen05_backward_launch_count(int type, uint32_t R, uint32_t C, uint32_t batch, uint32_t min_blocks,
                                       uint32_t max_splits, bool convert_dO);
bool tcgen05_backward_converts_dO_first(uint32_t C, uint32_t batch);
void tcgen05_backward_geometry(int type, uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par,
                               uint32_t *trav, uint32_t *head);
// layout-generic backward (tcgen05_backward_generic.cu): 128 < D <= 256, and transposed operands at any D <= 256
bool tcgen05_backward_transposes_ok(uint32_t R, uint32_t C, bool tQ, bool tK, bool tV, bool tO);
cudaError_t launch_tcgen05_backward_generic(const AttentionParams &p, cudaStream_t stream, bool key_value);
uint32_t tcgen05_backward_generic_launch_count(int type, uint32_t R, uint32_t C, uint32_t D, uint32_t batch,
                                               uint32_t min_blocks, uint32_t max_splits, bool convert_dO);
void tcgen05_backward_generic_geometry(int type, uint32_t D, uint32_t *threads, uint32_t *smem_bytes, uint32_t *par,
                                       uint32_t *trav, uint32_t *head);

cudaError_t launch_tcgen05_forward_trace(const AttentionParams &p, cudaStream_t stream, long long *trace);  // debug
cudaError_t launch_tcgen05_forward_d256_trace(const AttentionParams &p, cudaStream_t stream, long long *trace);  // debug
// head-dimension padding for D % 8 != 0 on the tensor-core family (pad_head.cu)
cudaError_t launch_pad_columns(const void *src, void *dst, uint64_t rows, uint32_t D, uint32_t Dp, uint32_t element_bytes,
                               cudaStream_t stream);
cudaError_t launch_bf16_to_f16(const void *src, void *dst, uint64_t elements, cudaStream_t stream);
cudaError_t launch_unpad_columns(const void *src, void *dst, uint64_t rows, uint32_t D, uint32_t Dp, cudaStream_t stream);
const char *last_launch_detail();  // thread-local detail string for MFA_ERROR_CUDA messages

}  // namespace mfa

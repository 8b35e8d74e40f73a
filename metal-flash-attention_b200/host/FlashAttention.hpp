// FlashAttention.hpp -- header-only C++ mirror of the reference's Swift value types over the C ABI
// (include/mfa_b200.h).  The reference is compiled Swift; Swift is not installed in this image, so this is the
// compiled-language host layer "above the C ABI": same type and member names as
// Sources/FlashAttention/Attention/{AttentionDescriptor,AttentionKernelDescriptor,AttentionKernel}.swift and
// Sources/FlashAttention/GEMM/{GEMMDescriptor,GEMMKernelDescriptor,GEMMKernel}.swift, same validation, and fatalError() behaviour surfaced as std::runtime_error carrying the reference's message.
#pragma once
#include <array>
#include <optional>
#include <stdexcept>
#include <string>
#include <tuple>

#include "../../include/mfa_b200.h"

namespace FlashAttention {

enum class GEMMOperandPrecision : uint16_t { FP32 = 0, FP16 = 1, BF16 = 2 };  // GEMMOperandPrecision.swift:33-37
enum class AttentionKernelType { forward = 0, backwardQuery = 1, backwardKeyValue = 2 };  // AttentionKernelType.swift
enum class AttentionOperand { Q = 0, K, V, O, L, D, dO, dV, dK, dQ, S, P, dP, dS };      // AttentionOperand.swift

inline std::optional<uint8_t> bufferBinding(AttentionOperand operand) {  // AttentionOperand.swift:52-71
  int binding = mfa_operand_buffer_binding(static_cast<mfa_operand_t>(operand));
  return binding < 0 ? std::nullopt : std::optional<uint8_t>(static_cast<uint8_t>(binding));
}

inline void check(int status) {
  if (status != MFA_SUCCESS) throw std::runtime_error(mfa_last_error());
}

struct MatrixDimensions { uint32_t row, column; uint16_t head; };
struct TransposeState { bool Q, K, V, O; };

struct AttentionKernelDescriptor {  // AttentionKernelDescriptor.swift:7-48
  mfa_attention_kernel_descriptor_t c;
  AttentionKernelDescriptor() { mfa_attention_kernel_descriptor_init(&c); }
  std::optional<std::tuple<uint16_t, uint16_t, uint16_t>> blockDimensions() const {
    if (!c.has_block_dimensions) return std::nullopt;
    return std::make_tuple(c.block_parallelization, c.block_traversal, c.block_head);
  }
  std::optional<uint16_t> headDimension() const {
    return c.has_head_dimension ? std::optional<uint16_t>(c.head_dimension) : std::nullopt;
  }
  // B200 extension: the tuning columns of the parameter-table row (editable like every other field)
  uint8_t &exp2FmaQuarters() { return c.exp2_fma_quarters; }
  uint8_t &splitMinBlocks() { return c.split_min_blocks; }
  uint8_t &splitMax() { return c.split_max; }
  bool tensorCoreFamily() const { return c.backend == MFA_BACKEND_TCGEN05; }
};

// The parameter tables are data (AttentionDescriptor+Parameters.swift:106-285 analogue): replace one at run time.
inline void setParameterTable(AttentionKernelType type, const char *text, bool transposed = false) {
  check(mfa_set_parameter_table(static_cast<mfa_kernel_type_t>(type), transposed ? 1 : 0, text));
}

struct AttentionDescriptor {  // AttentionDescriptor.swift:10-27
  bool lowPrecisionInputs = false;
  bool lowPrecisionIntermediates = false;
  std::optional<MatrixDimensions> matrixDimensions;
  std::optional<TransposeState> transposeState;
  std::optional<GEMMOperandPrecision> inputPrecisionOverride;  // B200 extension
  uint32_t batchCount = 1;                                     // B200 extension

  mfa_attention_descriptor_t c() const {
    mfa_attention_descriptor_t d;
    mfa_attention_descriptor_init(&d);
    d.low_precision_inputs = lowPrecisionInputs;
    d.low_precision_intermediates = lowPrecisionIntermediates;
    if (matrixDimensions) {
      d.has_matrix_dimensions = 1;
      d.row = matrixDimensions->row; d.column = matrixDimensions->column; d.head = matrixDimensions->head;
    }
    if (transposeState) {
      d.has_transpose_state = 1;
      d.transpose_Q = transposeState->Q; d.transpose_K = transposeState->K;
      d.transpose_V = transposeState->V; d.transpose_O = transposeState->O;
    }
    d.input_precision_override = inputPrecisionOverride ? static_cast<uint8_t>(*inputPrecisionOverride) : 0;
    d.batch_count = batchCount;
    return d;
  }
  AttentionKernelDescriptor kernelDescriptor(AttentionKernelType type) const {  // AttentionDescriptor.swift:33-130
    mfa_attention_descriptor_t d = c();
    AttentionKernelDescriptor out;
    check(mfa_attention_descriptor_kernel_descriptor(&d, static_cast<mfa_kernel_type_t>(type), &out.c));
    return out;
  }
  GEMMOperandPrecision memoryPrecision(AttentionOperand operand) const {  // +Precisions.swift:10-146
    mfa_attention_descriptor_t d = c();
    mfa_precision_t p;
    check(mfa_attention_descriptor_memory_precision(&d, static_cast<mfa_operand_t>(operand), &p));
    return static_cast<GEMMOperandPrecision>(p);
  }
  GEMMOperandPrecision registerPrecision(AttentionOperand operand) const {  // +Precisions.swift:149-215
    mfa_attention_descriptor_t d = c();
    mfa_precision_t p;
    check(mfa_attention_descriptor_register_precision(&d, static_cast<mfa_operand_t>(operand), &p));
    return static_cast<GEMMOperandPrecision>(p);
  }
  std::string parameterFile(AttentionKernelType type) const {  // +Parameters.swift:13-39
    mfa_attention_descriptor_t d = c();
    return mfa_attention_descriptor_parameter_file(&d, static_cast<mfa_kernel_type_t>(type));
  }
  void setFunctionConstants(mfa_function_constants_t &constants) const {  // AttentionDescriptor.swift:139-148
    mfa_attention_descriptor_t d = c();
    check(mfa_attention_descriptor_set_function_constants(&d, &constants));
  }
  // end-to-end call on HOST pointers: H2D -> kernels (fwd -> dQ -> dK/dV, SquareAttentionTest.swift:355-368) -> D2H
  void runHost(uint32_t runMask, const std::array<void *, MFA_BUFFER_COUNT> &hostBuffers, int device = 0) const {
    mfa_attention_descriptor_t d = c();
    check(mfa_attention_run_host(&d, runMask, hostBuffers.data(), device));
  }
};

class AttentionKernel {  // AttentionKernel.swift:11-50
 public:
  explicit AttentionKernel(const AttentionKernelDescriptor &descriptor) { check(mfa_attention_kernel_create(&descriptor.c, &handle_)); }
  // library-owned kernel object from the descriptor-keyed cache (the analogue of GEMMKernel.pipelineCache[descriptor],
  // GEMMDescriptor+PipelineCache.swift:16-36)
  AttentionKernel(const AttentionDescriptor &descriptor, AttentionKernelType type) : owned_(false) {
    mfa_attention_descriptor_t d = descriptor.c();
    const mfa_attention_kernel_t *out = nullptr;
    check(mfa_attention_kernel_cache_fetch(&d, static_cast<mfa_kernel_type_t>(type), &out));
    handle_ = const_cast<mfa_attention_kernel_t *>(out);
  }
  ~AttentionKernel() { if (owned_) mfa_attention_kernel_destroy(handle_); }
  AttentionKernel(const AttentionKernel &) = delete;
  AttentionKernel &operator=(const AttentionKernel &) = delete;
  std::tuple<uint16_t, uint16_t, uint16_t> blockDimensions() const {
    uint16_t out[3];
    check(mfa_attention_kernel_block_dimensions(handle_, out));
    return {out[0], out[1], out[2]};
  }
  uint32_t threadgroupSize() const { uint32_t v; check(mfa_attention_kernel_threadgroup_size(handle_, &v)); return v; }
  uint32_t threadgroupMemoryAllocation() const {
    uint32_t v; check(mfa_attention_kernel_threadgroup_memory_allocation(handle_, &v)); return v;
  }
  uint32_t gridSize(const mfa_function_constants_t &constants) const {  // SquareAttentionTest.swift:328-339
    uint32_t v; check(mfa_attention_kernel_grid_size(handle_, &constants, &v)); return v;
  }
  uint32_t launchCount(const mfa_function_constants_t &constants) const {
    uint32_t v; check(mfa_attention_kernel_launch_count(handle_, &constants, &v)); return v;
  }
  std::string sourceName() const { return mfa_attention_kernel_source_name(handle_); }
  // compile + bind + dispatch (SquareAttentionTest.swift:240-372): device pointers by buffer binding
  void encode(const mfa_function_constants_t &constants, const std::array<void *, MFA_BUFFER_COUNT> &buffers,
              void *cudaStream = nullptr) const {
    check(mfa_attention_kernel_encode(handle_, &constants, buffers.data(), cudaStream));
  }
 private:
  mfa_attention_kernel_t *handle_ = nullptr;
  bool owned_ = true;
};

// ------------------------------------------------------------------------------------------------------------------
// GEMM (Sources/FlashAttention/GEMM/): C = A . B, or C += A . B with loadPreviousC
// ------------------------------------------------------------------------------------------------------------------
struct GEMMMatrixDimensions { uint32_t M, N, K; };
struct GEMMLeadingDimensions { uint32_t A, B, C; };
struct GEMMPrecisions { GEMMOperandPrecision A, B, C; };
struct GEMMTransposeState { bool A, B; };

struct GEMMDescriptor {  // GEMMDescriptor.swift:10-44
  uint32_t batchDimension = 1;  // > 1: B200 extension, independent problems stored back to back
  std::optional<GEMMLeadingDimensions> leadingDimensions;
  bool loadPreviousC = false;
  std::optional<GEMMMatrixDimensions> matrixDimensions;
  std::optional<GEMMPrecisions> memoryPrecisions;
  std::optional<GEMMTransposeState> transposeState;

  mfa_gemm_descriptor_t c() const {
    mfa_gemm_descriptor_t d;
    mfa_gemm_descriptor_init(&d);
    d.batch_dimension = batchDimension;
    if (leadingDimensions) {
      d.has_leading_dimensions = 1;
      d.leading_dimensions[0] = leadingDimensions->A;
      d.leading_dimensions[1] = leadingDimensions->B;
      d.leading_dimensions[2] = leadingDimensions->C;
    }
    d.load_previous_C = loadPreviousC;
    if (matrixDimensions) {
      d.has_matrix_dimensions = 1;
      d.M = matrixDimensions->M; d.N = matrixDimensions->N; d.K = matrixDimensions->K;
    }
    if (memoryPrecisions) {
      d.has_memory_precisions = 1;
      d.memory_precisions[0] = static_cast<uint8_t>(memoryPrecisions->A);
      d.memory_precisions[1] = static_cast<uint8_t>(memoryPrecisions->B);
      d.memory_precisions[2] = static_cast<uint8_t>(memoryPrecisions->C);
    }
    if (transposeState) {
      d.has_transpose_state = 1;
      d.transpose_A = transposeState->A; d.transpose_B = transposeState->B;
    }
    return d;
  }
  void setFunctionConstants(mfa_gemm_function_constants_t &constants) const {  // GEMMDescriptor.swift:327-380
    mfa_gemm_descriptor_t d = c();
    check(mfa_gemm_descriptor_set_function_constants(&d, &constants));
  }
};

struct GEMMKernelDescriptor {  // GEMMKernelDescriptor.swift:21-181; the raw fields stay editable through `c`
  mfa_gemm_kernel_descriptor_t c;
  GEMMKernelDescriptor() { mfa_gemm_kernel_descriptor_init(&c); }
  explicit GEMMKernelDescriptor(const GEMMDescriptor &descriptor) {  // GEMMDescriptor.swift:106-234
    mfa_gemm_descriptor_t d = descriptor.c();
    check(mfa_gemm_descriptor_kernel_descriptor(&d, &c));
  }
  std::optional<std::tuple<uint16_t, uint16_t, uint16_t>> blockDimensions() const {
    if (!c.has_block_dimensions) return std::nullopt;
    return std::make_tuple(c.block_dimensions[0], c.block_dimensions[1], c.block_dimensions[2]);
  }
  bool tensorCoreFamily() const { return c.backend == MFA_BACKEND_TCGEN05; }
};

class GEMMKernel {  // GEMMKernel.swift:10-270
 public:
  explicit GEMMKernel(const GEMMKernelDescriptor &descriptor) { check(mfa_gemm_kernel_create(&descriptor.c, &handle_)); }
  // GEMMKernel.register(descriptor:) + pipelineCache[descriptor] (GEMMDescriptor+PipelineCache.swift:16-36): the
  // library-owned kernel object of the descriptor (`register` is a C++ keyword, hence the underscore)
  static void register_(const GEMMDescriptor &descriptor) { GEMMKernel unused(descriptor); }
  static GEMMKernel cached(const GEMMDescriptor &descriptor) { return GEMMKernel(descriptor); }
  explicit GEMMKernel(const GEMMDescriptor &descriptor) : owned_(false) {
    mfa_gemm_descriptor_t d = descriptor.c();
    const mfa_gemm_kernel_t *out = nullptr;
    check(mfa_gemm_kernel_cache_fetch(&d, &out));
    handle_ = const_cast<mfa_gemm_kernel_t *>(out);
  }
  static int cacheSize() { return mfa_gemm_kernel_cache_size(); }
  ~GEMMKernel() { if (owned_) mfa_gemm_kernel_destroy(handle_); }
  GEMMKernel(const GEMMKernel &) = delete;
  GEMMKernel &operator=(const GEMMKernel &) = delete;
  std::tuple<uint16_t, uint16_t, uint16_t> blockDimensions() const {
    uint16_t out[3];
    check(mfa_gemm_kernel_block_dimensions(handle_, out));
    return {out[0], out[1], out[2]};
  }
  uint32_t threadgroupSize() const { uint32_t v; check(mfa_gemm_kernel_threadgroup_size(handle_, &v)); return v; }
  uint32_t threadgroupMemoryAllocation() const {
    uint32_t v; check(mfa_gemm_kernel_threadgroup_memory_allocation(handle_, &v)); return v;
  }
  uint32_t gridSize(const mfa_gemm_function_constants_t &constants) const {
    uint32_t v; check(mfa_gemm_kernel_grid_size(handle_, &constants, &v)); return v;
  }
  uint32_t launchCount(const mfa_gemm_function_constants_t &constants) const {
    uint32_t v; check(mfa_gemm_kernel_launch_count(handle_, &constants, &v)); return v;
  }
  std::string sourceName() const { return mfa_gemm_kernel_source_name(handle_); }
  // bind A, B, C (device pointers, bindings 0, 1, 2; GEMMKernel+Source.swift:42-44) + dispatch
  void encode(const mfa_gemm_function_constants_t &constants, const std::array<void *, MFA_GEMM_BUFFER_COUNT> &buffers,
              void *cudaStream = nullptr) const {
    check(mfa_gemm_kernel_encode(handle_, &constants, buffers.data(), cudaStream));
  }
 private:
  mfa_gemm_kernel_t *handle_ = nullptr;
  bool owned_ = true;
};

// Page-locked host buffers on the GPU's NUMA node for AttentionDescriptor::runHost (B200 extension; the reference's
// buffers are Metal shared-storage buffers, MTLContext+Buffers.swift:5-45)
struct HostMemory {
  // upload: write-combined pages for buffers the host only writes and the GPU reads (Q, K, V, dO)
  static void *allocate(size_t byteCount, int device = 0, bool upload = false) {
    void *pointer = nullptr;
    check(upload ? mfa_host_alloc_upload(byteCount, device, &pointer) : mfa_host_alloc(byteCount, device, &pointer));
    return pointer;
  }
  static void free(void *pointer) { check(mfa_host_free(pointer)); }
  static int bindThread(int device) {
    int node = -1;
    check(mfa_host_bind_thread_to_device(device, &node));
    return node;
  }
  static void releaseResources(int device) { check(mfa_release_device_resources(device)); }
};

}  // namespace FlashAttention

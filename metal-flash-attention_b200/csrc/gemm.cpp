// GEMM side of the C ABI: GEMMDescriptor, GEMMKernelDescriptor(descriptor:), GEMMKernel and its pipeline cache.
// Mirrors Sources/FlashAttention/GEMM/ (GEMMDescriptor.swift, GEMMKernelDescriptor.swift, GEMMKernel.swift,
// GEMMDescriptor+PipelineCache.swift); encode() is the bind + dispatch the reference leaves to its caller
// (Tests/FlashAttentionTests/GEMM/AdversarialShapeTest.swift:140-169).
#include <cuda_runtime.h>

#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "internal.h"
#include "kernels/device_state.h"
#include "kernels/gemm_params.h"

struct mfa_gemm_kernel {
  mfa_gemm_kernel_descriptor_t descriptor;
  int backend;
  uint32_t threads, smem_bytes;
  uint16_t block[3];
  std::string source_name;
};

namespace mfa {
namespace {

bool valid_precision(uint8_t p) { return p == MFA_FP32 || p == MFA_FP16 || p == MFA_BF16; }

// both 16-bit inputs of one type: the only mix tcgen05 kind::f16 multiplies (FP16 beside BF16 is not an MMA format)
bool tensor_core_inputs(uint8_t a, uint8_t b) { return a == b && (a == MFA_FP16 || a == MFA_BF16); }

// checkOperandPair (GEMMKernel.swift:46-84): the register precision equals the memory precision, or is FP32
bool register_pair_valid(uint8_t memory, uint8_t reg) { return reg == memory || reg == MFA_FP32; }

// the leading block dimensions the compiled kernel uses (chooseLeadingBlockDimension, GEMMKernel.swift:107-149)
void leading_block_dimensions(const uint16_t block[3], bool tA, bool tB, uint16_t out[3]) {
  out[0] = tA ? block[0] : block[2];
  out[1] = tB ? block[2] : block[1];
  out[2] = block[1];
}

uint32_t batch_of(const mfa_gemm_function_constants_t &c) { return c.batch_count ? c.batch_count : 1; }

}  // namespace
}  // namespace mfa

using namespace mfa;

extern "C" {

void mfa_gemm_descriptor_init(mfa_gemm_descriptor_t *d) {
  if (!d) return;
  std::memset(d, 0, sizeof(*d));
  d->batch_dimension = 1;
}

int mfa_gemm_descriptor_set_function_constants(const mfa_gemm_descriptor_t *d, mfa_gemm_function_constants_t *c) {
  if (!d || !c) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  // guard let matrixDimensions, transposeState else fatalError (GEMMDescriptor.swift:328-331)
  if (!d->has_matrix_dimensions || !d->has_transpose_state)
    return fail(MFA_ERROR_INCOMPLETE_DESCRIPTOR, "Descriptor was incomplete.");
  // chooseLeadingDimension (:340-364): transposed -> untransposed rows, else untransposed columns
  const uint32_t expected[3] = {d->transpose_A ? d->M : d->K, d->transpose_B ? d->K : d->N, d->N};
  mfa_gemm_function_constants_t out;
  std::memset(&out, 0, sizeof(out));
  for (int i = 0; i < 3; ++i) {
    if (d->has_leading_dimensions) {
      if (d->leading_dimensions[i] < expected[i])
        return fail(MFA_ERROR_INVALID_ARGUMENT, "Leading block dimension was too small.");
      out.leading_dimensions[i] = d->leading_dimensions[i];
    } else {
      out.leading_dimensions[i] = expected[i];
    }
  }
  out.M = d->M;
  out.N = d->N;
  out.K = d->K;
  out.load_previous_C = d->load_previous_C ? 1 : 0;
  out.batch_count = d->batch_dimension ? d->batch_dimension : 1;
  *c = out;
  return MFA_SUCCESS;
}

void mfa_gemm_kernel_descriptor_init(mfa_gemm_kernel_descriptor_t *kd) {
  if (!kd) return;
  std::memset(kd, 0, sizeof(*kd));
  kd->prefer_async_load = 1;     // "The default value is `true`." (GEMMKernelDescriptor.swift:134)
  kd->prefer_async_store = 0xFF;
}

int mfa_gemm_descriptor_kernel_descriptor(const mfa_gemm_descriptor_t *d, mfa_gemm_kernel_descriptor_t *out) {
  if (!d || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  // guard let matrixDimensions, memoryPrecisions, transposeState else fatalError (GEMMDescriptor.swift:107-111)
  if (!d->has_matrix_dimensions || !d->has_memory_precisions || !d->has_transpose_state)
    return fail(MFA_ERROR_INCOMPLETE_DESCRIPTOR, "Descriptor was incomplete.");
  for (int i = 0; i < 3; ++i)
    if (!valid_precision(d->memory_precisions[i]))
      return fail(MFA_ERROR_INVALID_ARGUMENT, "Unrecognized memory precision.");
  mfa_gemm_kernel_descriptor_t kd;
  mfa_gemm_kernel_descriptor_init(&kd);
  const bool tc = tensor_core_inputs(d->memory_precisions[0], d->memory_precisions[1]);
  kd.backend = tc ? MFA_BACKEND_TCGEN05 : MFA_BACKEND_SIMT_FP32;
  kd.has_block_dimensions = 1;
  if (tc) {
    kd.block_dimensions[0] = kTcGemmBlockM;
    kd.block_dimensions[1] = kTcGemmBlockN;
    kd.block_dimensions[2] = kTcGemmBlockK;
    // the 128-row accumulator tile is read out of TMEM by four warps of 32 lanes each
    kd.splits[0] = 4;
    kd.splits[1] = 1;
  } else {
    kd.block_dimensions[0] = kSimtGemmBlockM;
    kd.block_dimensions[1] = kSimtGemmBlockN;
    kd.block_dimensions[2] = kSimtGemmBlockK;
    kd.splits[0] = 2;   // 32 * 2 * 4 = 256 threads, each owning a 4 x 4 patch of the 64 x 64 tile
    kd.splits[1] = 4;
  }
  kd.has_splits = 1;
  kd.has_leading_block_dimensions = 1;
  leading_block_dimensions(kd.block_dimensions, d->transpose_A, d->transpose_B, kd.leading_block_dimensions);
  kd.has_memory_precisions = 1;
  std::memcpy(kd.memory_precisions, d->memory_precisions, 3);
  // registerPrecisions (GEMMDescriptor.swift:192-208): A and B as in memory; C is FP32 because both families accumulate
  // in FP32 -- the reference's FP16 accumulator for an all-FP16 problem would only lose accuracy here
  kd.has_register_precisions = 1;
  kd.register_precisions[0] = d->memory_precisions[0];
  kd.register_precisions[1] = d->memory_precisions[1];
  kd.register_precisions[2] = MFA_FP32;
  // "async" == TMA on B200: the tensor-core family loads with TMA and stores with plain st.global
  kd.prefer_async_load = tc ? 1 : 0;
  kd.prefer_async_store = 0;
  kd.has_transpose_state = 1;
  kd.transpose_A = d->transpose_A ? 1 : 0;
  kd.transpose_B = d->transpose_B ? 1 : 0;
  *out = kd;
  return MFA_SUCCESS;
}

int mfa_gemm_kernel_create(const mfa_gemm_kernel_descriptor_t *kd, mfa_gemm_kernel_t **out) {
  if (!kd || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  // guard let blockDimensions, memoryPrecisions, preferAsyncStore, registerPrecisions, splits, transposeState
  // (GEMMKernel.swift:27-34)
  if (!kd->has_block_dimensions || !kd->has_memory_precisions || kd->prefer_async_store == 0xFF ||
      !kd->has_register_precisions || !kd->has_splits || !kd->has_transpose_state)
    return fail(MFA_ERROR_INCOMPLETE_DESCRIPTOR, "Descriptor was incomplete.");
  for (int i = 0; i < 3; ++i)
    if (!valid_precision(kd->memory_precisions[i]) || !valid_precision(kd->register_precisions[i]))
      return fail(MFA_ERROR_INVALID_ARGUMENT, "Unrecognized precision.");
  // truth table (:46-97)
  static const char *kOperand[3] = {"A", "B", "C"};
  for (int i = 0; i < 3; ++i)
    if (!register_pair_valid(kd->memory_precisions[i], kd->register_precisions[i]))
      return fail(MFA_ERROR_INVALID_PRECISIONS,
                  std::string("Operand ") + kOperand[i] + " had an invalid register precision.");
  if (kd->register_precisions[2] == MFA_BF16)
    return fail(MFA_ERROR_INVALID_PRECISIONS, "BF16 cannot be used as the register precision for C.");

  const bool tA = kd->transpose_A != 0, tB = kd->transpose_B != 0;
  mfa_gemm_kernel *k = new mfa_gemm_kernel();
  k->descriptor = *kd;
  k->backend = kd->backend;
  if (k->backend == MFA_BACKEND_TCGEN05) {
    if (!tensor_core_inputs(kd->memory_precisions[0], kd->memory_precisions[1])) {
      delete k;
      return fail(MFA_ERROR_UNSUPPORTED,
                  "MFA_BACKEND_TCGEN05 needs A and B both FP16 or both BF16; use MFA_BACKEND_SIMT_FP32 for this "
                  "descriptor.");
    }
    k->block[0] = kTcGemmBlockM;
    k->block[1] = kTcGemmBlockN;
    k->block[2] = kTcGemmBlockK;
    k->threads = kTcGemmThreads;
    k->smem_bytes = tcgen05_gemm_smem_bytes();
  } else if (k->backend == MFA_BACKEND_SIMT_FP32) {
    k->block[0] = kSimtGemmBlockM;
    k->block[1] = kSimtGemmBlockN;
    k->block[2] = kSimtGemmBlockK;
    k->threads = kSimtGemmThreads;
    k->smem_bytes = simt_gemm_smem_bytes();
  } else {
    delete k;
    return fail(MFA_ERROR_INVALID_ARGUMENT, "Unrecognized backend.");
  }
  // The kernel object reports the tile shape the compiled kernel really uses; edits away from it are rejected.
  for (int i = 0; i < 3; ++i)
    if (kd->block_dimensions[i] != k->block[i]) {
      std::string msg = "Block dimensions " + std::to_string(kd->block_dimensions[0]) + "x" +
                        std::to_string(kd->block_dimensions[1]) + "x" + std::to_string(kd->block_dimensions[2]) +
                        " have no compiled sm_100a kernel (available: " + std::to_string(k->block[0]) + "x" +
                        std::to_string(k->block[1]) + "x" + std::to_string(k->block[2]) + ").";
      delete k;
      return fail(MFA_ERROR_UNSUPPORTED, msg);
    }
  if (kd->has_leading_block_dimensions) {
    uint16_t expected[3];
    leading_block_dimensions(k->block, tA, tB, expected);
    for (int i = 0; i < 3; ++i) {
      if (kd->leading_block_dimensions[i] < expected[i]) {  // GEMMKernel.swift:122-124
        delete k;
        return fail(MFA_ERROR_INVALID_ARGUMENT, "Leading block dimension was too small.");
      }
      if (kd->leading_block_dimensions[i] != expected[i]) {
        delete k;
        return fail(MFA_ERROR_UNSUPPORTED, "Padded leading block dimensions have no compiled sm_100a kernel.");
      }
    }
  }
  k->source_name = std::string("gemm_") + (k->backend == MFA_BACKEND_TCGEN05 ? "tcgen05" : "simt_fp32") + "<" +
                   mfa_precision_name((mfa_precision_t)kd->memory_precisions[0]) + ", " +
                   mfa_precision_name((mfa_precision_t)kd->memory_precisions[1]) + ", " +
                   mfa_precision_name((mfa_precision_t)kd->memory_precisions[2]) + ", " + (tA ? "T" : "N") +
                   (tB ? "T" : "N") + ">";
  *out = k;
  return MFA_SUCCESS;
}

void mfa_gemm_kernel_destroy(mfa_gemm_kernel_t *kernel) { delete kernel; }

int mfa_gemm_kernel_block_dimensions(const mfa_gemm_kernel_t *kernel, uint16_t out[3]) {
  if (!kernel || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  std::memcpy(out, kernel->block, sizeof(kernel->block));
  return MFA_SUCCESS;
}

int mfa_gemm_kernel_threadgroup_size(const mfa_gemm_kernel_t *kernel, uint32_t *out) {
  if (!kernel || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  *out = kernel->threads;
  return MFA_SUCCESS;
}

int mfa_gemm_kernel_threadgroup_memory_allocation(const mfa_gemm_kernel_t *kernel, uint32_t *out) {
  if (!kernel || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  *out = kernel->smem_bytes;
  return MFA_SUCCESS;
}

int mfa_gemm_kernel_grid_size(const mfa_gemm_kernel_t *kernel, const mfa_gemm_function_constants_t *c, uint32_t *out) {
  if (!kernel || !c || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  const uint64_t tiles = static_cast<uint64_t>((c->N + kernel->block[1] - 1) / kernel->block[1]) *
                         ((c->M + kernel->block[0] - 1) / kernel->block[0]) * batch_of(*c);
  *out = static_cast<uint32_t>(tiles);
  return MFA_SUCCESS;
}

int mfa_gemm_kernel_launch_count(const mfa_gemm_kernel_t *kernel, const mfa_gemm_function_constants_t *c,
                                 uint32_t *out) {
  if (!kernel || !c || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  *out = 1;
  if (kernel->backend == MFA_BACKEND_TCGEN05) {
    if (c->leading_dimensions[0] % 8 != 0) *out += 1;
    if (c->leading_dimensions[1] % 8 != 0) *out += 1;
  }
  return MFA_SUCCESS;
}

const char *mfa_gemm_kernel_source_name(const mfa_gemm_kernel_t *kernel) {
  return kernel ? kernel->source_name.c_str() : "";
}

int mfa_gemm_kernel_encode(const mfa_gemm_kernel_t *kernel, const mfa_gemm_function_constants_t *c,
                           void *const buffers[MFA_GEMM_BUFFER_COUNT], void *cuda_stream) {
  if (!kernel || !c || !buffers) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  int status = check_device();
  if (status != MFA_SUCCESS) return status;
  if (c->M == 0 || c->N == 0 || c->K == 0) return fail(MFA_ERROR_INVALID_ARGUMENT, "M, N and K must be at least 1.");
  const mfa_gemm_kernel_descriptor_t &kd = kernel->descriptor;
  const bool tA = kd.transpose_A != 0, tB = kd.transpose_B != 0;
  const uint32_t minimum[3] = {tA ? c->M : c->K, tB ? c->K : c->N, c->N};
  for (int i = 0; i < 3; ++i) {
    if (c->leading_dimensions[i] < minimum[i])
      return fail(MFA_ERROR_INVALID_ARGUMENT, "Leading block dimension was too small.");
    if (!buffers[i])
      return fail(MFA_ERROR_INVALID_ARGUMENT, std::string("Buffer ") + "ABC"[i] + " (binding " + std::to_string(i) +
                                                  ") is NULL.");
  }
  GemmParams p;
  p.M = c->M;
  p.N = c->N;
  p.K = c->K;
  p.batch = batch_of(*c);
  p.lda = c->leading_dimensions[0];
  p.ldb = c->leading_dimensions[1];
  p.ldc = c->leading_dimensions[2];
  p.A = buffers[0];
  p.B = buffers[1];
  p.C = buffers[2];
  p.precA = kd.memory_precisions[0];
  p.precB = kd.memory_precisions[1];
  p.precC = kd.memory_precisions[2];
  p.transA = tA;
  p.transB = tB;
  p.load_previous_C = c->load_previous_C ? 1 : 0;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  const cudaError_t e =
      kernel->backend == MFA_BACKEND_TCGEN05 ? launch_tcgen05_gemm(p, stream) : launch_simt_gemm(p, stream);
  if (e != cudaSuccess)
    return fail(MFA_ERROR_CUDA, std::string("launch of ") + kernel->source_name + " failed: " + cudaGetErrorString(e) +
                                    " " + last_launch_detail());
  return MFA_SUCCESS;
}

// ------------------------------------------------------------------------------------------------
// Pipeline cache (GEMMDescriptor+PipelineCache.swift:16-36).  The reference keys on the whole GEMMDescriptor because its
// kernels specialise on M, N, K through function constants; here those are launch arguments, so the key is what
// GEMMKernelDescriptor(descriptor:) reads: the memory precisions and the transposes.
// ------------------------------------------------------------------------------------------------
namespace {
struct GemmCacheKey {
  uint8_t precisions[3];
  uint8_t transpose_A, transpose_B;
};
std::mutex g_gemm_cache_mutex;
std::vector<std::pair<GemmCacheKey, mfa_gemm_kernel_t *>> g_gemm_cache;
}  // namespace

int mfa_gemm_kernel_cache_fetch(const mfa_gemm_descriptor_t *descriptor, const mfa_gemm_kernel_t **out) {
  if (!descriptor || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  mfa_gemm_kernel_descriptor_t kd;
  int status = mfa_gemm_descriptor_kernel_descriptor(descriptor, &kd);  // validates completeness first
  if (status != MFA_SUCCESS) return status;
  GemmCacheKey key;
  std::memcpy(key.precisions, descriptor->memory_precisions, 3);
  key.transpose_A = descriptor->transpose_A ? 1 : 0;
  key.transpose_B = descriptor->transpose_B ? 1 : 0;
  std::lock_guard<std::mutex> lock(g_gemm_cache_mutex);
  for (const auto &entry : g_gemm_cache)
    if (std::memcmp(entry.first.precisions, key.precisions, 3) == 0 && entry.first.transpose_A == key.transpose_A &&
        entry.first.transpose_B == key.transpose_B) {
      *out = entry.second;
      return MFA_SUCCESS;
    }
  mfa_gemm_kernel_t *kernel = nullptr;
  if ((status = mfa_gemm_kernel_create(&kd, &kernel)) != MFA_SUCCESS) return status;
  g_gemm_cache.push_back({key, kernel});
  *out = kernel;
  return MFA_SUCCESS;
}

int mfa_gemm_kernel_cache_size(void) {
  std::lock_guard<std::mutex> lock(g_gemm_cache_mutex);
  return static_cast<int>(g_gemm_cache.size());
}

}  // extern "C"

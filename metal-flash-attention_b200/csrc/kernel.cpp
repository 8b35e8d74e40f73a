// AttentionKernel side of the C ABI: handle creation/validation, launch geometry, and encode()
// -- the compile + bind + dispatch the reference leaves to its caller
// (Tests/FlashAttentionTests/Attention/SquareAttentionTest.swift:240-372).
// Mirrors Sources/FlashAttention/Attention/AttentionKernel/AttentionKernel.swift.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "internal.h"
#include "kernels/device_state.h"
#include "kernels/tma_host.h"

namespace mfa {
// The tcgen05 kernel that serves a descriptor; decided once, when the kernel object is created.
enum class Tcgen05Family : uint8_t {
  kForward,           // row-major, pad8(D) <= 128 (tcgen05_forward.cu)
  kForwardWide,       // row-major, 128 < pad8(D) <= 256 (tcgen05_forward_d256.cu)
  kForwardGeneric,    // transposed operands (tcgen05_forward_d256.cu)
  kBackward,          // row-major, pad8(D) <= 128 (tcgen05_backward.cu)
  kBackwardGeneric,   // transposed operands, or pad8(D) > 128 (tcgen05_backward_generic.cu)
};

// `transposed`: any of the operands the launchers look at is transposed -- Q, K, V, O for the forward, all eight matrix
// operands for the backward kernels
static Tcgen05Family tcgen05_family(int type, uint32_t padded_head, bool transposed) {
  if (type == MFA_FORWARD)
    return transposed ? Tcgen05Family::kForwardGeneric
                      : (padded_head > 128 ? Tcgen05Family::kForwardWide : Tcgen05Family::kForward);
  return transposed || padded_head > 128 ? Tcgen05Family::kBackwardGeneric : Tcgen05Family::kBackward;
}
}  // namespace mfa

struct mfa_attention_kernel {
  mfa_attention_kernel_descriptor_t descriptor;
  int type;
  int backend;
  mfa::Tcgen05Family family;  // (backend == MFA_BACKEND_TCGEN05 only)
  uint32_t threads, smem_bytes, par, trav, head;
  std::string source_name;
};

namespace mfa {

// loadFunction / storeFunction legality (AttentionKernel.swift:81-139): a 16-bit memory format may
// only be widened to FP32 or kept as is; FP32 memory can only be FP32 in registers.
static bool precision_pair_valid(int memory, int reg) {
  if (memory == MFA_FP16) return reg == MFA_FP16 || reg == MFA_FP32;
  if (memory == MFA_BF16) return reg == MFA_BF16 || reg == MFA_FP32;
  if (memory == MFA_FP32) return reg == MFA_FP32;
  return false;
}

static const int *operands_of(int type, int *count) {
  static const int fwd[] = {MFA_Q, MFA_K, MFA_V, MFA_O, MFA_L};
  static const int dq[] = {MFA_Q, MFA_K, MFA_V, MFA_O, MFA_L, MFA_D, MFA_dO, MFA_dQ};
  static const int dkv[] = {MFA_Q, MFA_K, MFA_V, MFA_L, MFA_D, MFA_dO, MFA_dV, MFA_dK};
  switch (type) {
    case MFA_FORWARD: *count = 5; return fwd;
    case MFA_BACKWARD_QUERY: *count = 8; return dq;
    default: *count = 8; return dkv;
  }
}

// sm_100 check of the current device, cached per device ordinal (encode() of a microsecond-scale kernel must not pay
// two runtime queries per call)
int check_device() {
  const int device = current_device();
  if (device < 0)
    return fail(MFA_ERROR_NO_DEVICE, "No CUDA device (cudaGetDevice failed; this library has no CPU fallback).");
  static std::mutex mutex;
  static int8_t verdict[kMaxDevices] = {};  // 0 unknown, 1 sm_100, -1 other
  if (device < kMaxDevices) {
    std::lock_guard<std::mutex> lock(mutex);
    if (verdict[device] == 1) return MFA_SUCCESS;
  }
  int major = 0;
  cudaError_t e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
  if (e != cudaSuccess) return fail(MFA_ERROR_NO_DEVICE, std::string("cudaDeviceGetAttribute: ") + cudaGetErrorString(e));
  if (major != 10)
    return fail(MFA_ERROR_NO_DEVICE, "Device is not sm_100 (compute capability " + std::to_string(major) +
                                         ".x); these kernels are built for sm_100a only.");
  if (device < kMaxDevices) {
    std::lock_guard<std::mutex> lock(mutex);
    verdict[device] = 1;
  }
  return MFA_SUCCESS;
}

static int build_params(const mfa_attention_kernel *k, const mfa_function_constants_t *c, void *const buffers[],
                        AttentionParams &p) {
  if (c->row == 0 || c->column == 0) return fail(MFA_ERROR_INVALID_ARGUMENT, "R and C must be at least 1.");
  p.R = c->row;
  p.C = c->column;
  p.D = k->descriptor.head_dimension;
  p.batch = c->batch_count ? c->batch_count : 1;
  for (int s = 0; s < kSlots; ++s) {
    p.buf[s] = buffers[s];
    uint8_t mp = k->descriptor.memory_precisions[s];
    p.prec[s] = mp == 0xFF ? 0 : mp;
    p.transposed[s] = (k->descriptor.transpose_state_mask >> s) & 1;
  }
  // dotProductScale (AttentionKernel+Softmax.swift:17-26)
  p.scale = 1.0f / std::sqrt(static_cast<float>(p.D));
  p.scale_log2 = 1.442695041f * p.scale;
  // the tuning columns of the parameter-table row this kernel was created from
  p.exp2_fma_quarters = k->descriptor.exp2_fma_quarters;
  p.split_min_blocks = k->descriptor.split_min_blocks;
  p.split_max = k->descriptor.split_max ? k->descriptor.split_max : 1;
  int n = 0;
  const int *ops = operands_of(k->type, &n);
  for (int i = 0; i < n; ++i)
    if (buffers[ops[i]] == nullptr)
      return fail(MFA_ERROR_INVALID_ARGUMENT, std::string("Buffer ") + mfa_operand_name((mfa_operand_t)ops[i]) +
                                                  " (binding " + std::to_string(ops[i]) + ") is NULL.");
  return MFA_SUCCESS;
}

// The encode-time checks (R and C against the TMA pitch rule for transposed operands, output precisions) come after the
// head-dimension padding copies have been queued, then the kernel chosen at creation is launched.
static cudaError_t launch_tcgen05(const mfa_attention_kernel *k, const AttentionParams &p, cudaStream_t stream) {
  const bool key_value = k->type == MFA_BACKWARD_KEY_VALUE;
  if (k->type == MFA_FORWARD && !tcgen05_forward_supported(p)) {
    set_launch_detail("descriptor is outside the tcgen05 forward kernel's domain");
    return cudaErrorInvalidValue;
  }
  if (k->type != MFA_FORWARD && !tcgen05_backward_supported(p)) {
    set_launch_detail("descriptor is outside the tcgen05 backward kernels' domain");
    return cudaErrorInvalidValue;
  }
  switch (k->family) {
    case Tcgen05Family::kForward: return launch_tcgen05_forward(p, stream);
    case Tcgen05Family::kForwardWide: return launch_tcgen05_forward_d256(p, stream);
    case Tcgen05Family::kForwardGeneric: return launch_tcgen05_forward_generic(p, stream);
    case Tcgen05Family::kBackward: return launch_tcgen05_backward(p, stream, key_value);
    case Tcgen05Family::kBackwardGeneric: return launch_tcgen05_backward_generic(p, stream, key_value);
  }
  return cudaErrorInvalidValue;
}

}  // namespace mfa

using namespace mfa;

extern "C" {

int mfa_attention_kernel_create(const mfa_attention_kernel_descriptor_t *kd, mfa_attention_kernel_t **out) {
  if (!kd || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  // guard let ... else fatalError("Descriptor was incomplete.")  (AttentionKernel.swift:28-34)
  if (!kd->has_block_dimensions || !kd->has_head_dimension || kd->prefer_async_cache == 0xFF ||
      kd->prefer_async_load == 0xFF || kd->type == 0xFF)
    return fail(MFA_ERROR_INCOMPLETE_DESCRIPTOR, "Descriptor was incomplete.");
  if (kd->type > MFA_BACKWARD_KEY_VALUE) return fail(MFA_ERROR_INVALID_ARGUMENT, "Unrecognized kernel type.");
  if (kd->head_dimension == 0) return fail(MFA_ERROR_INVALID_ARGUMENT, "Head dimension must be at least 1.");

  int n = 0;
  const int *ops = operands_of(kd->type, &n);
  for (int i = 0; i < n; ++i) {
    int op = ops[i];
    uint8_t mem = kd->memory_precisions[op], reg = kd->register_precisions[op];
    if (mem == 0xFF || reg == 0xFF)
      return fail(MFA_ERROR_INCOMPLETE_DESCRIPTOR,
                  std::string("Precision of ") + mfa_operand_name((mfa_operand_t)op) + " was not specified.");
    if (!precision_pair_valid(mem, reg)) return fail(MFA_ERROR_INVALID_PRECISIONS, "Invalid precisions.");
    if (op != MFA_L && op != MFA_D && !((kd->transpose_state_valid_mask >> op) & 1))
      return fail(MFA_ERROR_INCOMPLETE_DESCRIPTOR,
                  std::string("Transpose state of ") + mfa_operand_name((mfa_operand_t)op) + " was not specified.");
  }

  mfa_attention_kernel *k = new mfa_attention_kernel();
  k->descriptor = *kd;
  k->type = kd->type;
  k->backend = kd->backend;
  const uint32_t D = kd->head_dimension;

  if (k->backend == MFA_BACKEND_TCGEN05) {
    // The tcgen05 kernels only exist for 16-bit row-major operands; reject descriptors edited into
    // something they cannot serve instead of silently computing something else.
    const uint8_t pq = kd->memory_precisions[MFA_Q];
    const uint32_t Dp = (D + 7) / 8 * 8;  // D % 8 != 0: operands are staged with pad8(D) columns (kernels/pad_head.cu)
    bool ok = (pq == MFA_FP16 || pq == MFA_BF16) && kd->memory_precisions[MFA_K] == pq &&
              kd->memory_precisions[MFA_V] == pq &&
              Dp <= (k->type == MFA_FORWARD ? tcgen05_forward_max_head() : tcgen05_backward_max_head());
    bool transposed = false;
    for (int i = 0; i < n; ++i)
      if ((kd->transpose_state_mask >> ops[i]) & 1) transposed = true;
    if (transposed && D % 8 != 0) ok = false;  // padding is implemented for row-major operands
    // dO: same element type, or BF16 beside FP16 Q/K/V (the reference's policy; converted on chip)
    if (k->type != MFA_FORWARD && kd->memory_precisions[MFA_dO] != pq &&
        !(pq == MFA_FP16 && kd->memory_precisions[MFA_dO] == MFA_BF16))
      ok = false;
    if (!ok) {
      delete k;
      return fail(MFA_ERROR_UNSUPPORTED,
                  "MFA_BACKEND_TCGEN05 needs FP16/BF16 Q,K,V (row-major for head % 8 != 0; dO of the same "
                  "type, or BF16 with FP16 Q,K,V) and pad8(head) <= the compiled maximum; use MFA_BACKEND_SIMT_FP32 for this "
                  "descriptor.");
    }
    // tuning columns: every compiled exp2 variant is accepted, anything else is rejected with the list of what exists
    const uint32_t max_quarters = k->type == MFA_FORWARD ? kMaxForwardExp2Quarters : kMaxBackwardExp2Quarters;
    if (kd->exp2_fma_quarters > max_quarters) {
      delete k;
      return fail(MFA_ERROR_UNSUPPORTED, "exp2-on-FMA-pipe fraction " + std::to_string(kd->exp2_fma_quarters) +
                                             "/4 has no compiled sm_100a kernel (available: 0.." +
                                             std::to_string(max_quarters) + ").");
    }
    constexpr uint16_t kForwardMatrices = (1u << MFA_Q) | (1u << MFA_K) | (1u << MFA_V) | (1u << MFA_O);
    constexpr uint16_t kAllMatrices = kForwardMatrices | (1u << MFA_dO) | (1u << MFA_dV) | (1u << MFA_dK) | (1u << MFA_dQ);
    const uint16_t routed = k->type == MFA_FORWARD ? kForwardMatrices : kAllMatrices;
    k->family = tcgen05_family(k->type, Dp, (kd->transpose_state_mask & routed) != 0);
    switch (k->family) {
      case Tcgen05Family::kForward:
        tcgen05_forward_geometry(Dp, &k->threads, &k->smem_bytes, &k->par, &k->trav, &k->head);
        break;
      case Tcgen05Family::kForwardWide:
      case Tcgen05Family::kForwardGeneric:
        tcgen05_forward_generic_geometry(Dp, &k->threads, &k->smem_bytes, &k->par, &k->trav, &k->head);
        break;
      case Tcgen05Family::kBackward:
        tcgen05_backward_geometry(k->type, Dp, &k->threads, &k->smem_bytes, &k->par, &k->trav, &k->head);
        break;
      case Tcgen05Family::kBackwardGeneric:
        tcgen05_backward_generic_geometry(k->type, Dp, &k->threads, &k->smem_bytes, &k->par, &k->trav, &k->head);
        break;
    }
  } else if (k->backend == MFA_BACKEND_SIMT_FP32) {
    if (D > 512) {
      delete k;
      return fail(MFA_ERROR_UNSUPPORTED, "Head dimension " + std::to_string(D) + " exceeds 512.");
    }
    simt_geometry(k->type, D, &k->threads, &k->smem_bytes, &k->par, &k->trav, &k->head);
  } else {
    delete k;
    return fail(MFA_ERROR_INVALID_ARGUMENT, "Unrecognized backend.");
  }
  // The kernel object reports the tile shape the compiled kernel really uses; a descriptor whose
  // block dimensions were edited away from a compiled configuration is rejected.
  if (kd->block_parallelization != k->par || kd->block_traversal != k->trav) {
    std::string msg = "Block dimensions " + std::to_string(kd->block_parallelization) + "x" +
                      std::to_string(kd->block_traversal) + " have no compiled sm_100a kernel (available: " +
                      std::to_string(k->par) + "x" + std::to_string(k->trav) + ").";
    delete k;
    return fail(MFA_ERROR_UNSUPPORTED, msg);
  }
  static const char *typeNames[] = {"forward", "backward_query", "backward_key_value"};
  // the exp2 column selects an instantiation of the D <= 128 row-major kernels only
  const bool exp2_variants = k->backend == MFA_BACKEND_TCGEN05 &&
                             (k->family == Tcgen05Family::kForward || k->family == Tcgen05Family::kBackward);
  k->source_name = std::string("attention_") + typeNames[k->type] +
                   (k->backend == MFA_BACKEND_TCGEN05 ? "_tcgen05" : "_simt_fp32") + "<D=" + std::to_string(D) +
                   (exp2_variants && kd->exp2_fma_quarters
                        ? ", exp2 on FMA pipe " + std::to_string(kd->exp2_fma_quarters) + "/4"
                        : std::string()) +
                   ">";
  *out = k;
  return MFA_SUCCESS;
}

void mfa_attention_kernel_destroy(mfa_attention_kernel_t *kernel) { delete kernel; }

int mfa_attention_kernel_block_dimensions(const mfa_attention_kernel_t *kernel, uint16_t out[3]) {
  if (!kernel || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  out[0] = static_cast<uint16_t>(kernel->par);
  out[1] = static_cast<uint16_t>(kernel->trav);
  out[2] = static_cast<uint16_t>(kernel->head);
  return MFA_SUCCESS;
}

int mfa_attention_kernel_threadgroup_size(const mfa_attention_kernel_t *kernel, uint32_t *out) {
  if (!kernel || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  *out = kernel->threads;
  return MFA_SUCCESS;
}

int mfa_attention_kernel_threadgroup_memory_allocation(const mfa_attention_kernel_t *kernel, uint32_t *out) {
  if (!kernel || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  *out = kernel->smem_bytes;
  return MFA_SUCCESS;
}

int mfa_attention_kernel_grid_size(const mfa_attention_kernel_t *kernel, const mfa_function_constants_t *c,
                                   uint32_t *out) {
  if (!kernel || !c || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  // parallelization dimension: R for forward / backwardQuery, C for backwardKeyValue
  // (AttentionKernel.swift:197-204; dispatch: SquareAttentionTest.swift:328-339)
  const uint32_t dim = kernel->type == MFA_BACKWARD_KEY_VALUE ? c->column : c->row;
  const uint32_t batch = c->batch_count ? c->batch_count : 1;
  *out = ((dim + kernel->par - 1) / kernel->par) * batch;
  return MFA_SUCCESS;
}

const char *mfa_attention_kernel_source_name(const mfa_attention_kernel_t *kernel) {
  return kernel ? kernel->source_name.c_str() : "";
}

int mfa_attention_kernel_launch_count(const mfa_attention_kernel_t *kernel, const mfa_function_constants_t *c,
                                      uint32_t *out) {
  if (!kernel || !c || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  *out = 1;
  if (kernel->backend != MFA_BACKEND_TCGEN05) return MFA_SUCCESS;
  const mfa_attention_kernel_descriptor_t &kd = kernel->descriptor;
  const uint32_t Dp = (kd.head_dimension + 7u) / 8u * 8u;
  const uint32_t b = c->batch_count ? c->batch_count : 1;
  const bool convert = kd.memory_precisions[MFA_dO] != kd.memory_precisions[MFA_Q];
  switch (kernel->family) {
    case Tcgen05Family::kForward:
      *out = tcgen05_forward_launch_count(c->row, c->column, b, kd.split_min_blocks, kd.split_max);
      break;
    case Tcgen05Family::kForwardWide:
    case Tcgen05Family::kForwardGeneric:
      break;  // (these never split)
    case Tcgen05Family::kBackward:
      *out = tcgen05_backward_launch_count(kernel->type, c->row, c->column, b, kd.split_min_blocks, kd.split_max, convert);
      break;
    case Tcgen05Family::kBackwardGeneric:
      *out = tcgen05_backward_generic_launch_count(kernel->type, c->row, c->column, Dp, b, kd.split_min_blocks, kd.split_max,
                                                   convert);
      break;
  }
  // head % 8 != 0: one padding copy per staged input, one un-padding copy per output
  if (kd.head_dimension % 8 != 0) *out += kernel->type == MFA_FORWARD ? 4 : 6;
  return MFA_SUCCESS;
}

int mfa_attention_kernel_encode(const mfa_attention_kernel_t *kernel, const mfa_function_constants_t *constants,
                                void *const buffers[MFA_BUFFER_COUNT], void *cuda_stream) {
  if (!kernel || !constants || !buffers) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  int status = check_device();
  if (status != MFA_SUCCESS) return status;
  AttentionParams p;
  status = build_params(kernel, constants, buffers, p);
  if (status != MFA_SUCCESS) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);

  // Several kernels carry the batch in gridDim.y (limit 65535; the SIMT dK/dV kernel multiplies it by up to four head
  // slices): larger batches go out as several launches over slices of the batch -- the problems are independent and
  // stored back to back, so a slice is just a pointer offset.
  constexpr uint32_t kMaxBatchPerLaunch = 16384;
  const uint32_t batch = p.batch;
  size_t head_bytes[kSlots];
  for (int slot = 0; slot < kSlots; ++slot) {
    const size_t seq = (slot == sK || slot == sV || slot == sdK || slot == sdV) ? p.C : p.R;
    const size_t elements = (slot == sL || slot == sD) ? seq : seq * p.D;
    head_bytes[slot] = elements * (p.prec[slot] == FP32 ? 4 : 2);
  }
  // D % 8 != 0 on the tensor-core family: stage the operands with pad8(D) columns, run the kernels at the padded head
  // dimension (the softmax scale stays 1 / sqrt(D) of the true D), copy the FP32 outputs back without the padding.
  const bool padded = kernel->backend == MFA_BACKEND_TCGEN05 && p.D % 8 != 0;
  const uint32_t Dp = (p.D + 7) / 8 * 8;
  const int device = padded ? current_device() : 0;
  for (uint32_t h0 = 0; h0 < batch; h0 += kMaxBatchPerLaunch) {
    AttentionParams q = p;
    q.batch = batch - h0 < kMaxBatchPerLaunch ? batch - h0 : kMaxBatchPerLaunch;
    for (int slot = 0; slot < kSlots; ++slot)
      if (q.buf[slot]) q.buf[slot] = static_cast<char *>(q.buf[slot]) + head_bytes[slot] * h0;
    cudaError_t e = cudaSuccess;
    void *user_out[kSlots] = {};  // padded path: where the un-padded outputs go
    if (padded) {
      // operands with a head dimension, by kernel type: inputs are staged, outputs are computed into staging
      static const int fwd_in[] = {sQ, sK, sV}, fwd_out[] = {sO};
      static const int dq_in[] = {sQ, sK, sV, sO, sdO}, dq_out[] = {sdQ};
      static const int dkv_in[] = {sQ, sK, sV, sdO}, dkv_out[] = {sdV, sdK};
      const int *ins = kernel->type == MFA_FORWARD ? fwd_in : (kernel->type == MFA_BACKWARD_QUERY ? dq_in : dkv_in);
      const int nin = kernel->type == MFA_FORWARD ? 3 : (kernel->type == MFA_BACKWARD_QUERY ? 5 : 4);
      const int *outs = kernel->type == MFA_FORWARD ? fwd_out : (kernel->type == MFA_BACKWARD_QUERY ? dq_out : dkv_out);
      const int nout = kernel->type == MFA_BACKWARD_KEY_VALUE ? 2 : 1;
      auto rows_of = [&](int slot) -> uint64_t {
        return static_cast<uint64_t>(q.batch) * ((slot == sK || slot == sV || slot == sdK || slot == sdV) ? p.C : p.R);
      };
      auto bytes_of = [&](int slot) -> size_t {
        return ((rows_of(slot) * Dp * (p.prec[slot] == FP32 ? 4 : 2)) + 255) & ~size_t(255);
      };
      size_t total = 0;
      for (int i = 0; i < nin; ++i) total += bytes_of(ins[i]);
      for (int i = 0; i < nout; ++i) total += bytes_of(outs[i]);
      void *ws = nullptr;
      if ((e = workspace_for(device, stream, total, &ws, /*slot=*/1)) != cudaSuccess)
        return fail(MFA_ERROR_CUDA, std::string("padding workspace: ") + cudaGetErrorString(e) + " " + last_launch_detail());
      char *cursor = static_cast<char *>(ws);
      for (int i = 0; i < nin && e == cudaSuccess; ++i) {
        const int slot = ins[i];
        e = launch_pad_columns(q.buf[slot], cursor, rows_of(slot), p.D, Dp, p.prec[slot] == FP32 ? 4 : 2, stream);
        q.buf[slot] = cursor;
        cursor += bytes_of(slot);
      }
      for (int i = 0; i < nout; ++i) {
        const int slot = outs[i];
        user_out[slot] = q.buf[slot];
        q.buf[slot] = cursor;
        cursor += bytes_of(slot);
      }
      q.D = Dp;  // (q.scale / q.scale_log2 keep the true head dimension)
      if (e != cudaSuccess)
        return fail(MFA_ERROR_CUDA, std::string("head-dimension padding failed: ") + cudaGetErrorString(e));
    }
    if (kernel->backend == MFA_BACKEND_TCGEN05) {
      e = launch_tcgen05(kernel, q, stream);
    } else {
      switch (kernel->type) {
        case MFA_FORWARD: e = launch_simt_forward(q, stream); break;
        case MFA_BACKWARD_QUERY: e = launch_simt_backward_query(q, stream); break;
        default: e = launch_simt_backward_key_value(q, stream); break;
      }
    }
    if (e != cudaSuccess)
      return fail(MFA_ERROR_CUDA, std::string("launch of ") + kernel->source_name + " failed: " + cudaGetErrorString(e) +
                                      " " + last_launch_detail());
    if (padded) {
      for (int slot = 0; slot < kSlots && e == cudaSuccess; ++slot)
        if (user_out[slot]) {
          const uint64_t rows = static_cast<uint64_t>(q.batch) * ((slot == sdK || slot == sdV) ? p.C : p.R);
          e = launch_unpad_columns(q.buf[slot], user_out[slot], rows, p.D, Dp, stream);
        }
      if (e != cudaSuccess)
        return fail(MFA_ERROR_CUDA, std::string("head-dimension un-padding failed: ") + cudaGetErrorString(e));
    }
  }
  return MFA_SUCCESS;
}

// Debug-only export (deliberately absent from include/mfa_b200.h): forward with pipeline timestamps.
MFA_API int mfa_debug_forward_trace(const mfa_attention_kernel_t *kernel, const mfa_function_constants_t *constants,
                                    void *const buffers[MFA_BUFFER_COUNT], void *cuda_stream, long long *trace) {
  if (!kernel || !constants || !buffers || !trace) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  const bool row_major_forward = kernel->backend == MFA_BACKEND_TCGEN05 && (kernel->family == Tcgen05Family::kForward ||
                                                                           kernel->family == Tcgen05Family::kForwardWide);
  if (!row_major_forward)
    return fail(MFA_ERROR_INVALID_ARGUMENT, "Pipeline traces exist for the row-major tcgen05 forward kernels only.");
  AttentionParams p;
  int status = build_params(kernel, constants, buffers, p);
  if (status != MFA_SUCCESS) return status;
  cudaStream_t stream = static_cast<cudaStream_t>(cuda_stream);
  cudaError_t e = kernel->family == Tcgen05Family::kForwardWide ? launch_tcgen05_forward_d256_trace(p, stream, trace)
                                                                : launch_tcgen05_forward_trace(p, stream, trace);
  if (e != cudaSuccess) return fail(MFA_ERROR_CUDA, std::string("trace launch failed: ") + cudaGetErrorString(e));
  return MFA_SUCCESS;
}

// ------------------------------------------------------------------------------------------------
// Kernel cache keyed by descriptor -- the useful half of the reference's pipeline cache
// (GEMMKernel.pipelineCache / register(descriptor:), GEMM/GEMMDescriptor/GEMMDescriptor+PipelineCache.swift:16-36):
// the reference caches (kernel, MTLComputePipelineState) per problem descriptor because a Metal JIT compile costs
// milliseconds; here the kernels are compiled ahead of time, so what is worth keeping is the validated kernel object.
// Handles returned from the cache are owned by the library and live until process exit.
// ------------------------------------------------------------------------------------------------
namespace {
struct CacheKey {
  mfa_attention_descriptor_t descriptor;
  int type;
  unsigned table_generation;  // kernels created from an older parameter table are not handed out again
};
std::mutex g_cache_mutex;
std::vector<std::pair<CacheKey, mfa_attention_kernel_t *>> g_kernel_cache;

bool same_descriptor(const mfa_attention_descriptor_t &a, const mfa_attention_descriptor_t &b) {
  // field-wise (struct padding is not part of the value); the matrix dimensions R, C and the batch count are launch-time
  // constants (setFunctionConstants), not part of the kernel -- only the head dimension is
  return a.low_precision_inputs == b.low_precision_inputs &&
         a.low_precision_intermediates == b.low_precision_intermediates &&
         a.has_matrix_dimensions == b.has_matrix_dimensions && a.has_transpose_state == b.has_transpose_state &&
         a.head == b.head && a.transpose_Q == b.transpose_Q && a.transpose_K == b.transpose_K &&
         a.transpose_V == b.transpose_V && a.transpose_O == b.transpose_O &&
         a.input_precision_override == b.input_precision_override &&
         // with transposed operands the kernel family depends on R % 8 / C % 8 (TMA row pitch)
         select_backend(a, MFA_FORWARD) == select_backend(b, MFA_FORWARD);
}
}  // namespace

int mfa_attention_kernel_cache_fetch(const mfa_attention_descriptor_t *descriptor, mfa_kernel_type_t type,
                                     const mfa_attention_kernel_t **out) {
  if (!descriptor || !out) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  std::lock_guard<std::mutex> lock(g_cache_mutex);
  for (const auto &entry : g_kernel_cache)
    if (entry.first.type == static_cast<int>(type) && entry.first.table_generation == parameter_table_generation() &&
        same_descriptor(entry.first.descriptor, *descriptor)) {
      *out = entry.second;
      return MFA_SUCCESS;
    }
  mfa_attention_kernel_descriptor_t kd;
  int status = mfa_attention_descriptor_kernel_descriptor(descriptor, type, &kd);
  if (status != MFA_SUCCESS) return status;
  mfa_attention_kernel_t *kernel = nullptr;
  if ((status = mfa_attention_kernel_create(&kd, &kernel)) != MFA_SUCCESS) return status;
  g_kernel_cache.push_back({CacheKey{*descriptor, static_cast<int>(type), parameter_table_generation()}, kernel});
  *out = kernel;
  return MFA_SUCCESS;
}

int mfa_attention_kernel_cache_size(void) {
  std::lock_guard<std::mutex> lock(g_cache_mutex);
  return static_cast<int>(g_kernel_cache.size());
}

// ------------------------------------------------------------------------------------------------
// Host-buffer path: H2D -> kernels -> D2H (the end-to-end call bench.py times as `e2e`).
//
// The independent single-head problems of a batch are cut into chunks that flow through three streams -- upload,
// compute, download -- linked by one event pair per chunk, so the host->device copy of chunk i+1, the kernels of chunk
// i and the device->host copy of chunk i-1 overlap (PCIe is full duplex and the GPU has a copy engine per direction) and
// the upload stream never waits for anything.  With pinned host buffers the call then costs max(H2D, D2H) + one chunk
// of fill/drain instead of H2D + kernels + D2H.
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int kHostStreams = 3;  // 0 upload, 1 compute, 2 download
constexpr uint32_t kMaxChunks = 32;
struct Scratch {
  void *ptr[MFA_BUFFER_COUNT] = {};
  size_t bytes[MFA_BUFFER_COUNT] = {};
  bool ready = false;  // streams and events exist
  cudaStream_t stream[kHostStreams] = {};
  cudaEvent_t uploaded[kMaxChunks] = {}, computed[kMaxChunks] = {};
};
// One scratch set per (calling thread, device): a thread that alternates between devices keeps both sets, nothing
// leaks on a device switch, and a set is only marked ready once every stream and event exists.  Released by
// mfa_release_device_resources() (thread exit does not free device memory: the context may already be gone).
thread_local std::map<int, Scratch> g_scratch;

// RAII: mfa_attention_run_host selects `device` for the duration of the call and restores the caller's device
struct DeviceGuard {
  int previous = -1;
  bool active = false;
  cudaError_t enter(int device) {
    if (cudaGetDevice(&previous) != cudaSuccess) {
      cudaGetLastError();
      previous = -1;
    }
    cudaError_t e = cudaSetDevice(device);
    active = e == cudaSuccess && previous >= 0 && previous != device;
    return e;
  }
  ~DeviceGuard() {
    if (active) cudaSetDevice(previous);
  }
};

void destroy_scratch(Scratch &s) {
  for (int i = 0; i < MFA_BUFFER_COUNT; ++i) {
    if (s.ptr[i]) cudaFree(s.ptr[i]);
    s.ptr[i] = nullptr;
    s.bytes[i] = 0;
  }
  for (int i = 0; i < kHostStreams; ++i)
    if (s.stream[i]) cudaStreamDestroy(s.stream[i]);
  for (uint32_t i = 0; i < kMaxChunks; ++i) {
    if (s.uploaded[i]) cudaEventDestroy(s.uploaded[i]);
    if (s.computed[i]) cudaEventDestroy(s.computed[i]);
  }
  s = Scratch();
}

// heads per chunk: about sixteen chunks (fill + drain = two chunk times), but no chunk smaller than ~4 MB of traffic
// (copy launch overheads), at most kMaxChunks chunks, and no chunking at all for a single problem
uint32_t chunk_heads(uint32_t batch, size_t bytes_per_head) {
  if (batch <= 1) return 1;
  // tuning knob (scripts/gpu_runs: chunk-count sweep of the host-buffer path): MFA_B200_HOST_CHUNKS=<n>
  if (const char *env = getenv("MFA_B200_HOST_CHUNKS")) {
    const uint32_t n = static_cast<uint32_t>(atoi(env));
    if (n >= 1 && n <= kMaxChunks) return (batch + n - 1) / n;
  }
  uint32_t heads = (batch + 15) / 16;
  const size_t kMinChunkBytes = size_t(4) << 20;
  if (bytes_per_head * heads < kMinChunkBytes)
    heads = static_cast<uint32_t>((kMinChunkBytes + bytes_per_head - 1) / bytes_per_head);
  if ((batch + heads - 1) / heads > kMaxChunks) heads = (batch + kMaxChunks - 1) / kMaxChunks;
  return heads < batch ? heads : batch;
}
}  // namespace

int mfa_attention_run_host(const mfa_attention_descriptor_t *descriptor, uint32_t run_mask,
                           void *const host_buffers[MFA_BUFFER_COUNT], int device) {
  if (!descriptor || !host_buffers) return fail(MFA_ERROR_INVALID_ARGUMENT, "NULL argument.");
  if (!(run_mask & 7u)) return fail(MFA_ERROR_INVALID_ARGUMENT, "run_mask selects no kernel.");
  DeviceGuard guard;  // the caller's current device is restored on every exit
  cudaError_t e = guard.enter(device);
  if (e != cudaSuccess)
    return fail(MFA_ERROR_NO_DEVICE, std::string("cudaSetDevice: ") + cudaGetErrorString(e) +
                                         " (this library has no CPU fallback).");
  Scratch &s = g_scratch[device];
  if (!s.ready) {
    for (int i = 0; i < kHostStreams && e == cudaSuccess; ++i)
      e = cudaStreamCreateWithFlags(&s.stream[i], cudaStreamNonBlocking);
    for (uint32_t i = 0; i < kMaxChunks && e == cudaSuccess; ++i) {
      e = cudaEventCreateWithFlags(&s.uploaded[i], cudaEventDisableTiming);
      if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.computed[i], cudaEventDisableTiming);
    }
    if (e != cudaSuccess) {
      destroy_scratch(s);  // never leave a half-initialised set behind
      return fail(MFA_ERROR_CUDA, std::string("stream / event creation: ") + cudaGetErrorString(e));
    }
    s.ready = true;
  }

  // which operands each kernel reads / writes (AttentionKernelType.swift:10-22)
  uint32_t inputs = 0, outputs = 0;
  if (run_mask & MFA_RUN_FORWARD) {
    inputs |= (1u << MFA_Q) | (1u << MFA_K) | (1u << MFA_V);
    outputs |= (1u << MFA_O) | (1u << MFA_L);
  }
  if (run_mask & MFA_RUN_BACKWARD_QUERY) {
    inputs |= (1u << MFA_Q) | (1u << MFA_K) | (1u << MFA_V) | (1u << MFA_dO);
    if (!(run_mask & MFA_RUN_FORWARD)) inputs |= (1u << MFA_O) | (1u << MFA_L);
    outputs |= (1u << MFA_D) | (1u << MFA_dQ);
  }
  if (run_mask & MFA_RUN_BACKWARD_KEY_VALUE) {
    inputs |= (1u << MFA_Q) | (1u << MFA_K) | (1u << MFA_V) | (1u << MFA_dO);
    if (!(run_mask & MFA_RUN_FORWARD)) inputs |= (1u << MFA_L);
    if (!(run_mask & MFA_RUN_BACKWARD_QUERY)) inputs |= (1u << MFA_D);
    outputs |= (1u << MFA_dV) | (1u << MFA_dK);
  }

  mfa_function_constants_t constants;
  int status = mfa_attention_descriptor_set_function_constants(descriptor, &constants);
  if (status != MFA_SUCCESS) return status;
  const uint32_t batch = constants.batch_count ? constants.batch_count : 1;

  void *dev[MFA_BUFFER_COUNT] = {};
  size_t head_bytes[MFA_BUFFER_COUNT] = {};  // bytes of one single-head problem, per operand
  size_t traffic_per_head = 0;
  for (int op = 0; op < MFA_BUFFER_COUNT; ++op) {
    if (!((inputs | outputs) & (1u << op))) continue;
    size_t elements = 0;
    status = mfa_attention_descriptor_operand_elements(descriptor, (mfa_operand_t)op, &elements);
    if (status != MFA_SUCCESS) return status;
    const size_t nbytes = elements * (memory_precision(*descriptor, op) == MFA_FP32 ? 4 : 2);
    head_bytes[op] = nbytes / batch;
    if (s.bytes[op] < nbytes) {
      if (s.ptr[op]) cudaFree(s.ptr[op]);
      s.ptr[op] = nullptr;
      s.bytes[op] = 0;
      if ((e = cudaMalloc(&s.ptr[op], nbytes)) != cudaSuccess)
        return fail(MFA_ERROR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e));
      s.bytes[op] = nbytes;
    }
    dev[op] = s.ptr[op];
    if ((inputs & (1u << op)) && !host_buffers[op])
      return fail(MFA_ERROR_INVALID_ARGUMENT,
                  std::string("Host buffer ") + mfa_operand_name((mfa_operand_t)op) + " is NULL.");
    if ((inputs & (1u << op)) || host_buffers[op]) traffic_per_head += head_bytes[op];
  }

  // reference order: forward -> backwardQuery -> backwardKeyValue (SquareAttentionTest.swift:355-368)
  const mfa_attention_kernel_t *kernels[3] = {};
  for (int type = MFA_FORWARD; type <= MFA_BACKWARD_KEY_VALUE; ++type)
    if (run_mask & (1u << type))
      if ((status = mfa_attention_kernel_cache_fetch(descriptor, (mfa_kernel_type_t)type, &kernels[type])) != MFA_SUCCESS)
        return status;

  const uint32_t per_chunk = chunk_heads(batch, traffic_per_head);
  cudaStream_t upload = s.stream[0], compute = s.stream[1], download = s.stream[2];
  // every exit drains the three streams: the call is synchronous and the scratch is reused by the next one
  auto drained = [&](int result) {
    for (int i = 0; i < kHostStreams; ++i) cudaStreamSynchronize(s.stream[i]);
    return result;
  };
  // per-row statistics (L, D: a few KB per head) are not worth one copy per chunk: they come back in ONE copy after the
  // last chunk (the download stream is then behind every kernel)
  uint32_t small_outputs = 0;
  const char *stats_env = getenv("MFA_B200_HOST_BATCH_STATS");  // tuning knob: 0 = one copy per chunk, as for O
  if (per_chunk < batch && !(stats_env && stats_env[0] == '0'))
    for (int op = 0; op < MFA_BUFFER_COUNT; ++op)
      if ((outputs & (1u << op)) && host_buffers[op] && head_bytes[op] * batch <= (size_t(4) << 20)) small_outputs |= 1u << op;
  uint32_t chunk_index = 0;
  for (uint32_t h0 = 0; h0 < batch; h0 += per_chunk, ++chunk_index) {
    const uint32_t heads = batch - h0 < per_chunk ? batch - h0 : per_chunk;
    void *chunk_dev[MFA_BUFFER_COUNT] = {};
    for (int op = 0; op < MFA_BUFFER_COUNT; ++op) {
      if (!dev[op]) continue;
      chunk_dev[op] = static_cast<char *>(dev[op]) + head_bytes[op] * h0;
      if (inputs & (1u << op)) {
        const char *src = static_cast<const char *>(host_buffers[op]) + head_bytes[op] * h0;
        if ((e = cudaMemcpyAsync(chunk_dev[op], src, head_bytes[op] * heads, cudaMemcpyHostToDevice, upload)) != cudaSuccess)
          return drained(fail(MFA_ERROR_CUDA, std::string("H2D copy: ") + cudaGetErrorString(e)));
      }
    }
    if ((e = cudaEventRecord(s.uploaded[chunk_index], upload)) != cudaSuccess ||
        (e = cudaStreamWaitEvent(compute, s.uploaded[chunk_index], 0)) != cudaSuccess)
      return drained(fail(MFA_ERROR_CUDA, std::string("event: ") + cudaGetErrorString(e)));
    mfa_function_constants_t chunk_constants = constants;
    chunk_constants.batch_count = heads;
    for (int type = MFA_FORWARD; type <= MFA_BACKWARD_KEY_VALUE; ++type)
      if (kernels[type] &&
          (status = mfa_attention_kernel_encode(kernels[type], &chunk_constants, chunk_dev, compute)) != MFA_SUCCESS)
        return drained(status);
    if ((e = cudaEventRecord(s.computed[chunk_index], compute)) != cudaSuccess ||
        (e = cudaStreamWaitEvent(download, s.computed[chunk_index], 0)) != cudaSuccess)
      return drained(fail(MFA_ERROR_CUDA, std::string("event: ") + cudaGetErrorString(e)));
    for (int op = 0; op < MFA_BUFFER_COUNT; ++op) {
      if (!(outputs & (1u << op)) || !host_buffers[op] || (small_outputs & (1u << op))) continue;
      char *dst = static_cast<char *>(host_buffers[op]) + head_bytes[op] * h0;
      if ((e = cudaMemcpyAsync(dst, chunk_dev[op], head_bytes[op] * heads, cudaMemcpyDeviceToHost, download)) != cudaSuccess)
        return drained(fail(MFA_ERROR_CUDA, std::string("D2H copy: ") + cudaGetErrorString(e)));
    }
  }
  for (int op = 0; op < MFA_BUFFER_COUNT; ++op)
    if (small_outputs & (1u << op))
      if ((e = cudaMemcpyAsync(host_buffers[op], dev[op], head_bytes[op] * batch, cudaMemcpyDeviceToHost, download)) != cudaSuccess)
        return drained(fail(MFA_ERROR_CUDA, std::string("D2H copy: ") + cudaGetErrorString(e)));
  // (the device scratch is reused by the next call on this thread: every stream must have drained before returning,
  // which the synchronous contract of this entry point requires anyway)
  for (int i = 0; i < kHostStreams; ++i)
    if ((e = cudaStreamSynchronize(s.stream[i])) != cudaSuccess)
      return fail(MFA_ERROR_CUDA, std::string("kernel execution failed: ") + cudaGetErrorString(e));
  return MFA_SUCCESS;
}

int mfa_release_device_resources(int device) {
  DeviceGuard guard;
  cudaError_t e = guard.enter(device);
  if (e != cudaSuccess) return fail(MFA_ERROR_NO_DEVICE, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  if ((e = cudaDeviceSynchronize()) != cudaSuccess)
    return fail(MFA_ERROR_CUDA, std::string("cudaDeviceSynchronize: ") + cudaGetErrorString(e));
  auto it = g_scratch.find(device);
  if (it != g_scratch.end()) {
    destroy_scratch(it->second);
    g_scratch.erase(it);
  }
  release_workspaces(device);
  return MFA_SUCCESS;
}

}  // extern "C"

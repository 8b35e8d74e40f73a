// Per-device launch state shared by the kernel launchers.  CUDA function attributes (the > 48 KB dynamic shared-memory
// opt-in), the SM count and scratch memory all belong to a device, and one process may drive several
// (mfa_attention_run_host takes an explicit device; encode() runs on whatever device is current), so nothing here is
// cached per process.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace mfa {

constexpr int kMaxDevices = 64;

// cudaGetDevice with the error folded into the return value (-1)
int current_device();

// multiprocessors of `device` (cached per device; 148 on B200)
uint32_t device_sm_count(int device);

// cudaFuncSetAttribute(kernel, MaxDynamicSharedMemorySize, bytes) once per (kernel, device)
cudaError_t ensure_max_dynamic_smem(const void *kernel, uint32_t bytes, int device);

// Library-owned scratch for kernels that split small grids (forward split-KV partials, backward traversal splits): one
// growing allocation per (device, stream), so launches on one stream reuse it in stream order and launches on
// different streams never share it.  `*out` stays valid until the next request for the same (device, stream) that
// needs more room.  The block is cudaMalloc-aligned (256 B), which the tensor map over the forward's split partials needs.
// `slot` separates independent users inside one encode(): 0 = split partials (forward / backward launchers), 1 = the
// head-dimension padding staging of kernel.cpp, which is live across the launcher's own use of slot 0, 2 = the FP16
// copy of a BF16 dO (backward launchers), which is live across their use of slot 0, 3 = the zero-padded staging copies
// of GEMM operands TMA cannot address in place (tcgen05_gemm.cu: leading dimension not a multiple of 8 elements, or a
// base that is not 16-byte aligned).
cudaError_t workspace_for(int device, cudaStream_t stream, size_t bytes, void **out, int slot = 0);

// Frees every workspace of `device` (the device must be idle); used by tests and by mfa_release_device_resources().
void release_workspaces(int device);

}  // namespace mfa

// Host-side TMA tensor-map construction (cuTensorMapEncodeTiled resolved through the runtime's
// driver entry point, so the library needs no link-time dependency on libcuda).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace mfa {

// Row-major [batch][seq][D] matrix of 16-bit elements, tiled as boxes of 64 (D) x box_rows (seq) x 1,
// 128-byte swizzle, out-of-bounds elements read as zero (the analogue of the reference's zero-padded
// async copies, GEMMHeaders.swift:111-114).
cudaError_t make_tensor_map_16bit(CUtensorMap *map, const void *base, uint32_t seq, uint32_t D, uint32_t batch,
                                  uint32_t box_rows);

// The same operand stored transposed, [batch][D][seq] (leading dimension = seq; AttentionKernel.swift:189-195): boxes of
// 64 (seq) x box_d_rows (D) x 1.  Needs seq % 8 == 0 (16-byte row pitch).
cudaError_t make_tensor_map_16bit_transposed(CUtensorMap *map, const void *base, uint32_t seq, uint32_t D, uint32_t batch,
                                             uint32_t box_d_rows);

// Row-major [batch][seq][D] matrix of FP32 elements, boxes of 32 (D) x box_rows x 1, 128-byte swizzle.
cudaError_t make_tensor_map_f32(CUtensorMap *map, const void *base, uint32_t seq, uint32_t D, uint32_t batch,
                                uint32_t box_rows);

// A [batch][rows][cols] matrix of 16-bit elements whose rows are `row_pitch` elements apart and whose problems are
// `batch_stride` elements apart (a GEMM operand with a leading dimension larger than its width), tiled as boxes of
// box_cols x box_rows x 1 with 128-byte swizzle; elements beyond `cols` or `rows` read as zero.  The pitch and the
// stride must be multiples of 8 elements and the base 16-byte aligned.
cudaError_t make_tensor_map_16bit_strided(CUtensorMap *map, const void *base, uint32_t rows, uint32_t cols,
                                          uint32_t batch, uint64_t row_pitch, uint64_t batch_stride, uint32_t box_cols,
                                          uint32_t box_rows);

void set_launch_detail(const char *fmt, ...);

}  // namespace mfa

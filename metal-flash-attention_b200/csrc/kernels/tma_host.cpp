#include "tma_host.h"

#include <cstdarg>
#include <cstdio>
#include <mutex>
#include <string>

#include "attention_params.h"

namespace mfa {

static thread_local std::string g_detail;

void set_launch_detail(const char *fmt, ...) {
  char buf[512];
  va_list args;
  va_start(args, fmt);
  vsnprintf(buf, sizeof(buf), fmt, args);
  va_end(args);
  g_detail = buf;
}

const char *last_launch_detail() { return g_detail.c_str(); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn resolve_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void *ptr = nullptr;
    cudaDriverEntryPointQueryResult query;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &query);
    if (e == cudaSuccess && query == cudaDriverEntryPointSuccess) fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

// A tensor map is a pure function of (base, shape, box, type): callers that re-encode the same buffers (a training
// loop, the benchmark's back-to-back dispatches) get the 128-byte descriptor from a small per-thread table instead of
// a cuTensorMapEncodeTiled driver call (~1.5 us each, three or four per launch, against kernels of 15-25 us for one
// head).  The descriptor says nothing about buffer *contents*, so a hit can never be stale.
namespace {
struct MapKey {
  const void *base;
  uint32_t seq, D, batch, boxCols, boxRows, dtype;
  uint64_t rowPitch, batchStride;  // bytes
  bool operator==(const MapKey &o) const {
    return base == o.base && seq == o.seq && D == o.D && batch == o.batch && boxCols == o.boxCols &&
           boxRows == o.boxRows && dtype == o.dtype && rowPitch == o.rowPitch && batchStride == o.batchStride;
  }
};
struct MapEntry {
  MapKey key;
  CUtensorMap map;
  bool valid = false;
};
constexpr uint32_t kMapCacheEntries = 32;  // direct-mapped
thread_local MapEntry g_map_cache[kMapCacheEntries];
uint32_t map_slot(const MapKey &k) {
  uint64_t h = reinterpret_cast<uintptr_t>(k.base) * 0x9E3779B97F4A7C15ull;
  h ^= (static_cast<uint64_t>(k.seq) << 32 | k.D) * 0xC2B2AE3D27D4EB4Full;
  h ^= (static_cast<uint64_t>(k.batch) << 32 | (k.boxRows << 8) | k.dtype) * 0x165667B19E3779F9ull;
  h ^= (k.rowPitch ^ (k.batchStride << 20)) * 0x27D4EB2F165667C5ull;
  return static_cast<uint32_t>(h >> 40) % kMapCacheEntries;
}
}  // namespace

// [batch][seq][D] with rows rowPitch bytes apart and problems batchStride bytes apart, boxes of boxCols x boxRows x 1
static cudaError_t encode_strided(CUtensorMap *map, CUtensorMapDataType dtype, uint32_t elemBytes, const void *base,
                                  uint32_t seq, uint32_t D, uint32_t batch, uint64_t rowPitch, uint64_t batchStride,
                                  uint32_t boxCols, uint32_t boxRows) {
  const MapKey key{base, seq, D, batch, boxCols, boxRows, static_cast<uint32_t>(dtype), rowPitch, batchStride};
  MapEntry &entry = g_map_cache[map_slot(key)];
  if (entry.valid && entry.key == key) {
    *map = entry.map;
    return cudaSuccess;
  }
  EncodeTiledFn fn = resolve_encode();
  if (!fn) {
    set_launch_detail("cuTensorMapEncodeTiled is not available from this driver");
    return cudaErrorNotSupported;
  }
  if (reinterpret_cast<uintptr_t>(base) % 16 != 0 || rowPitch % 16 != 0 || batchStride % 16 != 0) {
    set_launch_detail("TMA needs 16-byte aligned buffers and row pitch (base=%p, D=%u, pitch=%llu B)", base, D,
                      (unsigned long long)rowPitch);
    return cudaErrorInvalidValue;
  }
  cuuint64_t dims[3] = {D, seq, batch};
  cuuint64_t strides[2] = {rowPitch, batchStride};
  cuuint32_t box[3] = {boxCols, boxRows, 1};
  cuuint32_t elemStrides[3] = {1, 1, 1};
  CUresult r = fn(map, dtype, 3, const_cast<void *>(base), dims, strides, box, elemStrides, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_launch_detail("cuTensorMapEncodeTiled failed with CUresult %d (seq=%u D=%u batch=%u box=%ux%u)", (int)r, seq, D,
                      batch, boxCols, boxRows);
    return cudaErrorInvalidValue;
  }
  entry.key = key;
  entry.map = *map;
  entry.valid = true;
  return cudaSuccess;
}

// contiguous rows of D elements and contiguous problems: what every attention operand is
static cudaError_t encode(CUtensorMap *map, CUtensorMapDataType dtype, uint32_t elemBytes, const void *base,
                          uint32_t seq, uint32_t D, uint32_t batch, uint32_t boxCols, uint32_t boxRows) {
  const uint64_t pitch = static_cast<uint64_t>(D) * elemBytes;
  return encode_strided(map, dtype, elemBytes, base, seq, D, batch, pitch, pitch * seq, boxCols, boxRows);
}

cudaError_t make_tensor_map_16bit(CUtensorMap *map, const void *base, uint32_t seq, uint32_t D, uint32_t batch,
                                  uint32_t box_rows) {
  // BF16 and FP16 move identically through TMA; the 16-bit "type" only matters for OOB fill (zeros).
  return encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, seq, D, batch, 64, box_rows);
}

// Transposed operand: [batch][D][seq] (leading dimension = seq), tiled as boxes of 64 (seq) x box_d_rows (D) x 1.
cudaError_t make_tensor_map_16bit_transposed(CUtensorMap *map, const void *base, uint32_t seq, uint32_t D, uint32_t batch,
                                             uint32_t box_d_rows) {
  // same encoder with the roles of the two inner dimensions swapped: inner extent = seq, rows = D
  return encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, D, seq, batch, 64, box_d_rows);
}

cudaError_t make_tensor_map_f32(CUtensorMap *map, const void *base, uint32_t seq, uint32_t D, uint32_t batch,
                                uint32_t box_rows) {
  return encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, seq, D, batch, 32, box_rows);
}

cudaError_t make_tensor_map_16bit_strided(CUtensorMap *map, const void *base, uint32_t rows, uint32_t cols,
                                          uint32_t batch, uint64_t row_pitch, uint64_t batch_stride, uint32_t box_cols,
                                          uint32_t box_rows) {
  return encode_strided(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, rows, cols, batch, row_pitch * 2,
                        batch_stride * 2, box_cols, box_rows);
}

}  // namespace mfa

#include "device_state.h"

#include <map>
#include <mutex>
#include <utility>
#include <vector>

#include "tma_host.h"

namespace mfa {

int current_device() {
  int device = -1;
  if (cudaGetDevice(&device) != cudaSuccess) {
    cudaGetLastError();
    return -1;
  }
  return device;
}

uint32_t device_sm_count(int device) {
  static std::mutex mutex;
  static int cached[kMaxDevices] = {};
  if (device < 0) return 148;
  std::lock_guard<std::mutex> lock(mutex);
  if (device < kMaxDevices && cached[device] > 0) return static_cast<uint32_t>(cached[device]);
  int count = 0;
  if (cudaDeviceGetAttribute(&count, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || count <= 0) {
    cudaGetLastError();
    return 148;
  }
  if (device < kMaxDevices) cached[device] = count;
  return static_cast<uint32_t>(count);
}

cudaError_t ensure_max_dynamic_smem(const void *kernel, uint32_t bytes, int device) {
  static std::mutex mutex;
  static std::map<std::pair<const void *, int>, uint32_t> done;  // (kernel, device) -> bytes already opted in
  std::lock_guard<std::mutex> lock(mutex);
  auto key = std::make_pair(kernel, device);
  auto it = done.find(key);
  if (it != done.end() && it->second >= bytes) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
  if (e != cudaSuccess) {
    set_launch_detail("cudaFuncSetAttribute(MaxDynamicSharedMemorySize = %u) failed on device %d", bytes, device);
    return e;
  }
  done[key] = bytes;
  return cudaSuccess;
}

namespace {
struct Workspace {
  void *ptr = nullptr;
  size_t bytes = 0;
};
std::mutex g_workspace_mutex;
std::map<std::pair<std::pair<int, int>, cudaStream_t>, Workspace> g_workspaces;  // ((device, slot), stream)
}  // namespace

cudaError_t workspace_for(int device, cudaStream_t stream, size_t bytes, void **out, int slot) {
  std::lock_guard<std::mutex> lock(g_workspace_mutex);
  Workspace &w = g_workspaces[std::make_pair(std::make_pair(device, slot), stream)];
  if (w.bytes < bytes) {
    // growing means allocating: not possible while the stream is being captured into a graph (warm the kernel up once
    // before capturing, as every graph user does)
    cudaStreamCaptureStatus capture = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &capture) == cudaSuccess && capture != cudaStreamCaptureStatusNone) {
      set_launch_detail("the split-grid workspace (%zu bytes) must be allocated before stream capture: run the kernel "
                        "once outside the capture first", bytes);
      return cudaErrorStreamCaptureUnsupported;
    }
    if (w.ptr) {
      // the old block may still be in use by work queued on this stream
      cudaError_t e = cudaStreamSynchronize(stream);
      if (e != cudaSuccess) return e;
      cudaFree(w.ptr);
      w.ptr = nullptr;
      w.bytes = 0;
    }
    size_t rounded = (bytes + (size_t(1) << 20) - 1) & ~((size_t(1) << 20) - 1);
    cudaError_t e = cudaMalloc(&w.ptr, rounded);
    if (e != cudaSuccess) {
      set_launch_detail("cudaMalloc of the %zu-byte split-grid workspace failed", rounded);
      return e;
    }
    w.bytes = rounded;
  }
  *out = w.ptr;
  return cudaSuccess;
}

void release_workspaces(int device) {
  std::lock_guard<std::mutex> lock(g_workspace_mutex);
  for (auto it = g_workspaces.begin(); it != g_workspaces.end();) {
    if (it->first.first.first == device) {
      if (it->second.ptr) cudaFree(it->second.ptr);
      it = g_workspaces.erase(it);
    } else {
      ++it;
    }
  }
}

}  // namespace mfa

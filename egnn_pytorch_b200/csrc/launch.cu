// Process-wide launch state (launch.cuh): the dynamic shared-memory opt-ins and the SM counts, per device.
#include <map>
#include <mutex>
#include <utility>
#include "launch.cuh"

namespace egnn {
namespace {
std::mutex mu;
std::map<std::pair<int, const void*>, size_t> smem_opted;     // (device, kernel) -> bytes opted in
std::map<int, int> sm_counts;                                   // device -> multiprocessors
}  // namespace

int opt_in_dynamic_smem(const void* kernel, size_t smem) {
  int dev = 0;
  EGNN_CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = smem_opted[{dev, kernel}];
  if (have < smem) {
    EGNN_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    have = smem;
  }
  return EGNN_OK;
}

int device_sm_count(int* out) {
  int dev = 0;
  EGNN_CUDA_TRY(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  int& n = sm_counts[dev];
  if (n == 0) EGNN_CUDA_TRY(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  *out = n;
  return EGNN_OK;
}

}  // namespace egnn

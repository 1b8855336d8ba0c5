// The one way the library launches a kernel: opt the kernel in to the dynamic shared memory it asks for, launch it,
// check the launch without synchronising and count it (profile.h).  The process-wide state lives in launch.cu.
#pragma once
#include <utility>
#include "common.cuh"
#include "profile.h"

namespace egnn {

// Largest dynamic shared memory a SIMT kernel may use.  The backward preflight (backward_supported) checks its kernels'
// sizes against the same constant, so a configuration it accepts cannot fail at launch time.
constexpr size_t DYN_SMEM_MAX = 220 * 1024;
// Largest dynamic shared memory of one block on sm_100a: the limit of the tensor-core kernels.
constexpr size_t TC_SMEM_MAX = 227 * 1024;

// Raises the dynamic shared-memory limit of `kernel` on the current device to at least `smem` bytes.  One cache keyed on
// (device, kernel) under a mutex; the limit is never lowered.
int opt_in_dynamic_smem(const void* kernel, size_t smem);

// Multiprocessor count of the current device, read once per device.
int device_sm_count(int* out);

// Launches `kernel` on `st`; EGNN_ERR_UNSUPPORTED without launching when it needs more than `smem_max` bytes.
template <typename... P, typename... A>
int launch_upto(size_t smem_max, void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args) {
  if (smem > smem_max) return EGNN_ERR_UNSUPPORTED;
  if (smem > 48 * 1024) EGNN_TRY(opt_in_dynamic_smem(reinterpret_cast<const void*>(kernel), smem));
  kernel<<<grid, block, smem, st>>>(std::forward<A>(args)...);
  EGNN_CUDA_TRY(cudaPeekAtLastError());             // catches a bad configuration at enqueue time, without synchronising
  count_launch();
  return EGNN_OK;
}

template <typename... P, typename... A>
int launch(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A&&... args) {
  return launch_upto(DYN_SMEM_MAX, kernel, grid, block, smem, st, std::forward<A>(args)...);
}

}  // namespace egnn

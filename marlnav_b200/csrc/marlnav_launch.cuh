// marlnav_b200/csrc/marlnav_launch.cuh
//
// Host-side launch set-up shared by the library's units: marlnav_rollout.cu and the
// step library (marlnav_abi.cu, marlnav_step_*.cu, marlnav_step_launch.cuh).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <atomic>

namespace mnl {

inline int current_device() { int d = 0; cudaGetDevice(&d); return d; }

// Set kKernel's function attributes on the current device before a launch: the dynamic shared
// memory limit to `smem` bytes (unless 0) and, with `carveout`, the preferred carveout to the
// largest shared-memory share -- the same carveout for every kernel, so SMs need not drain and
// reconfigure between them.  Attributes are per device and are set again only when a launch
// needs a larger limit.  Setting them is idempotent, so two threads racing here at worst both
// set them (the record itself is atomic).
template <auto kKernel>
cudaError_t set_attributes_once(size_t smem, bool carveout) {
    static std::atomic<size_t> configured[64];      // per device: 0, or 1 + the limit set
    std::atomic<size_t>& done = configured[current_device() & 63];
    if (smem < done.load(std::memory_order_acquire)) return cudaSuccess;
    cudaError_t e = cudaSuccess;
    if (smem > 0) e = cudaFuncSetAttribute(kKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess && carveout)
        e = cudaFuncSetAttribute(kKernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    if (e == cudaSuccess) done.store(smem + 1, std::memory_order_release);
    return e;
}

}  // namespace mnl

// Small host-side helpers shared by the launch wrappers.
#pragma once
#include <atomic>
#include <cuda_runtime.h>

namespace b2p {

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device (per-context) attribute: remember, per device, the
// largest value a kernel was opted into.  Lock-free; a racing second caller at worst repeats the (idempotent) call.
// Any non-zero size is opted into: a kernel's STATIC shared memory counts against the same 48 KB default, so a dynamic
// size below 48 KB can still need the attribute (peaks_kernel: 4.2 KB static + 45 KB dynamic for a 70 x 138 map).
struct DynSmemOptIn {
    static constexpr int kMaxDevices = 64;
    std::atomic<size_t> set[kMaxDevices];
    DynSmemOptIn() { for (auto& s : set) s.store(0); }
    template <class Kernel>
    cudaError_t ensure(Kernel kernel, size_t bytes) {
        if (bytes == 0) return cudaSuccess;
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        if (dev < 0 || dev >= kMaxDevices) return cudaErrorInvalidDevice;
        if (set[dev].load(std::memory_order_acquire) >= bytes) return cudaSuccess;
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return e;
        size_t cur = set[dev].load();
        while (cur < bytes && !set[dev].compare_exchange_weak(cur, bytes)) {}
        return cudaSuccess;
    }
};

}  // namespace b2p

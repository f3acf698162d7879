// tmpc_devptr.h -- validation of the device pointers the device-resident entries take, before anything is queued.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace tmpc {

// p is 16-byte aligned device or managed memory of `device`.  A host pointer passed by mistake (pageable or pinned) or memory of
// another device is refused here instead of faulting the kernel that would dereference it.
inline bool device_ptr_on(const void* p, int device) {
    if (reinterpret_cast<uintptr_t>(p) & 15u) return false;
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) && a.device == device;
}

}  // namespace tmpc

// host_guard.h -- host-side helpers of the C ABI: run a call on the device that owns its stream / buffers, and
// launch a kernel, optionally as a programmatic dependent of the previous kernel in the stream.
//
// The ABI promises "safe to call on any device": a launch on a stream of device B while device A is current
// fails with an invalid resource handle, so every entry point that enqueues work switches to the owning
// device for the duration of the call and restores the caller's current device afterwards.
//   * a non-default stream names its device (cudaStreamGetDevice);
//   * the default / per-thread stream handles (0, 1, 2) do not: the device is then the one that owns `ptr`
//     (cudaPointerGetAttributes), or the current one when `ptr` is not device memory.
#pragma once
#include <cuda_runtime.h>
#include <utility>

namespace dd {

inline cudaError_t owning_device(cudaStream_t st, const void* ptr, int* dev)
{
    if (st != nullptr && st != cudaStreamLegacy && st != cudaStreamPerThread) return cudaStreamGetDevice(st, dev);
    if (ptr) {
        cudaPointerAttributes at;
        const cudaError_t e = cudaPointerGetAttributes(&at, ptr);
        if (e == cudaSuccess && (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged)) { *dev = at.device; return cudaSuccess; }
        if (e != cudaSuccess) (void)cudaGetLastError();          // unknown pointer kinds are not an error here
    }
    return cudaGetDevice(dev);
}

struct DeviceGuard {
    int prev = -1, dev = -1;
    bool switched = false;
    cudaError_t err = cudaSuccess;
    explicit DeviceGuard(int device) { enter(device); }
    DeviceGuard(cudaStream_t st, const void* ptr)
    {
        int d = -1;
        err = owning_device(st, ptr, &d);
        if (err == cudaSuccess) enter(d);
    }
    ~DeviceGuard() { if (switched) (void)cudaSetDevice(prev); }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;

private:
    void enter(int device)
    {
        dev = device;
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) { err = cudaSetDevice(device); switched = err == cudaSuccess; }
    }
};

// One launch, optionally as a programmatic dependent of the previous kernel in the stream (the kernel then calls
// pdl_wait() before it reads what that kernel wrote, drone_device.cuh).
template <typename... KP, typename... AP>
inline int launch(void (*kern)(KP...), int grid, int block, cudaStream_t st, bool pdl, AP&&... args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = 0; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    return (int)cudaLaunchKernelEx(&cfg, kern, std::forward<AP>(args)...);
}

}  // namespace dd

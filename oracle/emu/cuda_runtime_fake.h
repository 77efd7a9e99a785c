// cuda_runtime_fake.h -- TEST INFRASTRUCTURE.  The CUDA runtime calls that ddc_api.cu makes, on the host:
// device memory is malloc'ed memory, copies are memcpy, streams and events do nothing because every kernel
// "launch" (cuda_emu::launch, see make_api_emu.py for how <<< >>> gets there) runs to completion before it
// returns.  With this header and ddc_host_emu.h the product's own C-ABI implementation compiles into
// oracle/libddc_cuda_emu.so, so that its HOST logic -- the assumed plan and the re-run on a mismatch, the
// capacity re-run of the neighbour fill pass, DDC_ASYNC, the getters, the error paths -- is exercised by
// the CPU suite (one rank; several ranks are emulated by emu_pipeline.cpp).  One device, no NCCL, no IPC.
#pragma once
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "cuda_emu.h"

typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorMemoryAllocation = 2, cudaErrorNotSupported = 801 };
typedef struct ddc_fake_stream* cudaStream_t;
typedef struct ddc_fake_event* cudaEvent_t;
struct cudaIpcMemHandle_t {
    char reserved[64];
};
enum cudaMemcpyKind { cudaMemcpyHostToHost = 0, cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaMemcpyDeviceToDevice = 3 };
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2, cudaHostAllocMapped = 2, cudaHostAllocPortable = 1, cudaHostAllocDefault = 0, cudaIpcMemLazyEnablePeerAccess = 1 };
enum cudaDeviceAttr { cudaDevAttrMultiProcessorCount = 16, cudaDevAttrMaxSharedMemoryPerBlockOptin = 97 };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };

struct dim3 {
    unsigned x, y, z;
    dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1)
        : x(x_)
        , y(y_)
        , z(z_)
    {
    }
};

inline const char* cudaGetErrorString(cudaError_t e) { return e == cudaSuccess ? "no error" : "emulated CUDA error"; }
inline cudaError_t cudaGetLastError() { return cudaSuccess; }
inline cudaError_t cudaGetDeviceCount(int* n)
{
    *n = 1;
    return cudaSuccess;
}
inline cudaError_t cudaSetDevice(int) { return cudaSuccess; }
inline cudaError_t cudaGetDevice(int* d)
{
    *d = 0;
    return cudaSuccess;
}
inline cudaError_t cudaDeviceGetAttribute(int* v, cudaDeviceAttr a, int)
{
    *v = a == cudaDevAttrMultiProcessorCount ? 148 : 232448; // B200: 148 SMs, 227 KB of shared memory per block
    return cudaSuccess;
}
inline cudaError_t cudaDeviceGetStreamPriorityRange(int* least, int* greatest)
{
    *least = 0;
    *greatest = -5;
    return cudaSuccess;
}
template <typename T>
inline cudaError_t cudaMalloc(T** p, size_t n)
{
    *p = static_cast<T*>(std::malloc(n ? n : 1));
    return *p ? cudaSuccess : cudaErrorMemoryAllocation;
}
inline cudaError_t cudaFree(void* p)
{
    std::free(p);
    return cudaSuccess;
}
template <typename T>
inline cudaError_t cudaHostAlloc(T** p, size_t n, unsigned)
{
    *p = static_cast<T*>(std::malloc(n ? n : 1));
    return *p ? cudaSuccess : cudaErrorMemoryAllocation;
}
template <typename T, typename U>
inline cudaError_t cudaHostGetDevicePointer(T** dev, U* host, unsigned)
{
    *dev = reinterpret_cast<T*>(host);
    return cudaSuccess;
}
inline cudaError_t cudaFreeHost(void* p)
{
    std::free(p);
    return cudaSuccess;
}
inline cudaError_t cudaMemcpyAsync(void* dst, const void* src, size_t n, cudaMemcpyKind, cudaStream_t)
{
    std::memcpy(dst, src, n);
    return cudaSuccess;
}
inline cudaError_t cudaMemset(void* p, int v, size_t n)
{
    std::memset(p, v, n);
    return cudaSuccess;
}
inline cudaError_t cudaMemsetAsync(void* p, int v, size_t n, cudaStream_t) { return cudaMemset(p, v, n); }
inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned)
{
    *s = reinterpret_cast<cudaStream_t>(std::malloc(1));
    return cudaSuccess;
}
inline cudaError_t cudaStreamCreateWithPriority(cudaStream_t* s, unsigned f, int) { return cudaStreamCreateWithFlags(s, f); }
inline cudaError_t cudaStreamDestroy(cudaStream_t s)
{
    std::free(s);
    return cudaSuccess;
}
inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
inline cudaError_t cudaEventCreate(cudaEvent_t* e)
{
    *e = reinterpret_cast<cudaEvent_t>(std::malloc(1));
    return cudaSuccess;
}
inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { return cudaEventCreate(e); }
inline cudaError_t cudaEventDestroy(cudaEvent_t e)
{
    std::free(e);
    return cudaSuccess;
}
inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return cudaSuccess; }
inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t)
{
    *ms = 0.0f;
    return cudaSuccess;
}
template <typename K>
inline cudaError_t cudaFuncSetAttribute(K, cudaFuncAttribute, int) { return cudaSuccess; }
struct cudaFuncAttributes {
    size_t sharedSizeBytes;
};
template <typename K>
inline cudaError_t cudaFuncGetAttributes(cudaFuncAttributes* a, K)
{
    a->sharedSizeBytes = 1400; // about what the cut kernels hold statically
    return cudaSuccess;
}
template <typename K>
inline cudaError_t cudaOccupancyMaxActiveBlocksPerMultiprocessor(int* n, K, int, size_t)
{
    *n = 4;
    return cudaSuccess;
}
inline cudaError_t cudaDeviceCanAccessPeer(int* can, int, int)
{
    *can = 0;
    return cudaSuccess;
}
enum { cudaErrorPeerAccessAlreadyEnabled = 704 };
inline cudaError_t cudaDeviceEnablePeerAccess(int, unsigned) { return cudaErrorNotSupported; }
// peer memory between processes does not exist here
inline cudaError_t cudaIpcGetMemHandle(cudaIpcMemHandle_t*, void*) { return cudaErrorNotSupported; }
inline cudaError_t cudaIpcOpenMemHandle(void**, cudaIpcMemHandle_t, unsigned) { return cudaErrorNotSupported; }
inline cudaError_t cudaIpcCloseMemHandle(void*) { return cudaErrorNotSupported; }

// launch_k() of ddc_api.cu runs the kernel through DDC_EMU_LAUNCH(grid, block, smem, kernel(args)) in these builds
#define DDC_EMU_LAUNCH(grid, block, smem, ...)                                                     \
    do {                                                                                           \
        const dim3 g_ = dim3(grid), b_ = dim3(block);                                               \
        if (!cuda_emu::launch(cuda_emu::Dim3(g_.x, g_.y, g_.z), cuda_emu::Dim3(b_.x, b_.y, b_.z), (size_t)(smem),    \
                [&] { __VA_ARGS__; })) {                                                            \
            std::fprintf(stderr, "ddc emulation: %s: %s\n", #__VA_ARGS__, cuda_emu::last_error());  \
            std::abort();                                                                          \
        }                                                                                          \
    } while (0)

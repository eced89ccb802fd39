// cuda_util.h -- host-side plumbing both engines of the library share (pmm_engine.cu, sw_engine.cu): the grow-only
// device / pinned buffer and the device check of their create functions.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstddef>
#include <string>

// Grow-only buffer, freed with its owner.  Buffers are recycled across jobs like the reference's scratch blocks
// (PairHMMTask.cpp:19-25,48,70); a reserve that grows adds a quarter of slack.
template <bool Pinned>
struct GrowBuf {
    void* p = nullptr;
    size_t cap = 0;

    GrowBuf() = default;
    GrowBuf(const GrowBuf&) = delete;
    GrowBuf& operator=(const GrowBuf&) = delete;
    ~GrowBuf() { release(); }

    cudaError_t reserve(size_t n)
    {
        if (n <= cap) return cudaSuccess;
        release();
        size_t want = std::max(n, (size_t)4096);
        want += want / 4;
        cudaError_t e = Pinned ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want; else p = nullptr;
        return e;
    }
    void release()
    {
        if (p) { if (Pinned) cudaFreeHost(p); else cudaFree(p); }
        p = nullptr; cap = 0;
    }
};
using DevBuf = GrowBuf<false>;
using PinBuf = GrowBuf<true>;

// Makes `device` (< 0: the current one) current after checking that it exists and is an sm_100 part, and returns its SM
// count.  Returns 0 or the caller's error code, with the reason in err; `engine` names the caller in the message.
template <int kInvalid, int kCuda, int kNoDevice>
int open_device(int& device, int& sm_count, std::string& err, const char* engine)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        err = std::string("no CUDA device visible; ") + engine + " has no CPU fallback";
        return kNoDevice;
    }
    if (device < 0 && cudaGetDevice(&device) != cudaSuccess) device = 0;
    if (device >= n) { err = "device index out of range"; return kInvalid; }
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        err = cudaGetErrorString(e);
        return kCuda;
    }
    if (prop.major != 10) { err = std::string("kernels are built for sm_100a only; device is ") + prop.name; return kNoDevice; }
    sm_count = prop.multiProcessorCount;
    return 0;
}

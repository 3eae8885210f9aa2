// trpl_host.cuh -- host-side pieces shared by the C-ABI files (trpl_kernels.cu, trpl_nccl.cu): error
// capture, the device-entry pattern, the grid rule of the small kernels and stream-ordered scratch.
// Each including file gets its own copy (anonymous namespace), so each library keeps its own error text.
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>

#include "trpl_b200.h"

namespace {

thread_local char g_cuda_err[256] = "";

int cuda_fail(cudaError_t e, const char *what)
{
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
    return TRPL_ECUDA;
}
#define CK(call)                                                   \
    do {                                                           \
        cudaError_t e_ = (call);                                   \
        if (e_ != cudaSuccess) return cuda_fail(e_, #call);        \
    } while (0)
// propagates a TRPL_E* code of a host helper
#define TRY(call)                                                  \
    do {                                                           \
        if (int rc_ = (call)) return rc_;                          \
    } while (0)

// stream-ordered device scratch, released on every exit path
struct Scratch {
    void *p = nullptr;
    cudaStream_t st;
    explicit Scratch(cudaStream_t s) : st(s) {}
    cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes, st); }
    ~Scratch() { if (p) cudaFreeAsync(p, st); }
    Scratch(const Scratch &) = delete;
    Scratch &operator=(const Scratch &) = delete;
};

// Grid of a grid-stride kernel over `work` items with `tb` threads per block: one item per thread, at most
// `per_sm` blocks per SM of `device`.  The reductions accumulate one partial sum per block, so their grouping
// (and last bits) follow this grid.
int stride_grid(int device, long long work, int tb, int per_sm, unsigned *grid)
{
    int nsm = 0;
    CK(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device));
    const long long want = (work + tb - 1) / tb, cap = (long long)nsm * per_sm;
    *grid = (unsigned)(want < cap ? want : cap);
    return TRPL_OK;
}

// Makes `device` current for the duration of one C-ABI call and restores the caller's device on every
// exit path (torch reads its current device from the runtime; a library must not change it).
struct DeviceGuard {
    int prev = -1;
    bool switched = false;
    int enter(int device)
    {
        int n = 0;
        if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
            cudaGetLastError();
            return TRPL_ENODEVICE;
        }
        CK(cudaGetDevice(&prev));
        if (prev != device) {
            CK(cudaSetDevice(device));
            switched = true;
        }
        return TRPL_OK;
    }
    ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};

// Runs `work` (returning a TRPL_* code) with `device` current, or returns why the device cannot be entered.
// Entry points validate their arguments before this and call it once, so every one has the same shape.
template <class F>
int on_device(int device, F &&work)
{
    DeviceGuard guard;
    TRY(guard.enter(device));
    return work();
}

}  // namespace

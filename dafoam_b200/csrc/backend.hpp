// Execution backend.  The product build (nvcc, sm_100a) launches every functor as a CUDA kernel on the
// solver's stream.  Defining DAB_HOSTSIM compiles the very same functors into plain host loops: that
// build exists ONLY so that the non-GPU test suite can check the hand-derived kernels against the
// oracle on a machine without a GPU (tests/hostsim); it is never loaded by the product package.
#pragma once
#include "foam_io.hpp"
#include "views.hpp"
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <vector>

#ifndef DAB_HOSTSIM
#include <cuda_runtime.h>
#endif

namespace dab
{

#ifndef DAB_HOSTSIM
#define DAB_CUDA_CHECK(x)                                                                              \
    do                                                                                                 \
    {                                                                                                  \
        cudaError_t e_ = (x);                                                                          \
        if (e_ != cudaSuccess) throw ::dab::Error(std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #x); \
    } while (0)

// per-functor occupancy hint: minimum resident blocks per SM (registers are capped accordingly)
#ifndef DAB_BLOCK
#define DAB_BLOCK 128
#endif
#ifndef DAB_MINBLOCKS
#define DAB_MINBLOCKS 6
#endif
template <class F>
struct LaunchTraits
{
    static constexpr int minBlocks = DAB_MINBLOCKS; // <= 80 registers per thread unless a functor says otherwise (latency-bound gathers: occupancy wins)
};

template <class F>
__global__ void __launch_bounds__(DAB_BLOCK, LaunchTraits<F>::minBlocks) kernel1d(int n, F f)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) f(i);
}

struct Backend
{
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr; // communication stream (halo exchange overlapped with interior cells)
    long launches = 0;
    int device_ = 0;
    void makeCurrent() { if (stream) cudaSetDevice(device_); }
    void init(int device)
    {
        device_ = device;
        int n = 0;
        cudaError_t e = cudaGetDeviceCount(&n);
        if (e != cudaSuccess || n == 0)
            throw Error("dab200 requires a CUDA device (sm_100a); none is visible and there is no CPU fallback");
        DAB_CUDA_CHECK(cudaSetDevice(device));
        DAB_CUDA_CHECK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        DAB_CUDA_CHECK(cudaStreamCreateWithFlags(&stream2, cudaStreamNonBlocking));
    }
    void destroy()
    {
        if (stream) cudaStreamDestroy(stream);
        if (stream2) cudaStreamDestroy(stream2);
        stream = nullptr;
        stream2 = nullptr;
    }
    void* alloc(size_t bytes)
    {
        void* p = nullptr;
        DAB_CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 8));
        return p;
    }
    void free(void* p) { cudaFree(p); }
    void h2d(void* d, const void* h, size_t b) { DAB_CUDA_CHECK(cudaMemcpyAsync(d, h, b, cudaMemcpyHostToDevice, stream)); DAB_CUDA_CHECK(cudaStreamSynchronize(stream)); }
    void d2h(void* h, const void* d, size_t b) { DAB_CUDA_CHECK(cudaMemcpyAsync(h, d, b, cudaMemcpyDeviceToHost, stream)); DAB_CUDA_CHECK(cudaStreamSynchronize(stream)); }
    void d2d(void* d, const void* s, size_t b) { DAB_CUDA_CHECK(cudaMemcpyAsync(d, s, b, cudaMemcpyDeviceToDevice, stream)); }
    void zero(void* d, size_t b) { DAB_CUDA_CHECK(cudaMemsetAsync(d, 0, b, stream)); }
    void sync() { DAB_CUDA_CHECK(cudaStreamSynchronize(stream)); }
    template <class F>
    void launch(int n, const F& f)
    {
        if (n <= 0) return;
        const int bs = DAB_BLOCK;
        kernel1d<F><<<(n + bs - 1) / bs, bs, 0, stream>>>(n, f);
        DAB_CUDA_CHECK(cudaGetLastError()); // a launch-configuration failure is not sticky: catch it here, not as wrong numbers later
        launches++;
    }
    // CUDA-event timer on the solver's stream
    struct Timer
    {
        cudaEvent_t a, b;
        cudaStream_t st;
        explicit Timer(cudaStream_t s) : st(s) { cudaEventCreate(&a); cudaEventCreate(&b); }
        ~Timer() { cudaEventDestroy(a); cudaEventDestroy(b); }
        void start() { cudaEventRecord(a, st); }
        double stopMs()
        {
            cudaEventRecord(b, st);
            cudaEventSynchronize(b);
            float ms = 0.f;
            cudaEventElapsedTime(&ms, a, b);
            return (double)ms;
        }
    };
    Timer timer() { return Timer(stream); }
};
#else
struct Backend
{
    long launches = 0;
    void makeCurrent() {}
    void init(int) {}
    void destroy() {}
    void* alloc(size_t bytes) { return std::malloc(bytes ? bytes : 8); }
    void free(void* p) { std::free(p); }
    void h2d(void* d, const void* h, size_t b) { std::memcpy(d, h, b); }
    void d2h(void* h, const void* d, size_t b) { std::memcpy(h, d, b); }
    void d2d(void* d, const void* s, size_t b) { std::memcpy(d, s, b); }
    void zero(void* d, size_t b) { std::memset(d, 0, b); }
    void sync() {}
    template <class F>
    void launch(int n, const F& f)
    {
        for (int i = 0; i < n; i++) f(i);
        launches++;
    }
    struct Timer
    {
        std::chrono::steady_clock::time_point t0;
        void start() { t0 = std::chrono::steady_clock::now(); }
        double stopMs() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); }
    };
    Timer timer() { return Timer(); }
};
#endif

// run a functor on the index range [c0, c0 + n)
template <class F>
struct Shifted
{
    F f;
    int c0;
    DAB_HD void operator()(int i) const { f(i + c0); }
};
#ifndef DAB_HOSTSIM
template <class F>
struct LaunchTraits<Shifted<F>>
{
    static constexpr int minBlocks = LaunchTraits<F>::minBlocks;
};
#endif

template <class T>
struct DevBuf
{
    Backend* be = nullptr;
    T* p = nullptr;
    size_t n = 0;
    DevBuf() {}
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release()
    {
        if (p && be) be->free(p);
        p = nullptr;
        n = 0;
    }
    void alloc(Backend& b, size_t count, bool zero = true)
    {
        release();
        be = &b;
        n = count;
        p = (T*)b.alloc(count * sizeof(T));
        if (zero) b.zero(p, count * sizeof(T));
    }
    void upload(Backend& b, const std::vector<T>& h)
    {
        alloc(b, h.size(), false);
        if (!h.empty()) b.h2d(p, h.data(), h.size() * sizeof(T));
    }
};

} // namespace dab

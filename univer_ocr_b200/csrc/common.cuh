// Shared host/device helpers of libuocr (error reporting, launch accounting, small math).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "uocr.h"

namespace uocr {

void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// caching device allocator (runtime.cu); also used for library-internal scratch
int pool_alloc(void** ptr, size_t bytes, cudaStream_t st);
int pool_free(void* ptr, cudaStream_t st);
int pool_trim();

struct Scratch {                     // stream-ordered scratch from libuocr's caching allocator
    void* ptr = nullptr;
    cudaStream_t st;
    explicit Scratch(cudaStream_t s) : st(s) {}
    Scratch(const Scratch&) = delete;
    Scratch& operator=(const Scratch&) = delete;
    int alloc(size_t bytes) { return pool_alloc(&ptr, bytes, st); }
    ~Scratch() { if (ptr) pool_free(ptr, st); }
};

constexpr int kThreads = 256;

// grid size for a grid-stride elementwise kernel: enough CTAs to fill 148 SMs a few times over,
// never more than the work needs
inline int ew_grid(int64_t n, int per_thread = 4) {
    int64_t blocks = (n + (int64_t)kThreads * per_thread - 1) / ((int64_t)kThreads * per_thread);
    const int64_t cap = 148 * 16;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace uocr

#define UOCR_REQUIRE(cond, ...)                 \
    do {                                        \
        if (!(cond)) {                          \
            uocr::set_error(__VA_ARGS__);       \
            return UOCR_ERR_INVALID;            \
        }                                       \
    } while (0)

#define UOCR_CUDA(expr)                                                              \
    do {                                                                             \
        cudaError_t err__ = (expr);                                                  \
        if (err__ != cudaSuccess) {                                                  \
            uocr::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(err__), \
                            __FILE__, __LINE__);                                     \
            return UOCR_ERR_CUDA;                                                    \
        }                                                                            \
    } while (0)

// after a <<<>>> launch: count it and surface launch-configuration errors
#define UOCR_LAUNCHED(name)                                                          \
    do {                                                                             \
        uocr::g_launches.fetch_add(1, std::memory_order_relaxed);                    \
        cudaError_t err__ = cudaGetLastError();                                      \
        if (err__ != cudaSuccess) {                                                  \
            uocr::set_error("launch of %s failed: %s", name, cudaGetErrorString(err__)); \
            return UOCR_ERR_CUDA;                                                    \
        }                                                                            \
    } while (0)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// block-wide sum for blockDim.x == kThreads (8 warps); result valid in every thread
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* smem /* >= 8 elements */) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) smem[wid] = v;
    __syncthreads();
    T r = (lane < (blockDim.x >> 5)) ? smem[lane] : T(0);
    r = warp_sum(r);
    return r;
}

// ragged batches (ragged.cu, loss_opt.cu): image i's extent (h_i, w_i) from the device table, clamped to the canvas
__device__ __forceinline__ void ragged_extent(const int32_t* __restrict__ ext, int64_t i, int64_t h, int64_t w,
                                              int64_t& hi, int64_t& wi) {
    hi = min((int64_t)max(__ldg(ext + 2 * i), 0), h);
    wi = min((int64_t)max(__ldg(ext + 2 * i + 1), 0), w);
}

// epilogue flavour for the convolution kernels: ex2.approx + fast reciprocal (|rel err| ~ 1e-6 on
// the sigmoid, far inside the 1e-4 conv tolerance) -- the IEEE expf + divide sequence costs ~25
// instructions per output, which made the Cin = 1 stencils issue-bound (ncu: issue slots 80 % busy)
__device__ __forceinline__ float apply_act_fast(float v, int act, float alpha) {
    if (act == UOCR_ACT_LEAKY) return v >= 0.f ? v : alpha * v;
    if (act == UOCR_ACT_SIGMOID) return __fdividef(1.f, 1.f + __expf(-v));
    return v;
}

__device__ __forceinline__ float apply_act(float v, int act, float alpha) {
    if (act == UOCR_ACT_LEAKY) return v >= 0.f ? v : alpha * v;
    if (act == UOCR_ACT_SIGMOID) return 1.f / (1.f + expf(-v));
    return v;
}

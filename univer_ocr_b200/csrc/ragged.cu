// Ragged batches: N images of different sizes on one zero-filled (N, H, W, C) canvas, image i in
// canvas[i, :h_i, :w_i, :] with (h_i, w_i) = extents[i] (int32 pairs on the device).  Every layer the networks run pads
// with zeros, so a valid output pixel computed on the canvas reads what it would read if the image ran alone as long as
// each intermediate map is zero outside its own extent (DESIGN.md §3).  Every kernel clamps the extents to the canvas,
// so a bad table cannot make it write outside the canvas.
#include "common.cuh"

namespace uocr {
namespace {

// One warp per canvas row (image, y).  A row inside the extent zeroes its columns [w_i, W); a row below it is zeroed
// whole.  Rows wholly inside cost the extent lookup only, so the kernel's traffic is the padding, not the tensor.
__global__ void __launch_bounds__(kThreads) zero_outside_kernel(float* __restrict__ x, const int32_t* __restrict__ ext,
                                                                int64_t n, int64_t h, int64_t w, int64_t c) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
    for (int64_t row = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); row < n * h; row += warps) {
        const int64_t i = row / h, y = row - i * h;
        int64_t hi, wi;
        ragged_extent(ext, i, h, w, hi, wi);
        int64_t lo = (y < hi ? wi : 0) * c;
        const int64_t end = w * c;
        if (lo >= end) continue;
        float* base = x + row * end;
        // scalar head up to a 16-byte boundary, float4 body, scalar tail
        const int64_t head = min(end, lo + (int64_t)((4 - ((reinterpret_cast<uintptr_t>(base + lo) >> 2) & 3)) & 3));
        for (int64_t j = lo + lane; j < head; j += 32) base[j] = 0.f;
        lo = head;
        const int64_t quads = (end - lo) >> 2;
        float4* body = reinterpret_cast<float4*>(base + lo);
        for (int64_t q = lane; q < quads; q += 32) body[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int64_t j = lo + 4 * quads + lane; j < end; j += 32) base[j] = 0.f;
    }
}

// One warp per canvas row: image i's row y (w_i * c contiguous floats of srcs[i]) and the zeros after it, or a row of
// zeros below the extent.
__global__ void __launch_bounds__(kThreads) pack_hw_kernel(const float* const* __restrict__ srcs,
                                                           const int32_t* __restrict__ ext, float* __restrict__ canvas,
                                                           int64_t n, int64_t h, int64_t w, int64_t c) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
    for (int64_t row = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); row < n * h; row += warps) {
        const int64_t i = row / h, y = row - i * h;
        int64_t hi, wi;
        ragged_extent(ext, i, h, w, hi, wi);
        const int64_t len = (y < hi ? wi : 0) * c, end = w * c;
        const float* src = len ? srcs[i] + y * len : nullptr;
        float* dst = canvas + row * end;
        for (int64_t j = lane; j < end; j += 32) dst[j] = j < len ? __ldg(src + j) : 0.f;
    }
}

// One warp per canvas row inside an extent: the row's w_i * c floats back to dsts[i].
__global__ void __launch_bounds__(kThreads) unpack_hw_kernel(const float* __restrict__ canvas, const int32_t* __restrict__ ext,
                                                             float* const* __restrict__ dsts, int64_t n, int64_t h,
                                                             int64_t w, int64_t c) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
    for (int64_t row = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); row < n * h; row += warps) {
        const int64_t i = row / h, y = row - i * h;
        int64_t hi, wi;
        ragged_extent(ext, i, h, w, hi, wi);
        if (y >= hi) continue;
        const int64_t len = wi * c;
        const float* src = canvas + row * w * c;
        float* dst = dsts[i] + y * len;
        for (int64_t j = lane; j < len; j += 32) dst[j] = __ldg(src + j);
    }
}

int row_grid(int64_t rows) {
    const int64_t per_block = kThreads / 32;
    int64_t blocks = (rows + per_block - 1) / per_block;
    if (blocks > 148 * 16) blocks = 148 * 16;
    return (int)(blocks < 1 ? 1 : blocks);
}

// the host array of N device pointers, staged in stream-ordered scratch
int stage_pointers(Scratch& table, const void* const* host, int64_t n, cudaStream_t st) {
    int rc = table.alloc((size_t)n * sizeof(void*));
    if (rc != UOCR_OK) return rc;
    UOCR_CUDA(cudaMemcpyAsync(table.ptr, host, (size_t)n * sizeof(void*), cudaMemcpyHostToDevice, st));
    return UOCR_OK;
}

}  // namespace
}  // namespace uocr

using namespace uocr;

#define RAGGED_REQUIRE_DIMS(n, h, w, c) \
    UOCR_REQUIRE((n) > 0 && (h) > 0 && (w) > 0 && (c) > 0, "non-positive dimension")

extern "C" int uocr_zero_outside_hw_f32(float* x, const int32_t* extents, int64_t n, int64_t h, int64_t w, int64_t c,
                                        void* stream) {
    UOCR_REQUIRE(x && extents, "NULL pointer");
    RAGGED_REQUIRE_DIMS(n, h, w, c);
    zero_outside_kernel<<<row_grid(n * h), kThreads, 0, as_stream(stream)>>>(x, extents, n, h, w, c);
    UOCR_LAUNCHED("zero_outside_hw");
    return UOCR_OK;
}

extern "C" int uocr_pack_hw_f32(const float* const* srcs, const int32_t* extents, float* canvas, int64_t n, int64_t h,
                                int64_t w, int64_t c, void* stream) {
    UOCR_REQUIRE(srcs && extents && canvas, "NULL pointer");
    RAGGED_REQUIRE_DIMS(n, h, w, c);
    for (int64_t i = 0; i < n; ++i) UOCR_REQUIRE(srcs[i], "NULL source pointer (image %lld)", (long long)i);
    const cudaStream_t st = as_stream(stream);
    Scratch table(st);
    int rc = stage_pointers(table, reinterpret_cast<const void* const*>(srcs), n, st);
    if (rc != UOCR_OK) return rc;
    pack_hw_kernel<<<row_grid(n * h), kThreads, 0, st>>>(static_cast<const float* const*>(table.ptr), extents, canvas,
                                                         n, h, w, c);
    UOCR_LAUNCHED("pack_hw");
    return UOCR_OK;
}

extern "C" int uocr_unpack_hw_f32(const float* canvas, const int32_t* extents, float* const* dsts, int64_t n, int64_t h,
                                  int64_t w, int64_t c, void* stream) {
    UOCR_REQUIRE(dsts && extents && canvas, "NULL pointer");
    RAGGED_REQUIRE_DIMS(n, h, w, c);
    for (int64_t i = 0; i < n; ++i) UOCR_REQUIRE(dsts[i], "NULL destination pointer (image %lld)", (long long)i);
    const cudaStream_t st = as_stream(stream);
    Scratch table(st);
    int rc = stage_pointers(table, reinterpret_cast<const void* const*>(dsts), n, st);
    if (rc != UOCR_OK) return rc;
    unpack_hw_kernel<<<row_grid(n * h), kThreads, 0, st>>>(canvas, extents, static_cast<float* const*>(table.ptr), n, h,
                                                           w, c);
    UOCR_LAUNCHED("unpack_hw");
    return UOCR_OK;
}

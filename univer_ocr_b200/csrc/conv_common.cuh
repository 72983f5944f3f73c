// Geometry shared by the convolution kernels + the dispatch seams between the general path
// (conv.cu) and the shape-specialised paths (conv_fast.cu).
#pragma once
#include "common.cuh"

namespace uocr {

struct ConvGeom {
    int n, h, w, cin, cout;
    int kh, kw, ph, pw, sh, sw;
    int ho, wo;
    float padding_value;
    int bias;
    int ups;            // 1 or 2: nearest upsample folded into the forward input read (h, w are
                        // the LOGICAL, upsampled sizes; the stored tensor is (h/ups, w/ups))
};

// Shape-specialised kernels.  Each returns UOCR_ERR_UNSUPPORTED when it has no kernel for the
// geometry / math mode, in which case the caller runs the general kernel.
int conv_fwd_fast(const ConvGeom& g, int ups, int math_mode, const float* x, const float* w,
                  const float* b, float* y, int act, float alpha, cudaStream_t st, const float* w_kmajor = nullptr);
int conv3x3_pair_fwd(const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                     float* y, int64_t n, int64_t h, int64_t w, int c1, int act1, float alpha1, int act2,
                     float alpha2, cudaStream_t st);
int conv_dgrad_fast(const ConvGeom& g, int math_mode, const float* dy, const float* w, float* dx,
                    cudaStream_t st);
size_t conv_wgrad_fast_workspace(const ConvGeom& g, int math_mode);
int conv_wgrad_fast(const ConvGeom& g, int math_mode, const float* x, const float* dy, float* dw,
                    float* db, int accumulate, float* ws, cudaStream_t st);

// tcgen05 implicit-GEMM forward (tc_gemm.cu): Cin % 32 == 0, stride_w == 1, zero padding
int conv_fwd_tc(const ConvGeom& g, const float* x, const float* w, const float* w_kmajor /* (Cout, K) or NULL */,
                const float* b, float* y, int act, float alpha, cudaStream_t st);

// 5x5 / stride 1 / Cin = 4 forward as a row GEMM on tcgen05 with TMEM-resident windows (conv_row_tc.cu)
int conv55_row_tc(const ConvGeom& g, const float* x, const float* w, const float* b, float* y, int act, float alpha,
                  cudaStream_t st);
// both convolutions as tcgen05.mma with TMEM-resident A operands (conv_pair_tc.cu)
int conv3x3_pair_tmem(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, float* y,
                      int64_t n, int64_t h, int64_t w, int c1, int act1, float alpha1, int act2, float alpha2,
                      cudaStream_t st);
// GEMM 1 reads the image rows in shared memory directly (overlapping descriptor rows), warp-specialised persistent
// kernel (conv_pair_rows_tc.cu); needs w % 4 == 0
int conv3x3_pair_rows(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, float* y,
                      int64_t n, int64_t h, int64_t w, int c1, int act1, float alpha1, int act2, float alpha2,
                      cudaStream_t st);
size_t conv3x3_pair_bwd_workspace(int64_t n, int64_t h, int64_t w, int c1);
int conv3x3_pair_bwd(const float* x, const float* w1, const float* b1, const float* w2, const float* dy, float* dx,
                     float* dw1, float* db1, float* dw2, float* db2, int64_t n, int64_t h, int64_t w, int c1,
                     int act1, float alpha1, int accumulate, float* ws, cudaStream_t st, int math_mode = UOCR_MATH_FP32);
// tensor-core assisted weight gradients of the pair (conv_pair_bwd_tc.cu): partial sums into ws
size_t conv3x3_pair_wgrad_tc_workspace(int64_t n, int64_t h, int64_t w, int c1);
int conv3x3_pair_wgrad_tc(const float* x, const float* w1, const float* b1, const float* w2, const float* dy, float* ws,
                          int64_t n, int64_t h, int64_t w, int c1, int act1, float alpha1, int* nblk_out, cudaStream_t st);
int conv_dgrad_tc(const ConvGeom& g, const float* dy, const float* w, float* dx, cudaStream_t st);
int conv_wgrad_tc(const ConvGeom& g, const float* x, const float* dy, float* dw, float* db, int accumulate,
                  cudaStream_t st);

// General kernels (conv.cu), exposed so the fast paths can delegate sub-problems.
int conv_fwd_general(const ConvGeom& g, const float* x, const float* w, const float* b, float* y,
                     int act, float alpha, cudaStream_t st);
int conv_dgrad_general(const ConvGeom& g, const float* dy, const float* w, float* dx, cudaStream_t st);
size_t conv_wgrad_general_workspace(const ConvGeom& g);
int conv_wgrad_general(const ConvGeom& g, const float* x, const float* dy, float* dw, float* db,
                       int accumulate, float* ws, cudaStream_t st);

}  // namespace uocr

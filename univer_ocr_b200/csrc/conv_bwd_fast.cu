// Shape-specialised BACKWARD kernels for my_model's small-channel convolutions
// (nn/layers/convolutional.py:101-145 / :197-288 are the reference semantics).
//
//   dgrad, stride 1 : dX = conv_fwd(dy, flip(w)^T, padding k-1-p) -- the tuned forward stencils
//                     are reused on a flipped / transposed copy of the (tiny) weight tensor
//   dgrad, strided  : gather form with the tap parity resolved at compile time
//                     (thread = PX consecutive input pixels x all input channels)
//   wgrad           : thread = strip of PX output columns x R output rows, ALL taps of one
//                     (ci-chunk, co-chunk) accumulated in registers while streaming down the rows;
//                     one block-level reduction per CTA at the end (warp shuffles + smem), partials
//                     to workspace[chunk][element][cta], summed by a finalize kernel -- deterministic,
//                     no atomics; db is accumulated alongside (padding_value border included in dW,
//                     as the reference's saved padded input does).
#include "conv_common.cuh"

namespace uocr {

template <int CIV> struct BVec;
template <> struct BVec<1> {
    float v[1];
    __device__ __forceinline__ void load(const float* p) { v[0] = __ldg(p); }
    __device__ __forceinline__ void fill(float f) { v[0] = f; }
};
template <> struct BVec<2> {
    float v[2];
    __device__ __forceinline__ void load(const float* p) {
        const float2 t = __ldg(reinterpret_cast<const float2*>(p));
        v[0] = t.x; v[1] = t.y;
    }
    __device__ __forceinline__ void fill(float f) { v[0] = v[1] = f; }
};
template <> struct BVec<4> {
    float v[4];
    __device__ __forceinline__ void load(const float* p) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void fill(float f) { v[0] = v[1] = v[2] = v[3] = f; }
};

// ------------------------------------------------------------------ weight flip + transpose
// wt[ky'][kx'][co][ci] = w[kh-1-ky'][kw-1-kx'][ci][co]
__global__ void __launch_bounds__(256) flip_transpose_kernel(const float* __restrict__ w, float* __restrict__ wt,
                                                             int kh, int kw, int cin, int cout) {
    const int total = kh * kw * cin * cout;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < total; i += gridDim.x * 256) {
        const int ci = i % cin;
        const int co = (i / cin) % cout;
        const int kx = (i / (cin * cout)) % kw;
        const int ky = i / (cin * cout * kw);
        wt[i] = w[(((kh - 1 - ky) * kw + (kw - 1 - kx)) * cin + ci) * cout + co];
    }
}

// ------------------------------------------------------------------ strided dgrad (COUT <= 4)
template <int KH, int KW, int SH, int SW, int PW, int CIN, int COUT, int PX>
__global__ void __launch_bounds__(256) conv_small_dgrad_kernel(ConvGeom g, const float* __restrict__ dy,
                                                               const float* __restrict__ w,
                                                               float* __restrict__ dx) {
    static_assert(PX % SW == 0, "strip start must keep the tap parity compile-time");
    __shared__ float s_w[KH * KW * CIN * COUT];              // [ky][kx][ci][co]
    for (int i = threadIdx.x; i < KH * KW * CIN * COUT; i += 256) s_w[i] = w[i];
    __syncthreads();
    // dy columns touched by this strip: ox = ix0 / SW + off, off in [OFF_LO, OFF_HI]
    constexpr int OFF_LO = (PW - (KW - 1)) >= 0 ? (PW - (KW - 1)) / SW : -(((KW - 1) - PW + SW - 1) / SW);
    constexpr int OFF_HI = (PX - 1 + PW) / SW;
    constexpr int NDY = OFF_HI - OFF_LO + 1;

    const int strips = (g.w + PX - 1) / PX;
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int xs = (int)(idx % strips);
    const int iy = (int)((idx / strips) % g.h);
    const int64_t n = idx / ((int64_t)strips * g.h);
    if (n >= g.n) return;
    const int ix0 = xs * PX;
    const int oxb = ix0 / SW + OFF_LO;

    float acc[PX][CIN];
#pragma unroll
    for (int p = 0; p < PX; ++p)
#pragma unroll
        for (int c = 0; c < CIN; ++c) acc[p][c] = 0.f;

#pragma unroll
    for (int ky = 0; ky < KH; ++ky) {
        const int ty = iy + g.ph - ky;
        if (ty < 0 || ty % SH != 0) continue;
        const int oy = ty / SH;
        if (oy >= g.ho) continue;
        const float* drow = dy + ((n * g.ho + oy) * (int64_t)g.wo) * COUT;
        BVec<COUT> seg[NDY];
#pragma unroll
        for (int j = 0; j < NDY; ++j) {
            const int ox = oxb + j;
            if (ox >= 0 && ox < g.wo) seg[j].load(drow + (int64_t)ox * COUT);
            else seg[j].fill(0.f);
        }
#pragma unroll
        for (int kx = 0; kx < KW; ++kx) {
#pragma unroll
            for (int p = 0; p < PX; ++p) {
                const int q = p + PW - kx;                       // compile-time after unrolling
                if (q % SW != 0) continue;
                const int j = (q >= 0 ? q / SW : -((-q) / SW)) - OFF_LO;
#pragma unroll
                for (int c = 0; c < CIN; ++c)
#pragma unroll
                    for (int o = 0; o < COUT; ++o)
                        acc[p][c] = fmaf(seg[j].v[o], s_w[((ky * KW + kx) * CIN + c) * COUT + o], acc[p][c]);
            }
        }
    }
    float* dp = dx + ((n * g.h + iy) * (int64_t)g.w + ix0) * CIN;
#pragma unroll
    for (int p = 0; p < PX; ++p) {
        if (ix0 + p >= g.w) break;
#pragma unroll
        for (int c = 0; c < CIN; ++c) dp[p * CIN + c] = acc[p][c];
    }
}

template <int KH, int KW, int SH, int SW, int PW, int CIN, int COUT, int PX>
static int launch_small_dgrad(const ConvGeom& g, const float* dy, const float* w, float* dx, cudaStream_t st) {
    const int strips = (g.w + PX - 1) / PX;
    const int64_t blocks = ceil_div((int64_t)g.n * g.h * strips, 256);
    if (blocks > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    conv_small_dgrad_kernel<KH, KW, SH, SW, PW, CIN, COUT, PX><<<(unsigned)blocks, 256, 0, st>>>(g, dy, w, dx);
    UOCR_LAUNCHED("conv_small_dgrad");
    return UOCR_OK;
}

// dgrad for Cin == 1, Cout % 64 == 0 (Char conv_1: 5x3, stride (2,1), 1 <- 64): dx(n, iy, ix) is a dot product over
// the taps that reach the pixel and all output channels.  Warp = one input pixel, lane = a channel pair (64-bit
// coalesced loads of dy, weights in shared memory), one shuffle reduction per pixel.  Any kernel / stride / padding.
// (Plain Model.train computes this gradient like the reference does although nothing consumes it; the general
// gather kernel needed 0.9 ms for it at batch 64.)
__global__ void __launch_bounds__(256) conv_dgrad_cin1_warp_kernel(ConvGeom g, const float* __restrict__ dy,
                                                                   const float* __restrict__ w,
                                                                   float* __restrict__ dx) {
    extern __shared__ float s_wd[];                          // (kh*kw, cout)
    for (int i = threadIdx.x; i < g.kh * g.kw * g.cout; i += 256) s_wd[i] = w[i];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t pixels = (int64_t)g.n * g.h * g.w;
    const int64_t warps = (int64_t)gridDim.x * 8;
    for (int64_t p = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); p < pixels; p += warps) {
        const int ix = (int)(p % g.w);
        const int iy = (int)((p / g.w) % g.h);
        const int64_t n = p / ((int64_t)g.w * g.h);
        float acc = 0.f;
        for (int ky = 0; ky < g.kh; ++ky) {
            const int ty = iy + g.ph - ky;
            if (ty < 0 || ty % g.sh) continue;
            const int oy = ty / g.sh;
            if (oy >= g.ho) continue;
            for (int kx = 0; kx < g.kw; ++kx) {
                const int tx = ix + g.pw - kx;
                if (tx < 0 || tx % g.sw) continue;
                const int ox = tx / g.sw;
                if (ox >= g.wo) continue;
                const float* d = dy + ((n * g.ho + oy) * g.wo + ox) * g.cout;
                const float* ww = s_wd + (ky * g.kw + kx) * g.cout;
                for (int c0 = 2 * lane; c0 < g.cout; c0 += 64) {
                    const float2 dv = *reinterpret_cast<const float2*>(d + c0);
                    const float2 wv = *reinterpret_cast<const float2*>(ww + c0);
                    acc = fmaf(dv.x, wv.x, acc);
                    acc = fmaf(dv.y, wv.y, acc);
                }
            }
        }
        acc = warp_sum(acc);
        if (lane == 0) dx[p] = acc;
    }
}

// Same gradient organised from the OUTPUT side (taps as the N dimension of a small GEMM): lane = one output pixel,
// Z[tap] = dy(pixel, :) . w(tap, :) for all KH*KW taps from one pass over the pixel's channel vector (weights broadcast
// from shared memory), then Z[tap] is added to the input pixel that tap reaches.  Each dy element is read once;
// dx must be zeroed by the caller.  The float atomics make the summation order of the <= KH*KW terms per input pixel
// run-dependent (as in the split-K GEMMs).
template <int KH, int KW>
__global__ void __launch_bounds__(128) conv_dgrad_cin1_scatter_kernel(ConvGeom g, const float* __restrict__ dy,
                                                                      const float* __restrict__ w,
                                                                      float* __restrict__ dx) {
    constexpr int NT = KH * KW, NTP = (NT + 3) & ~3;
    extern __shared__ __align__(16) float s_ws[];            // (cout, NTP): the taps of a channel are contiguous
    for (int i = threadIdx.x; i < NTP * g.cout; i += 128) {
        const int c = i / NTP, t = i - c * NTP;
        s_ws[i] = t < NT ? w[t * g.cout + c] : 0.f;
    }
    __syncthreads();
    const int64_t pixels = (int64_t)g.n * g.ho * g.wo;
    for (int64_t p = (int64_t)blockIdx.x * 128 + threadIdx.x; p < pixels; p += (int64_t)gridDim.x * 128) {
        const int ox = (int)(p % g.wo);
        const int oy = (int)((p / g.wo) % g.ho);
        const int64_t n = p / ((int64_t)g.wo * g.ho);
        float z[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) z[t] = 0.f;
        const float4* d = reinterpret_cast<const float4*>(dy + p * g.cout);
        for (int c4 = 0; c4 < g.cout / 4; ++c4) {
            const float4 v = d[c4];
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4* ws4 = reinterpret_cast<const float4*>(s_ws + (c4 * 4 + j) * NTP);
#pragma unroll
                for (int q = 0; q < NTP / 4; ++q) {
                    const float4 wv = ws4[q];                // broadcast: every lane reads the same 16 bytes
                    const float wq[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
                    for (int r = 0; r < 4; ++r)
                        if (4 * q + r < NT) z[4 * q + r] = fmaf(vv[j], wq[r], z[4 * q + r]);
                }
            }
        }
        float* xrow = dx + n * g.h * g.w;
#pragma unroll
        for (int ky = 0; ky < KH; ++ky) {
            const int iy = oy * g.sh + ky - g.ph;
            if (iy < 0 || iy >= g.h) continue;
#pragma unroll
            for (int kx = 0; kx < KW; ++kx) {
                const int ix = ox * g.sw + kx - g.pw;
                if (ix >= 0 && ix < g.w) atomicAdd(xrow + (int64_t)iy * g.w + ix, z[ky * KW + kx]);
            }
        }
    }
}

int conv_dgrad_fast(const ConvGeom& g, int math_mode, const float* dy, const float* w, float* dx,
                    cudaStream_t st) {
    if (math_mode == UOCR_MATH_TF32) {
        const int rc = conv_dgrad_tc(g, dy, w, dx, st);
        if (rc != UOCR_ERR_UNSUPPORTED) return rc;
    }
    if (g.sh == 1 && g.sw == 1 && g.kh - 1 - g.ph >= 0 && g.kw - 1 - g.pw >= 0 &&
        (int64_t)g.kh * g.kw * g.cin * g.cout <= 4096) {
        // stride 1: forward stencil on the flipped / transposed weights
        Scratch wt(st);
        int rc = wt.alloc(sizeof(float) * g.kh * g.kw * g.cin * g.cout);
        if (rc) return rc;
        flip_transpose_kernel<<<4, 256, 0, st>>>(w, (float*)wt.ptr, g.kh, g.kw, g.cin, g.cout);
        UOCR_LAUNCHED("flip_transpose");
        ConvGeom t = g;
        t.h = g.ho; t.w = g.wo; t.cin = g.cout; t.cout = g.cin;
        t.ph = g.kh - 1 - g.ph; t.pw = g.kw - 1 - g.pw;
        t.ho = g.h; t.wo = g.w; t.padding_value = 0.f; t.bias = 0; t.ups = 1;
        // TF32 mode: the 5x5 Cin = 4 row GEMM also serves the dgrad of the Line 4 -> 4 layers (no bias); everything
        // else stays on the FP32 stencils (conv_fwd_tc needs Cin % 32 == 0 and would only see tiny channel counts here)
        const bool row_tc = math_mode == UOCR_MATH_TF32 && t.cin == 4 && t.kh == 5 && t.kw == 5;
        rc = conv_fwd_fast(t, 1, row_tc ? UOCR_MATH_TF32 : UOCR_MATH_FP32, dy, (const float*)wt.ptr, nullptr, dx,
                           UOCR_ACT_NONE, 0.f, st);
        if (rc == UOCR_ERR_UNSUPPORTED)
            rc = conv_fwd_general(t, dy, (const float*)wt.ptr, nullptr, dx, UOCR_ACT_NONE, 0.f, st);
        return rc;
    }
#define UOCR_DG(KH_, KW_, SH_, SW_, PW_, CIN_, COUT_, PX_)                                             \
    if (g.kh == KH_ && g.kw == KW_ && g.sh == SH_ && g.sw == SW_ && g.pw == PW_ && g.cin == CIN_ &&     \
        g.cout == COUT_)                                                                                \
        return launch_small_dgrad<KH_, KW_, SH_, SW_, PW_, CIN_, COUT_, PX_>(g, dy, w, dx, st);
    if (((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx)) & 15) == 0) {
        UOCR_DG(5, 5, 2, 2, 2, 1, 1, 8)      // Paragraph down_*
        UOCR_DG(5, 5, 2, 2, 2, 1, 4, 8)      // Line down_1
        UOCR_DG(5, 5, 2, 2, 2, 4, 4, 4)      // Line down_2
    }
#undef UOCR_DG
    if (g.cin == 1 && g.kh == 5 && g.kw == 3 && g.cout % 4 == 0 && g.cout <= 256 &&
        (reinterpret_cast<uintptr_t>(dy) & 15) == 0) {       // Char conv_1
        UOCR_CUDA(cudaMemsetAsync(dx, 0, sizeof(float) * g.n * g.h * g.w, st));
        const int64_t pixels = (int64_t)g.n * g.ho * g.wo;
        int64_t blocks = ceil_div(pixels, 128);
        if (blocks > 148 * 64) blocks = 148 * 64;
        conv_dgrad_cin1_scatter_kernel<5, 3><<<(int)blocks, 128, sizeof(float) * 16 * g.cout, st>>>(g, dy, w, dx);
        UOCR_LAUNCHED("conv_dgrad_cin1_scatter");
        return UOCR_OK;
    }
    if (g.cin == 1 && g.cout % 64 == 0 && (int64_t)g.kh * g.kw * g.cout <= 8192 &&
        (reinterpret_cast<uintptr_t>(dy) & 7) == 0) {
        const int64_t pixels = (int64_t)g.n * g.h * g.w;
        int64_t blocks = ceil_div(pixels, 8 * 4);            // ~4 pixels per warp
        if (blocks > 148 * 32) blocks = 148 * 32;
        conv_dgrad_cin1_warp_kernel<<<(int)blocks, 256, sizeof(float) * g.kh * g.kw * g.cout, st>>>(g, dy, w, dx);
        UOCR_LAUNCHED("conv_dgrad_cin1_warp");
        return UOCR_OK;
    }
    return UOCR_ERR_UNSUPPORTED;
}

// ------------------------------------------------------------------ wgrad
template <int KH, int KW, int SH, int SW, int CIN, int CIV, int COT, int PX, int R>
__global__ void __launch_bounds__(256) conv_small_wgrad_kernel(ConvGeom g, const float* __restrict__ x,
                                                               const float* __restrict__ dy,
                                                               float* __restrict__ ws, int nblk) {
    constexpr int NACC = KH * KW * CIV * COT;
    constexpr int NOUT = NACC + COT;                         // + db partials
    constexpr int NIN = (PX - 1) * SW + KW;
    __shared__ float red[8][NOUT];
    const int cochunks = g.cout / COT;
    const int cic = blockIdx.y / cochunks, coc = blockIdx.y % cochunks;
    const int ci0 = cic * CIV, co0 = coc * COT;

    const int strips = (g.wo + PX - 1) / PX;
    const int rgroups = (g.ho + R - 1) / R;
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int xs = (int)(idx % strips);
    const int rg = (int)((idx / strips) % rgroups);
    const int64_t n = idx / ((int64_t)strips * rgroups);
    const bool live = n < g.n;

    float acc[KH][KW][CIV][COT];
    float dbacc[COT];
#pragma unroll
    for (int a = 0; a < KH; ++a)
#pragma unroll
        for (int b = 0; b < KW; ++b)
#pragma unroll
            for (int c = 0; c < CIV; ++c)
#pragma unroll
                for (int d = 0; d < COT; ++d) acc[a][b][c][d] = 0.f;
#pragma unroll
    for (int d = 0; d < COT; ++d) dbacc[d] = 0.f;

    if (live) {
        const int ox0 = xs * PX;
        const int ix0 = ox0 * SW - g.pw;
        const int oy_end = min(g.ho, (rg + 1) * R);
        for (int oy = rg * R; oy < oy_end; ++oy) {
            float dyv[PX][COT];
            const float* drow = dy + ((n * g.ho + oy) * (int64_t)g.wo + ox0) * g.cout + co0;
#pragma unroll
            for (int p = 0; p < PX; ++p) {
                if (ox0 + p < g.wo) {
                    BVec<COT> t;
                    t.load(drow + (int64_t)p * g.cout);
#pragma unroll
                    for (int d = 0; d < COT; ++d) dyv[p][d] = t.v[d];
                } else {
#pragma unroll
                    for (int d = 0; d < COT; ++d) dyv[p][d] = 0.f;
                }
#pragma unroll
                for (int d = 0; d < COT; ++d) dbacc[d] += dyv[p][d];
            }
#pragma unroll
            for (int ky = 0; ky < KH; ++ky) {
                const int iy = oy * SH + ky - g.ph;
                const bool yin = iy >= 0 && iy < g.h;
                const float* xrow = x + ((n * g.h + (yin ? iy : 0)) * (int64_t)g.w) * CIN + ci0;
                BVec<CIV> xin[NIN];
#pragma unroll
                for (int j = 0; j < NIN; ++j) {
                    const int ix = ix0 + j;
                    if (yin && ix >= 0 && ix < g.w) xin[j].load(xrow + (int64_t)ix * CIN);
                    else xin[j].fill(g.padding_value);
                }
#pragma unroll
                for (int kx = 0; kx < KW; ++kx)
#pragma unroll
                    for (int p = 0; p < PX; ++p)
#pragma unroll
                        for (int c = 0; c < CIV; ++c)
#pragma unroll
                            for (int d = 0; d < COT; ++d)
                                acc[ky][kx][c][d] = fmaf(xin[p * SW + kx].v[c], dyv[p][d], acc[ky][kx][c][d]);
            }
        }
    }

    // ---- CTA reduction: shuffle within warps, smem across the 8 warps
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < KH; ++a)
#pragma unroll
        for (int b = 0; b < KW; ++b)
#pragma unroll
            for (int c = 0; c < CIV; ++c)
#pragma unroll
                for (int d = 0; d < COT; ++d) {
                    const float s = warp_sum(acc[a][b][c][d]);
                    if (lane == 0) red[wid][((a * KW + b) * CIV + c) * COT + d] = s;
                }
#pragma unroll
    for (int d = 0; d < COT; ++d) {
        const float s = warp_sum(dbacc[d]);
        if (lane == 0) red[wid][NACC + d] = s;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < NOUT; e += 256) {
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) s += red[k][e];
        ws[((int64_t)blockIdx.y * NOUT + e) * nblk + blockIdx.x] = s;
    }
}

// 5 x 5 / stride 1 / 1 -> 1 channel weight gradient (Paragraph up_*, end): same decomposition and workspace layout
// as conv_small_wgrad_kernel<5,5,1,1,1,1,1,8,R>, but the five input rows an output row needs stay in a register
// ring while the thread walks down its R rows -- one new input row (6 x 64-bit loads) and one dy row (2 x 128-bit
// loads) per 200 FMA instead of 68 scalar loads (the generic kernel was L1-wavefront bound: 157 us for 187 MB).
// UPS: x is stored at half resolution (N, H/2, W/2) and the convolution reads its x2 nearest upsampling (the
// Upsample2D layer in front folded into the addressing, as in the forward kernels): input pixel (iy, ix) = x(iy/2, ix/2).
template <int R, bool UPS>
__global__ void __launch_bounds__(256) conv55_c1_wgrad_roll_kernel(ConvGeom g, const float* __restrict__ x,
                                                                   const float* __restrict__ dy,
                                                                   float* __restrict__ ws, int nblk) {
    constexpr int PX = 8, NIN = 12, NOUT = 26;
    __shared__ float red[8][NOUT];
    const int strips = (g.wo + PX - 1) / PX;
    const int rgroups = (g.ho + R - 1) / R;
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int xs = (int)(idx % strips);
    const int rg = (int)((idx / strips) % rgroups);
    const int64_t n = idx / ((int64_t)strips * rgroups);
    float acc[5][5];
    float dbacc = 0.f;
#pragma unroll
    for (int a = 0; a < 5; ++a)
#pragma unroll
        for (int b = 0; b < 5; ++b) acc[a][b] = 0.f;
    if (n < g.n) {
        const int ox0 = xs * PX, ix0 = ox0 - 2;
        const int oy0 = rg * R, oy_end = min(g.ho, oy0 + R);
        const int sw_ = UPS ? g.w / 2 : g.w;                 // stored row pitch
        const float* xim = x + n * (int64_t)(UPS ? g.h / 2 : g.h) * sw_;
        const float* dyim = dy + n * g.ho * (int64_t)g.wo;
        float xr[5][NIN];                                    // ring slot = (input row - (oy0 - 2)) % 5
        auto load_row = [&](int iy, float* dst) {
            const bool yin = iy >= 0 && iy < g.h;
            const float* row = xim + (int64_t)(yin ? (UPS ? iy >> 1 : iy) : 0) * sw_;
#pragma unroll
            for (int q = 0; q < NIN / 2; ++q) {
                const int ix = ix0 + 2 * q;                  // even; W even: the pair is inside or outside together
                float2 v = make_float2(g.padding_value, g.padding_value);
                if (yin && ix >= 0 && ix < g.w) {
                    if (UPS) { const float t = __ldg(row + (ix >> 1)); v = make_float2(t, t); }
                    else v = __ldg(reinterpret_cast<const float2*>(row + ix));
                }
                dst[2 * q] = v.x; dst[2 * q + 1] = v.y;
            }
        };
#pragma unroll
        for (int a = 0; a < 4; ++a) load_row(oy0 - 2 + a, xr[a]);
        for (int ob = 0; ob < R; ob += 5) {
#pragma unroll
            for (int u = 0; u < 5; ++u) {
                const int oy = oy0 + ob + u;
                if (oy < oy_end) {                           // thread-uniform
                    load_row(oy + 2, xr[(u + 4) % 5]);
                    float dyv[PX];
                    const float* drow = dyim + (int64_t)oy * g.wo + ox0;
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ox0 + 4 * q < g.wo) v = __ldg(reinterpret_cast<const float4*>(drow + 4 * q));   // wo % 4 == 0
                        dyv[4 * q] = v.x; dyv[4 * q + 1] = v.y; dyv[4 * q + 2] = v.z; dyv[4 * q + 3] = v.w;
                    }
#pragma unroll
                    for (int p = 0; p < PX; ++p) dbacc += dyv[p];
#pragma unroll
                    for (int ky = 0; ky < 5; ++ky)
#pragma unroll
                        for (int kx = 0; kx < 5; ++kx)
#pragma unroll
                            for (int p = 0; p < PX; ++p)
                                acc[ky][kx] = fmaf(xr[(u + ky) % 5][p + kx], dyv[p], acc[ky][kx]);
                }
            }
        }
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 5; ++a)
#pragma unroll
        for (int b = 0; b < 5; ++b) {
            const float t = warp_sum(acc[a][b]);
            if (lane == 0) red[wid][a * 5 + b] = t;
        }
    {
        const float t = warp_sum(dbacc);
        if (lane == 0) red[wid][25] = t;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < NOUT; e += 256) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][e];
        ws[((int64_t)blockIdx.y * NOUT + e) * nblk + blockIdx.x] = t;
    }
}

// 5 x 5 / stride 1 / padding 2 / Cin = 4 weight gradient (Line up_*, end: Cout = 4 or 2), shared-memory tiled.
// The generic kernel above re-reads every input window from L1 for each kernel row and each output-channel chunk
// (147 us for 67 MB: L1-wavefront bound).  Here a CTA stages a 16 x 64 output tile's x (20 x 68 pixels) and dy once
// (16-byte cp.async, zero fill outside the image = the zero padding) and its five warps each own one kernel ROW ky:
// lane = output column, 5 (kx) x 4 (ci) x Cout accumulators per thread, 6 conflict-free 128-bit shared loads per 80
// FMA.  CTAs are persistent over tiles; partial sums go to the workspace in conv_small_wgrad_finalize_kernel's layout
// (one chunk, civ = 4, cot = Cout).  UPS: x is stored at half resolution (folded Upsample2D(2)).
constexpr int WT_TY = 16, WT_TX = 64, WT_THREADS = 160;

template <int COUT, bool UPS>
__global__ void __launch_bounds__(WT_THREADS) conv55_c4_wgrad_tiled_kernel(ConvGeom g, const float* __restrict__ x,
                                                                           const float* __restrict__ dy,
                                                                           float* __restrict__ ws, int nblk) {
    constexpr int XP = WT_TX + 4, XR = WT_TY + 4;
    constexpr int NACC = 25 * 4 * COUT, NOUT = NACC + COUT;
    extern __shared__ __align__(16) float wt_smem[];
    float4* s_x = reinterpret_cast<float4*>(wt_smem);                       // [XR][XP]
    float* s_dy = wt_smem + XR * XP * 4;                                     // [TY][TX][COUT]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;              // warp = ky
    const int tiles_x = (g.wo + WT_TX - 1) / WT_TX, tiles_y = (g.ho + WT_TY - 1) / WT_TY;
    const int64_t ntiles = (int64_t)g.n * tiles_y * tiles_x;
    const int sw = UPS ? g.w / 2 : g.w, sh = UPS ? g.h / 2 : g.h;           // stored input size
    float acc[5][4][COUT];
    float dbacc[COUT];
#pragma unroll
    for (int a = 0; a < 5; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int c = 0; c < COUT; ++c) acc[a][b][c] = 0.f;
#pragma unroll
    for (int c = 0; c < COUT; ++c) dbacc[c] = 0.f;
    const uint32_t sx_addr = static_cast<uint32_t>(__cvta_generic_to_shared(s_x));
    const uint32_t sdy_addr = static_cast<uint32_t>(__cvta_generic_to_shared(s_dy));

    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int tx = (int)(tile % tiles_x), ty = (int)((tile / tiles_x) % tiles_y);
        const int64_t n = tile / ((int64_t)tiles_x * tiles_y);
        const int oy0 = ty * WT_TY, ox0 = tx * WT_TX;
        __syncthreads();                                                     // previous tile fully consumed
        for (int i = threadIdx.x; i < XR * XP; i += WT_THREADS) {
            const int r = i / XP, c = i - r * XP;
            const int iy = oy0 - 2 + r, ix = ox0 - 2 + c;
            const bool in = iy >= 0 && iy < g.h && ix >= 0 && ix < g.w;
            const float* src = x + ((n * sh + (in ? (UPS ? iy >> 1 : iy) : 0)) * (int64_t)sw + (in ? (UPS ? ix >> 1 : ix) : 0)) * 4;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(sx_addr + (uint32_t)i * 16u), "l"(src),
                         "r"(in ? 16 : 0) : "memory");
        }
        for (int i = threadIdx.x; i < WT_TY * WT_TX; i += WT_THREADS) {
            const int r = i / WT_TX, c = i - r * WT_TX;
            const int oy = oy0 + r, ox = ox0 + c;
            const bool in = oy < g.ho && ox < g.wo;
            const float* src = dy + ((n * g.ho + (in ? oy : 0)) * (int64_t)g.wo + (in ? ox : 0)) * COUT;
            if (COUT == 4)
                asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(sdy_addr + (uint32_t)i * 16u), "l"(src),
                             "r"(in ? 16 : 0) : "memory");
            else
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sdy_addr + (uint32_t)i * 8u), "l"(src),
                             "r"(in ? 8 : 0) : "memory");
        }
        asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        const int ky = warp;
#pragma unroll 2
        for (int r = 0; r < WT_TY; ++r) {
#pragma unroll
            for (int cg = 0; cg < WT_TX / 32; ++cg) {
                const int c = lane + 32 * cg;
                float d[COUT];
                if (COUT == 4) {
                    const float4 v = reinterpret_cast<const float4*>(s_dy)[r * WT_TX + c];
                    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
                } else {
                    const float2 v = reinterpret_cast<const float2*>(s_dy)[r * WT_TX + c];
                    d[0] = v.x; d[1] = v.y;
                }
                if (ky == 2) {                                               // warp-uniform: one warp also sums dy
#pragma unroll
                    for (int co = 0; co < COUT; ++co) dbacc[co] += d[co];
                }
                const float4* xrow = s_x + (r + ky) * XP + c;
#pragma unroll
                for (int kx = 0; kx < 5; ++kx) {
                    const float4 xv = xrow[kx];
                    const float xc[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
                    for (int ci = 0; ci < 4; ++ci)
#pragma unroll
                        for (int co = 0; co < COUT; ++co) acc[kx][ci][co] = fmaf(xc[ci], d[co], acc[kx][ci][co]);
                }
            }
        }
    }
    // warp reduction; element order of the finalize kernel: ((ky * 5 + kx) * 4 + ci) * COUT + co, then db[co]
    const int ky = warp;
#pragma unroll
    for (int kx = 0; kx < 5; ++kx)
#pragma unroll
        for (int ci = 0; ci < 4; ++ci)
#pragma unroll
            for (int co = 0; co < COUT; ++co) {
                const float t = warp_sum(acc[kx][ci][co]);
                if (lane == 0) ws[(int64_t)(((ky * 5 + kx) * 4 + ci) * COUT + co) * nblk + blockIdx.x] = t;
            }
    if (ky == 2) {
#pragma unroll
        for (int co = 0; co < COUT; ++co) {
            const float t = warp_sum(dbacc[co]);
            if (lane == 0) ws[(int64_t)(NACC + co) * nblk + blockIdx.x] = t;
        }
    }
    (void)NOUT;
}

static int wgrad_tiled_grid() { return 148 * 3; }

// one CTA per output element: sums its nblk partials and scatters into dw / db
__global__ void __launch_bounds__(256) conv_small_wgrad_finalize_kernel(
    const float* __restrict__ ws, int nblk, int kh, int kw, int cin, int civ, int cot, int cout, int bias,
    float* __restrict__ dw, float* __restrict__ db, int accumulate) {
    __shared__ float red[8];
    const int nacc = kh * kw * civ * cot, nout = nacc + cot;
    const int chunk = blockIdx.x / nout, e = blockIdx.x % nout;
    const int cochunks = cout / cot;
    const int cic = chunk / cochunks, coc = chunk % cochunks;
    const float* src = ws + (int64_t)blockIdx.x * nblk;
    float s = 0.f;
    for (int i = threadIdx.x; i < nblk; i += 256) s += src[i];
    s = block_sum(s, red);
    if (threadIdx.x != 0) return;
    if (e < nacc) {
        const int d = e % cot, c = (e / cot) % civ, tap = e / (cot * civ);
        float* dst = dw + ((int64_t)tap * cin + cic * civ + c) * cout + coc * cot + d;
        *dst = accumulate ? *dst + s : s;
    } else if (cic == 0) {
        float* dst = db + coc * cot + (e - nacc);
        const float v = bias ? s : 0.f;
        *dst = accumulate ? *dst + v : v;
    }
}

struct SmallWgradPlan {
    bool ok = false;
    int kh, kw, civ, cot, px, r;
};

static SmallWgradPlan plan_small_wgrad(const ConvGeom& g) {
    SmallWgradPlan p;
    auto set = [&](int civ, int cot, int px, int r) {
        p.ok = true; p.kh = g.kh; p.kw = g.kw; p.civ = civ; p.cot = cot; p.px = px; p.r = r;
    };
    const bool k33 = g.kh == 3 && g.kw == 3 && g.sh == 1 && g.sw == 1;
    const bool k55s1 = g.kh == 5 && g.kw == 5 && g.sh == 1 && g.sw == 1;
    const bool k55s2 = g.kh == 5 && g.kw == 5 && g.sh == 2 && g.sw == 2;
    const bool k53 = g.kh == 5 && g.kw == 3 && g.sh == 2 && g.sw == 1;
    if (k33 && g.cin == 1 && g.cout % 4 == 0) set(1, 4, 4, 16);
    else if (k33 && g.cin % 4 == 0 && g.cout == 1) set(4, 1, 4, 16);
    else if (k55s1 && g.cin == 1 && g.cout == 1) set(1, 1, 8, 16);
    else if (k55s2 && g.cin == 1 && g.cout == 1) set(1, 1, 4, 4);      // 4 rows per thread: 4x the CTAs of R = 16, the loop is latency-bound
    else if (k55s2 && g.cin == 1 && g.cout % 2 == 0) set(1, 2, 4, 2);      // Line down_1, down_2: two rows per thread --
    else if (k55s2 && g.cin == 4) set(4, 1, 4, 2);                         // 64 CTAs at R = 8 left most SMs idle (0.066 ms)
    else if (k55s1 && g.cin == 4) set(4, 1, 4, 8);
    else if (k53 && g.cin == 1 && g.cout % 4 == 0) set(1, 4, 4, 7);
    return p;
}

static void small_wgrad_dims(const ConvGeom& g, const SmallWgradPlan& p, int* nblk, int* chunks, int* nout) {
    const int strips = (g.wo + p.px - 1) / p.px, rgroups = (g.ho + p.r - 1) / p.r;
    *nblk = (int)ceil_div((int64_t)g.n * strips * rgroups, 256);
    *chunks = (g.cin / p.civ) * (g.cout / p.cot);
    *nout = p.kh * p.kw * p.civ * p.cot + p.cot;
}

static bool wgrad_tiled_ok(const ConvGeom& g) {
    return g.kh == 5 && g.kw == 5 && g.sh == 1 && g.sw == 1 && g.ph == 2 && g.pw == 2 && g.cin == 4 &&
           (g.cout == 4 || g.cout == 2) && g.padding_value == 0.f && (g.ups == 1 || g.ups == 2);
}

size_t conv_wgrad_fast_workspace(const ConvGeom& g, int) {
    const SmallWgradPlan p = plan_small_wgrad(g);
    size_t need = 0;
    if (p.ok) {
        int nblk, chunks, nout;
        small_wgrad_dims(g, p, &nblk, &chunks, &nout);
        need = sizeof(float) * (size_t)nblk * chunks * nout;
    }
    if (wgrad_tiled_ok(g)) {
        const size_t t = sizeof(float) * (size_t)wgrad_tiled_grid() * (25 * 4 * g.cout + g.cout);
        if (t > need) need = t;
    }
    return need;
}

template <int KH, int KW, int SH, int SW, int CIN, int CIV, int COT, int PX, int R>
static int launch_small_wgrad(const ConvGeom& g, const float* x, const float* dy, float* ws, int nblk, int chunks,
                              cudaStream_t st) {
    conv_small_wgrad_kernel<KH, KW, SH, SW, CIN, CIV, COT, PX, R><<<dim3(nblk, chunks), 256, 0, st>>>(g, x, dy, ws, nblk);
    UOCR_LAUNCHED("conv_small_wgrad");
    return UOCR_OK;
}

int conv_wgrad_fast(const ConvGeom& g, int math_mode, const float* x, const float* dy, float* dw, float* db,
                    int accumulate, float* ws, cudaStream_t st) {
    if (math_mode == UOCR_MATH_TF32 && g.ups == 1) {
        const int rc = conv_wgrad_tc(g, x, dy, dw, db, accumulate, st);
        if (rc != UOCR_ERR_UNSUPPORTED) return rc;
    }
    if (ws && wgrad_tiled_ok(g) && !((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy)) & 15)) {
        const int64_t ntiles = (int64_t)g.n * ceil_div(g.ho, WT_TY) * ceil_div(g.wo, WT_TX);
        const int nblk = (int)(ntiles < wgrad_tiled_grid() ? ntiles : wgrad_tiled_grid());
        const size_t smem = sizeof(float) * ((WT_TY + 4) * (WT_TX + 4) * 4 + WT_TY * WT_TX * g.cout);
        static bool configured = false;
        if (!configured) {
            cudaFuncSetAttribute(conv55_c4_wgrad_tiled_kernel<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
            cudaFuncSetAttribute(conv55_c4_wgrad_tiled_kernel<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
            cudaFuncSetAttribute(conv55_c4_wgrad_tiled_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
            cudaFuncSetAttribute(conv55_c4_wgrad_tiled_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
            configured = true;
        }
        if (g.cout == 4) {
            if (g.ups == 2) conv55_c4_wgrad_tiled_kernel<4, true><<<nblk, WT_THREADS, smem, st>>>(g, x, dy, ws, nblk);
            else conv55_c4_wgrad_tiled_kernel<4, false><<<nblk, WT_THREADS, smem, st>>>(g, x, dy, ws, nblk);
        } else {
            if (g.ups == 2) conv55_c4_wgrad_tiled_kernel<2, true><<<nblk, WT_THREADS, smem, st>>>(g, x, dy, ws, nblk);
            else conv55_c4_wgrad_tiled_kernel<2, false><<<nblk, WT_THREADS, smem, st>>>(g, x, dy, ws, nblk);
        }
        UOCR_LAUNCHED("conv55_c4_wgrad_tiled");
        const int nout = 25 * 4 * g.cout + g.cout;
        conv_small_wgrad_finalize_kernel<<<nout, 256, 0, st>>>(ws, nblk, 5, 5, 4, 4, g.cout, g.cout, g.bias, dw, db, accumulate);
        UOCR_LAUNCHED("conv_small_wgrad_finalize");
        return UOCR_OK;
    }
    const SmallWgradPlan p = plan_small_wgrad(g);
    if (!p.ok || !ws) return UOCR_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy)) & 15) return UOCR_ERR_UNSUPPORTED;
    int nblk, chunks, nout;
    small_wgrad_dims(g, p, &nblk, &chunks, &nout);
    if (chunks > 65535) return UOCR_ERR_UNSUPPORTED;
    const bool roll = g.kw == 5 && g.sh == 1 && g.cin == 1 && g.cout == 1 && g.w % 2 == 0 && g.wo % 4 == 0 &&
                      g.ph == 2 && g.pw == 2;
    if (g.ups != 1 && !roll) return UOCR_ERR_UNSUPPORTED;      // only the roll kernel reads an upsampled input
    int rc = UOCR_ERR_UNSUPPORTED;
    const bool k33 = g.kh == 3;
    if (k33 && g.cin == 1) rc = launch_small_wgrad<3, 3, 1, 1, 1, 1, 4, 4, 16>(g, x, dy, ws, nblk, chunks, st);
    else if (k33 && g.cin == 16) rc = launch_small_wgrad<3, 3, 1, 1, 16, 4, 1, 4, 16>(g, x, dy, ws, nblk, chunks, st);
    else if (k33 && g.cin == 4) rc = launch_small_wgrad<3, 3, 1, 1, 4, 4, 1, 4, 16>(g, x, dy, ws, nblk, chunks, st);
    else if (roll) {
        if (g.ups == 2) conv55_c1_wgrad_roll_kernel<16, true><<<dim3(nblk, chunks), 256, 0, st>>>(g, x, dy, ws, nblk);
        else conv55_c1_wgrad_roll_kernel<16, false><<<dim3(nblk, chunks), 256, 0, st>>>(g, x, dy, ws, nblk);   // plan: px 8, r 16
        UOCR_LAUNCHED("conv55_c1_wgrad_roll");
        rc = UOCR_OK;
    }
    else if (g.kw == 5 && g.sh == 1 && g.cin == 1) rc = launch_small_wgrad<5, 5, 1, 1, 1, 1, 1, 8, 16>(g, x, dy, ws, nblk, chunks, st);
    else if (g.kw == 5 && g.sh == 2 && g.cin == 1 && p.cot == 1) rc = launch_small_wgrad<5, 5, 2, 2, 1, 1, 1, 4, 4>(g, x, dy, ws, nblk, chunks, st);
    else if (g.kw == 5 && g.sh == 2 && g.cin == 1 && p.cot == 2) rc = launch_small_wgrad<5, 5, 2, 2, 1, 1, 2, 4, 2>(g, x, dy, ws, nblk, chunks, st);
    else if (g.kw == 5 && g.sh == 2 && g.cin == 4) rc = launch_small_wgrad<5, 5, 2, 2, 4, 4, 1, 4, 2>(g, x, dy, ws, nblk, chunks, st);
    else if (g.kw == 5 && g.sh == 1 && g.cin == 4) rc = launch_small_wgrad<5, 5, 1, 1, 4, 4, 1, 4, 8>(g, x, dy, ws, nblk, chunks, st);
    else if (g.kw == 3 && g.kh == 5 && g.cin == 1) rc = launch_small_wgrad<5, 3, 2, 1, 1, 1, 4, 4, 7>(g, x, dy, ws, nblk, chunks, st);
    if (rc) return rc;
    conv_small_wgrad_finalize_kernel<<<chunks * nout, 256, 0, st>>>(ws, nblk, p.kh, p.kw, g.cin, p.civ, p.cot, g.cout,
                                                                   g.bias, dw, db, accumulate);
    UOCR_LAUNCHED("conv_small_wgrad_finalize");
    return UOCR_OK;
}

// ------------------------------------------------------------------------------------------
// Fused backward of the 3x3 conv pair  x -(w1,b1)-> act1 -> h -(w2,b2)-> y   (1 -> C1 -> 1 channels,
// padding 1, stride 1; my_model's Monochrome net in training).  Layer by layer this needs the
// C1-channel hidden map four times (saved activation, its gradient, the activation mask, the
// pre-activation gradient: ~12 GB of traffic per 64 tiles at C1 = 16).  Here nothing C1-wide is
// ever stored: both kernels RECOMPUTE h from x (9 FMA per value) next to the gradient math.
//
//   pair_wgrad : thread = 8 hidden columns x 16 rows, channel loop OUTSIDE the row sweep so only
//                19 accumulators (dw1[9], db1, dw2[9]) are live; per hidden value 9 (h) + 9 (dh)
//                + 9 (dw2) + 9 (dw1) + 2 FMA; one CTA reduction per channel; partials to
//                workspace[(c, k)][cta], summed by a finalize kernel (deterministic)
//   pair_dgrad : dx = conv^T(w1, dpre), same row-streaming scheme as the forward pair kernel
//                (only launched when the caller wants the input gradient)
// ------------------------------------------------------------------------------------------
constexpr int PB_CW = 8, PB_R = 16, PB_THREADS = 128;

template <int CW, int R>
__global__ void __launch_bounds__(PB_THREADS, 4) conv3x3_pair_wgrad_kernel(
    const float* __restrict__ x, const float* __restrict__ w1, const float* __restrict__ b1,
    const float* __restrict__ w2, const float* __restrict__ dy, float* __restrict__ ws, int n_img, int H, int W,
    int C1, int act1, float alpha1, int nblk) {
    extern __shared__ __align__(16) float s_p[];             // per channel: w1[9], b1, w2[9], pad -> 20
    __shared__ float red[PB_THREADS / 32][20];
    for (int i = threadIdx.x; i < C1 * 20; i += PB_THREADS) {
        const int c = i / 20, k = i % 20;
        float v = 0.f;
        if (k < 9) v = w1[k * C1 + c];
        else if (k == 9) v = b1[c];
        else if (k < 19) v = w2[(k - 10) * C1 + c];
        s_p[i] = v;
    }
    __syncthreads();

    const int strips = (W + CW - 1) / CW, rchunks = (H + R - 1) / R;
    const int64_t idx = (int64_t)blockIdx.x * PB_THREADS + threadIdx.x;
    const int strip = (int)(idx % strips);
    const int rc = (int)((idx / strips) % rchunks);
    const int64_t n = idx / ((int64_t)strips * rchunks);
    const bool live = n < n_img;
    const int c0 = strip * CW, r0 = rc * R;
    const int r_end = min(r0 + R, H);
    const float* xim = x + (live ? n : 0) * (int64_t)H * W;
    const float* gim = dy + (live ? n : 0) * (int64_t)H * W;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;

    auto load_row = [&](const float* im, int row, float* dst) {
        const bool rin = live && row >= 0 && row < H;
#pragma unroll
        for (int j = 0; j < CW + 2; ++j) {
            const int col = c0 - 1 + j;
            dst[j] = (rin && col >= 0 && col < W) ? __ldg(im + (int64_t)row * W + col) : 0.f;
        }
    };

    for (int c = 0; c <= C1; ++c) {
        // c == C1: extra sweep-free slot for db2 (sum of dy over the owned pixels)
        float gw1[9], gw2[9], gb1 = 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) gw1[t] = gw2[t] = 0.f;
        if (c < C1) {
            const float4* pw = reinterpret_cast<const float4*>(s_p + c * 20);
            const float4 q0 = pw[0], q1 = pw[1], q2 = pw[2], q3 = pw[3], q4 = pw[4];
            const float k1[9] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x};
            const float bb = q2.y;
            const float k2[9] = {q2.z, q2.w, q3.x, q3.y, q3.z, q3.w, q4.x, q4.y, q4.z};
            float xw[3][CW + 2], gw[3][CW + 2];
            load_row(xim, r0 - 1, xw[0]); load_row(xim, r0, xw[1]);
            load_row(gim, r0 - 1, gw[0]); load_row(gim, r0, gw[1]);
            // rows in groups of 3 so that the 3-row windows are register RINGS with static slots
            // (slot = (row - (r0 - 1)) % 3) instead of being shifted after every row (40 MOV per row)
            for (int hb = r0; hb < r_end; hb += 3) {
#pragma unroll
                for (int u = 0; u < 3; ++u) {
                    const int hr = hb + u;
                    if (hr < r_end) {                                   // thread-uniform
                        load_row(xim, hr + 1, xw[(u + 2) % 3]);
                        load_row(gim, hr + 1, gw[(u + 2) % 3]);
#pragma unroll
                        for (int j = 0; j < CW; ++j) {
                            if (c0 + j < W) {
                                float hp = bb, dh = 0.f;
#pragma unroll
                                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                                    for (int kx = 0; kx < 3; ++kx) {
                                        hp = fmaf(k1[ky * 3 + kx], xw[(u + ky) % 3][j + kx], hp);
                                        dh = fmaf(k2[ky * 3 + kx], gw[(u + 2 - ky) % 3][j + 2 - kx], dh);
                                    }
                                float hval = hp, mask = 1.f;
                                if (act1 == UOCR_ACT_LEAKY && hp < 0.f) { hval = alpha1 * hp; mask = alpha1; }
                                const float dpre = dh * mask;
                                gb1 += dpre;
#pragma unroll
                                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                                    for (int kx = 0; kx < 3; ++kx) {
                                        gw1[ky * 3 + kx] = fmaf(dpre, xw[(u + ky) % 3][j + kx], gw1[ky * 3 + kx]);
                                        gw2[ky * 3 + kx] = fmaf(gw[(u + 2 - ky) % 3][j + 2 - kx], hval, gw2[ky * 3 + kx]);
                                    }
                            }
                        }
                    }
                }
            }
        } else {
            for (int hr = r0; hr < r_end; ++hr) {
                float row[CW + 2];
                load_row(gim, hr, row);
#pragma unroll
                for (int j = 0; j < CW; ++j) gb1 += row[j + 1];       // col c0 + j (beyond W reads as 0)
            }
        }
        // ---- CTA reduction of the 19 sums of this channel
        __syncthreads();
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const float a = warp_sum(gw1[t]), b = warp_sum(gw2[t]);
            if (lane == 0) { red[wid][t] = a; red[wid][10 + t] = b; }
        }
        {
            const float a = warp_sum(gb1);
            if (lane == 0) red[wid][9] = a;
        }
        __syncthreads();
        if (threadIdx.x < 19) {
            float s = 0.f;
#pragma unroll
            for (int k = 0; k < PB_THREADS / 32; ++k) s += red[k][threadIdx.x];
            ws[((int64_t)c * 19 + threadIdx.x) * nblk + blockIdx.x] = s;
        }
    }
}

// element e = c * 19 + k: k < 9 -> dw1[k][c]; k == 9 -> db1[c] (c == C1: db2); k >= 10 -> dw2[k-10][c]
__global__ void __launch_bounds__(256) conv3x3_pair_wgrad_finalize_kernel(const float* __restrict__ ws, int nblk,
                                                                          int C1, float* dw1, float* db1, float* dw2,
                                                                          float* db2, int accumulate) {
    __shared__ float red[8];
    const int c = blockIdx.x / 19, k = blockIdx.x % 19;
    const float* src = ws + (int64_t)blockIdx.x * nblk;
    float s = 0.f;
    for (int i = threadIdx.x; i < nblk; i += 256) s += src[i];
    s = block_sum(s, red);
    if (threadIdx.x != 0) return;
    float* dst = nullptr;
    if (c == C1) { if (k == 9) dst = db2; }
    else if (k < 9) dst = dw1 + k * C1 + c;
    else if (k == 9) dst = db1 + c;
    else dst = dw2 + (k - 10) * C1 + c;
    if (dst) *dst = accumulate ? *dst + s : s;
}

template <int CW, int R>
__global__ void __launch_bounds__(PB_THREADS) conv3x3_pair_dgrad_kernel(
    const float* __restrict__ x, const float* __restrict__ w1, const float* __restrict__ b1,
    const float* __restrict__ w2, const float* __restrict__ dy, float* __restrict__ dx, int n_img, int H, int W,
    int C1, int act1, float alpha1) {
    extern __shared__ __align__(16) float s_p[];
    for (int i = threadIdx.x; i < C1 * 20; i += PB_THREADS) {
        const int c = i / 20, k = i % 20;
        float v = 0.f;
        if (k < 9) v = w1[k * C1 + c];
        else if (k == 9) v = b1[c];
        else if (k < 19) v = w2[(k - 10) * C1 + c];
        s_p[i] = v;
    }
    __syncthreads();
    const int strips = (W + CW - 1) / CW, rchunks = (H + R - 1) / R;
    const int64_t idx = (int64_t)blockIdx.x * PB_THREADS + threadIdx.x;
    const int strip = (int)(idx % strips);
    const int rc = (int)((idx / strips) % rchunks);
    const int64_t n = idx / ((int64_t)strips * rchunks);
    if (n >= n_img) return;
    const int c0 = strip * CW, r0 = rc * R;
    const int r_end = min(r0 + R, H);
    const float* xim = x + n * (int64_t)H * W;
    const float* gim = dy + n * (int64_t)H * W;
    float* dim = dx + n * (int64_t)H * W;

    // windows cover hidden columns c0-1 .. c0+CW (CW + 2) and their 3x3 neighbourhoods (CW + 4)
    float xw[3][CW + 4], gw[3][CW + 4];
    float accA[CW], accB[CW], accC[CW];                      // dx rows hr-1, hr, hr+1
#pragma unroll
    for (int j = 0; j < CW; ++j) accA[j] = accB[j] = accC[j] = 0.f;
    auto load_row = [&](const float* im, int row, float* dst) {
        const bool rin = row >= 0 && row < H;
#pragma unroll
        for (int j = 0; j < CW + 4; ++j) {
            const int col = c0 - 2 + j;
            dst[j] = (rin && col >= 0 && col < W) ? __ldg(im + (int64_t)row * W + col) : 0.f;
        }
    };
    load_row(xim, r0 - 2, xw[0]); load_row(xim, r0 - 1, xw[1]);
    load_row(gim, r0 - 2, gw[0]); load_row(gim, r0 - 1, gw[1]);
    for (int hr = r0 - 1; hr <= r_end; ++hr) {
        load_row(xim, hr + 1, xw[2]);
        load_row(gim, hr + 1, gw[2]);
        if (hr >= 0 && hr < H) {
            for (int c = 0; c < C1; ++c) {
                const float4* pw = reinterpret_cast<const float4*>(s_p + c * 20);
                const float4 q0 = pw[0], q1 = pw[1], q2 = pw[2], q3 = pw[3], q4 = pw[4];
                const float k1[9] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x};
                const float bb = q2.y;
                const float k2[9] = {q2.z, q2.w, q3.x, q3.y, q3.z, q3.w, q4.x, q4.y, q4.z};
                float dp[CW + 2];
#pragma unroll
                for (int j = 0; j < CW + 2; ++j) {
                    float hp = bb, dh = 0.f;
#pragma unroll
                    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx) {
                            hp = fmaf(k1[ky * 3 + kx], xw[ky][j + kx], hp);
                            dh = fmaf(k2[ky * 3 + kx], gw[2 - ky][j + 2 - kx], dh);
                        }
                    const float mask = (act1 == UOCR_ACT_LEAKY && hp < 0.f) ? alpha1 : 1.f;
                    const int col = c0 - 1 + j;
                    dp[j] = (col >= 0 && col < W) ? dh * mask : 0.f;      // hidden pixel outside the image
                }
#pragma unroll
                for (int j = 0; j < CW; ++j) {
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        // hidden (hr, col) feeds dx(hr + ky - 1, col + kx - 1)
                        accA[j] = fmaf(k1[kx], dp[j + 2 - kx], accA[j]);          // ky = 0 -> row hr - 1
                        accB[j] = fmaf(k1[3 + kx], dp[j + 2 - kx], accB[j]);      // ky = 1 -> row hr
                        accC[j] = fmaf(k1[6 + kx], dp[j + 2 - kx], accC[j]);      // ky = 2 -> row hr + 1
                    }
                }
            }
        }
        const int orow = hr - 1;
        if (orow >= r0 && orow < r_end) {
            float* op = dim + (int64_t)orow * W + c0;
#pragma unroll
            for (int j = 0; j < CW; ++j)
                if (c0 + j < W) op[j] = accA[j];
        }
#pragma unroll
        for (int j = 0; j < CW; ++j) { accA[j] = accB[j]; accB[j] = accC[j]; accC[j] = 0.f; }
#pragma unroll
        for (int j = 0; j < CW + 4; ++j) {
            xw[0][j] = xw[1][j]; xw[1][j] = xw[2][j];
            gw[0][j] = gw[1][j]; gw[1][j] = gw[2][j];
        }
    }
}

size_t conv3x3_pair_bwd_workspace(int64_t n, int64_t h, int64_t w, int c1) {
    const int64_t nblk = ceil_div(n * ceil_div(w, PB_CW) * ceil_div(h, PB_R), PB_THREADS);
    const size_t cuda_cores = sizeof(float) * (size_t)nblk * (c1 + 1) * 19;
    const size_t tc = c1 == 16 ? conv3x3_pair_wgrad_tc_workspace(n, h, w, c1) : 0;
    return cuda_cores > tc ? cuda_cores : tc;
}

int conv3x3_pair_bwd(const float* x, const float* w1, const float* b1, const float* w2, const float* dy, float* dx,
                     float* dw1, float* db1, float* dw2, float* db2, int64_t n, int64_t h, int64_t w, int c1,
                     int act1, float alpha1, int accumulate, float* ws, cudaStream_t st, int math_mode) {
    const int64_t items = n * ceil_div(w, PB_CW) * ceil_div(h, PB_R);
    const int64_t nblk = ceil_div(items, PB_THREADS);
    if (nblk > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    const size_t smem = sizeof(float) * 20 * c1;
    // TF32 mode: tensor-core assisted weight gradients (conv_pair_bwd_tc.cu) where they have a kernel; same workspace
    // layout, same finalize
    int wgrad_nblk = 0;
    if (!(math_mode == UOCR_MATH_TF32 &&
          conv3x3_pair_wgrad_tc(x, w1, b1, w2, dy, ws, n, h, w, c1, act1, alpha1, &wgrad_nblk, st) == UOCR_OK)) {
        conv3x3_pair_wgrad_kernel<PB_CW, PB_R><<<(unsigned)nblk, PB_THREADS, smem, st>>>(
            x, w1, b1, w2, dy, ws, (int)n, (int)h, (int)w, c1, act1, alpha1, (int)nblk);
        UOCR_LAUNCHED("conv3x3_pair_wgrad");
        wgrad_nblk = (int)nblk;
    }
    conv3x3_pair_wgrad_finalize_kernel<<<(c1 + 1) * 19, 256, 0, st>>>(ws, wgrad_nblk, c1, dw1, db1, dw2, db2, accumulate);
    UOCR_LAUNCHED("conv3x3_pair_wgrad_finalize");
    if (dx) {
        conv3x3_pair_dgrad_kernel<PB_CW, PB_R><<<(unsigned)nblk, PB_THREADS, smem, st>>>(
            x, w1, b1, w2, dy, dx, (int)n, (int)h, (int)w, c1, act1, alpha1);
        UOCR_LAUNCHED("conv3x3_pair_dgrad");
    }
    return UOCR_OK;
}

}  // namespace uocr

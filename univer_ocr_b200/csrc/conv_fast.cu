// Shape-specialised convolution kernels for the my_model geometries (SURVEY.md 8a, row a1).
//
// All of my_model's convolutions except Char conv_2/conv_3 have tiny channel counts
// (1->16, 16->1, 1->1, 1->4, 4->4, 4->2, 1->64): their arithmetic intensity is far below the
// tensor-core ridge, so they are CUDA-core stencils bound by HBM / FFMA issue, not GEMMs.
// Design (forward): one thread = PX consecutive output pixels x COT output channels in
// registers; the input window row (PX*SW + KW - SW pixels, 128-bit loads over channels) is
// fetched once per kernel row through L1 and reused for every tap / output channel; weights are
// staged in shared memory once per CTA and read as warp-broadcast 128-bit loads; bias +
// activation are applied in the epilogue; an optional x2 nearest-neighbour upsample of the
// input is folded into the address computation (Upsample2D + Convolutional2D in one pass).
#include "conv_common.cuh"

namespace uocr {

template <int CIV> struct XVec;
template <> struct XVec<1> {
    float v[1];
    __device__ __forceinline__ void load(const float* p) { v[0] = __ldg(p); }
    __device__ __forceinline__ void fill(float f) { v[0] = f; }
};
template <> struct XVec<4> {
    float v[4];
    __device__ __forceinline__ void load(const float* p) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void fill(float f) { v[0] = v[1] = v[2] = v[3] = f; }
};

template <int KH, int KW, int SH, int SW, int CIN, int COT, int PX, int UPS>
__global__ void __launch_bounds__(256) conv_small_fwd_kernel(ConvGeom g, const float* __restrict__ x,
                                                             const float* __restrict__ w,
                                                             const float* __restrict__ b,
                                                             float* __restrict__ y, int act, float alpha) {
    constexpr int CIV = (CIN % 4 == 0) ? 4 : 1;
    constexpr int NIN = (PX - 1) * SW + KW;
    extern __shared__ __align__(16) float s_w[];            // [KH][KW][CIN][cout]
    const int cout = g.cout;
    for (int i = threadIdx.x; i < KH * KW * CIN * cout; i += 256) s_w[i] = w[i];
    __syncthreads();

    const int chunks = cout / COT;
    const int strips = (g.wo + PX - 1) / PX;
    const int64_t idx = (int64_t)blockIdx.x * 256 + threadIdx.x;
    const int chunk = (int)(idx % chunks);
    const int64_t s = idx / chunks;
    const int xs = (int)(s % strips);
    const int oy = (int)((s / strips) % g.ho);
    const int64_t n = s / ((int64_t)strips * g.ho);
    if (n >= g.n) return;
    const int co0 = chunk * COT;
    const int ox0 = xs * PX;
    const int iy0 = oy * SH - g.ph, ix0 = ox0 * SW - g.pw;
    const int hp = g.h / UPS, wp = g.w / UPS;               // physical input size

    float acc[PX][COT];
#pragma unroll
    for (int p = 0; p < PX; ++p)
#pragma unroll
        for (int c = 0; c < COT; ++c) acc[p][c] = 0.f;

#pragma unroll
    for (int ky = 0; ky < KH; ++ky) {
        const int iy = iy0 + ky;
        const bool yin = iy >= 0 && iy < g.h;
        const float* xrow = x + ((n * hp + (yin ? iy / UPS : 0)) * (int64_t)wp) * CIN;
#pragma unroll
        for (int cg = 0; cg < CIN / CIV; ++cg) {
            XVec<CIV> xin[NIN];
#pragma unroll
            for (int j = 0; j < NIN; ++j) {
                const int ix = ix0 + j;
                if (yin && ix >= 0 && ix < g.w) xin[j].load(xrow + (int64_t)(ix / UPS) * CIN + cg * CIV);
                else xin[j].fill(g.padding_value);
            }
#pragma unroll
            for (int kx = 0; kx < KW; ++kx) {
#pragma unroll
                for (int v = 0; v < CIV; ++v) {
                    const float* wp_ = s_w + ((ky * KW + kx) * CIN + cg * CIV + v) * cout + co0;
                    float wr[COT];
                    if (COT % 4 == 0) {
#pragma unroll
                        for (int c = 0; c < COT; c += 4) {
                            const float4 t = *reinterpret_cast<const float4*>(wp_ + c);
                            wr[c] = t.x; wr[c + 1] = t.y; wr[c + 2] = t.z; wr[c + 3] = t.w;
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < COT; ++c) wr[c] = wp_[c];
                    }
#pragma unroll
                    for (int p = 0; p < PX; ++p) {
                        const float xv = xin[p * SW + kx].v[v];
#pragma unroll
                        for (int c = 0; c < COT; ++c) acc[p][c] = fmaf(xv, wr[c], acc[p][c]);
                    }
                }
            }
        }
    }

    float bias[COT];
#pragma unroll
    for (int c = 0; c < COT; ++c) bias[c] = g.bias ? __ldg(b + co0 + c) : 0.f;
    float* yrow = y + ((n * g.ho + oy) * (int64_t)g.wo + ox0) * cout + co0;
    if (COT == 1 && cout == 1 && PX % 4 == 0 && (g.wo & 3) == 0 && ox0 + PX <= g.wo) {
#pragma unroll
        for (int p = 0; p < PX; p += 4) {
            float4 t;
            t.x = apply_act_fast(acc[p][0] + bias[0], act, alpha);
            t.y = apply_act_fast(acc[p + 1][0] + bias[0], act, alpha);
            t.z = apply_act_fast(acc[p + 2][0] + bias[0], act, alpha);
            t.w = apply_act_fast(acc[p + 3][0] + bias[0], act, alpha);
            *reinterpret_cast<float4*>(yrow + p) = t;
        }
        return;
    }
#pragma unroll
    for (int p = 0; p < PX; ++p) {
        if (ox0 + p >= g.wo) break;
        float* yp = yrow + (int64_t)p * cout;
        if (COT % 4 == 0) {
#pragma unroll
            for (int c = 0; c < COT; c += 4) {
                float4 t;
                t.x = apply_act_fast(acc[p][c] + bias[c], act, alpha);
                t.y = apply_act_fast(acc[p][c + 1] + bias[c + 1], act, alpha);
                t.z = apply_act_fast(acc[p][c + 2] + bias[c + 2], act, alpha);
                t.w = apply_act_fast(acc[p][c + 3] + bias[c + 3], act, alpha);
                *reinterpret_cast<float4*>(yp + c) = t;
            }
        } else {
#pragma unroll
            for (int c = 0; c < COT; ++c) yp[c] = apply_act_fast(acc[p][c] + bias[c], act, alpha);
        }
    }
}

template <int KH, int KW, int SH, int SW, int CIN, int COT, int PX>
static int launch_small_fwd(const ConvGeom& g, int ups, const float* x, const float* w, const float* b,
                            float* y, int act, float alpha, cudaStream_t st) {
    const int chunks = g.cout / COT;
    const int strips = (g.wo + PX - 1) / PX;
    const int64_t items = (int64_t)g.n * g.ho * strips * chunks;
    const int64_t blocks = ceil_div(items, 256);
    const size_t smem = sizeof(float) * KH * KW * CIN * g.cout;
    if (blocks > 0x7fffffff || smem > 48 * 1024) return UOCR_ERR_UNSUPPORTED;
    if (ups == 2)
        conv_small_fwd_kernel<KH, KW, SH, SW, CIN, COT, PX, 2><<<(unsigned)blocks, 256, smem, st>>>(
            g, x, w, b, y, act, alpha);
    else
        conv_small_fwd_kernel<KH, KW, SH, SW, CIN, COT, PX, 1><<<(unsigned)blocks, 256, smem, st>>>(
            g, x, w, b, y, act, alpha);
    UOCR_LAUNCHED("conv_small_fwd");
    return UOCR_OK;
}

// ------------------------------------------------------------------------------------------
// Cin == 1 forward stencil with a shared-memory input tile (Paragraph's five 5x5 1->1 layers,
// Monochrome conv_1, Line down_1, Char conv_1).  These layers move 4-8 bytes per 25-50 FMA and are
// HBM-bound; the register-strip kernel above reaches them through strided per-thread L1 loads
// (8 cache lines per warp load).  Here the CTA stages the (TH*SH + KH - SH) x (TW*SW + KW - SW)
// input tile with fully coalesced loads (border = padding_value, optional x2 upsample folded into
// the tile fill), then every thread reads its window as aligned 128-bit shared loads:
// warp = one output row of the tile, lane = PX consecutive outputs.
// ------------------------------------------------------------------------------------------
template <int KH, int KW, int SH, int SW, int COT, int PX, int UPS, int TH>
__global__ void __launch_bounds__(256) conv_c1_fwd_kernel(ConvGeom g, const float* __restrict__ x,
                                                          const float* __restrict__ w,
                                                          const float* __restrict__ b, float* __restrict__ y,
                                                          int act, float alpha) {
    constexpr int TW = 32 * PX;
    constexpr int IH = (TH - 1) * SH + KH;
    constexpr int NIN = (PX - 1) * SW + KW;
    constexpr int NV = (NIN + 3) / 4;                        // float4 loads per window row
    constexpr int IWP = (((TW - 1) * SW + KW) + 3 + 4) / 4 * 4;   // pitch: whole float4s past the last window
    extern __shared__ __align__(16) float s_mem[];
    float* s_in = s_mem;                                     // [IH][IWP]
    float* s_w = s_mem + IH * IWP;                           // [KH*KW][cout]
    const int cout = g.cout;
    const int chunks = cout / COT;
    const int n = blockIdx.z / chunks, chunk = blockIdx.z % chunks;
    const int co0 = chunk * COT;
    const int oy0 = blockIdx.y * TH, ox0 = blockIdx.x * TW;
    const int iy0 = oy0 * SH - g.ph, ix0 = ox0 * SW - g.pw;
    const int hp = g.h / UPS, wp = g.w / UPS;
    const float* xim = x + (int64_t)n * hp * wp;

    for (int i = threadIdx.x; i < KH * KW * cout; i += 256) s_w[i] = w[i];
    // asynchronous tile fill (LDGSTS): every in-bounds element is one 4-byte cp.async, so a thread
    // has all of its ~19 loads in flight at once instead of a load -> store dependency per element
    int fr = threadIdx.x / IWP, fc = threadIdx.x - fr * IWP;
    for (int i = threadIdx.x; i < IH * IWP; i += 256, fr += 256 / IWP, fc += 256 % IWP) {
        if (fc >= IWP) { fc -= IWP; ++fr; }
        const int iy = iy0 + fr, ix = ix0 + fc;
        if (iy >= 0 && iy < g.h && ix >= 0 && ix < g.w) {
            const float* src = xim + (int64_t)(iy / UPS) * wp + ix / UPS;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;"
                         ::"r"((uint32_t)__cvta_generic_to_shared(s_in + i)), "l"(src) : "memory");
        } else {
            s_in[i] = g.padding_value;
        }
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();

    const int lane = threadIdx.x & 31;
    const int oxl = ox0 + lane * PX;
    if (oxl >= g.wo) return;
    float bias[COT];
#pragma unroll
    for (int c = 0; c < COT; ++c) bias[c] = g.bias ? __ldg(b + co0 + c) : 0.f;

    float wreg[COT == 1 ? KH * KW : 1];                      // single-output-channel weights live in registers
    if (COT == 1) {
#pragma unroll
        for (int t = 0; t < KH * KW; ++t) wreg[t] = s_w[t * cout + co0];
    }
    // each warp walks rows ty, ty + 8, ... of the tile (a tall tile keeps ~20 KB of loads in flight
    // per CTA and cuts the halo re-read to (TH*SH + KH - SH) / (TH*SH))
    for (int ty = threadIdx.x >> 5; ty < TH; ty += 8) {
        const int oy = oy0 + ty;
        if (oy >= g.ho) break;
        float acc[PX][COT];
#pragma unroll
        for (int p = 0; p < PX; ++p)
#pragma unroll
            for (int c = 0; c < COT; ++c) acc[p][c] = 0.f;

#pragma unroll
        for (int ky = 0; ky < KH; ++ky) {
            const float4* row = reinterpret_cast<const float4*>(s_in + (ty * SH + ky) * IWP + lane * PX * SW);
            float xin[NV * 4];
#pragma unroll
            for (int v = 0; v < NV; ++v) {
                const float4 t = row[v];
                xin[4 * v] = t.x; xin[4 * v + 1] = t.y; xin[4 * v + 2] = t.z; xin[4 * v + 3] = t.w;
            }
#pragma unroll
            for (int kx = 0; kx < KW; ++kx) {
                const float* wp_ = s_w + (ky * KW + kx) * cout + co0;
                float wr[COT];
                if (COT == 1) {
                    wr[0] = wreg[ky * KW + kx];
                } else if (COT % 4 == 0) {
#pragma unroll
                    for (int c = 0; c < COT; c += 4) {
                        const float4 t = *reinterpret_cast<const float4*>(wp_ + c);
                        wr[c] = t.x; wr[c + 1] = t.y; wr[c + 2] = t.z; wr[c + 3] = t.w;
                    }
                } else {
#pragma unroll
                    for (int c = 0; c < COT; ++c) wr[c] = wp_[c];
                }
#pragma unroll
                for (int p = 0; p < PX; ++p)
#pragma unroll
                    for (int c = 0; c < COT; ++c) acc[p][c] = fmaf(xin[p * SW + kx], wr[c], acc[p][c]);
            }
        }

        float* yrow = y + (((int64_t)n * g.ho + oy) * g.wo + oxl) * cout + co0;
        if (COT == 1 && cout == 1 && PX == 4 && (g.wo & 3) == 0) {
            float4 t;
            t.x = apply_act_fast(acc[0][0] + bias[0], act, alpha);
            t.y = apply_act_fast(acc[1][0] + bias[0], act, alpha);
            t.z = apply_act_fast(acc[2][0] + bias[0], act, alpha);
            t.w = apply_act_fast(acc[3][0] + bias[0], act, alpha);
            *reinterpret_cast<float4*>(yrow) = t;
            continue;
        }
#pragma unroll
        for (int p = 0; p < PX; ++p) {
            if (oxl + p >= g.wo) break;
            float* yp = yrow + (int64_t)p * cout;
            if (COT % 4 == 0) {
#pragma unroll
                for (int c = 0; c < COT; c += 4) {
                    float4 t;
                    t.x = apply_act_fast(acc[p][c] + bias[c], act, alpha);
                    t.y = apply_act_fast(acc[p][c + 1] + bias[c + 1], act, alpha);
                    t.z = apply_act_fast(acc[p][c + 2] + bias[c + 2], act, alpha);
                    t.w = apply_act_fast(acc[p][c + 3] + bias[c + 3], act, alpha);
                    *reinterpret_cast<float4*>(yp + c) = t;
                }
            } else {
#pragma unroll
                for (int c = 0; c < COT; ++c) yp[c] = apply_act_fast(acc[p][c] + bias[c], act, alpha);
            }
        }
    }
}

template <int KH, int KW, int SH, int SW, int COT, int PX>
static int launch_c1_fwd(const ConvGeom& g, int ups, const float* x, const float* w, const float* b, float* y,
                         int act, float alpha, cudaStream_t st) {
    // tall tiles for big images (stride-1: 32 rows, 19.6 KB of input per CTA; stride-2: 16 rows, 37 KB)
    constexpr int TH = (SH == 1) ? 32 : 16;
    constexpr int TW = 32 * PX;
    constexpr int IH = (TH - 1) * SH + KH;
    constexpr int IWP = (((TW - 1) * SW + KW) + 3 + 4) / 4 * 4;
    const size_t smem = sizeof(float) * (IH * IWP + KH * KW * g.cout);
    const int64_t gz = (int64_t)g.n * (g.cout / COT);
    if (smem > 48 * 1024 || gz > 65535 || ceil_div(g.ho, TH) > 65535) return UOCR_ERR_UNSUPPORTED;
    dim3 grid((unsigned)ceil_div(g.wo, TW), (unsigned)ceil_div(g.ho, TH), (unsigned)gz);
    if (ups == 2)
        conv_c1_fwd_kernel<KH, KW, SH, SW, COT, PX, 2, TH><<<grid, 256, smem, st>>>(g, x, w, b, y, act, alpha);
    else
        conv_c1_fwd_kernel<KH, KW, SH, SW, COT, PX, 1, TH><<<grid, 256, smem, st>>>(g, x, w, b, y, act, alpha);
    UOCR_LAUNCHED("conv_c1_fwd");
    return UOCR_OK;
}

// ------------------------------------------------------------------------------------------
// 5 x 5 / stride 1 / padding 2 / 1 -> 1 channel (Paragraph up_*, end in training; their stride-1 dgrads on flipped
// weights): the two levels of the fused hourglass kernel (hourglass.cu) as stand-alone layers.
//   conv55_c1_tile_kernel     : 32 x 128 output block, its 36 x 136 input block staged with 16-byte cp.async (zero fill =
//                               padding), thread = 2 rows x 4 columns from conflict-free 128-bit shared loads
//   conv55_c1_ups_tile_kernel : the same convolution over a x2 nearest-upsampled input that is never materialised: four
//                               parity-specific 3 x 3 kernels with pre-summed weights on the low-resolution block (9 FMA
//                               per output instead of 25)
// Both need W % 4 == 0 (W % 8 for the upsampled one), zero padding and 16-byte aligned tensors; otherwise the generic
// Cin = 1 kernel above runs.
// ------------------------------------------------------------------------------------------
constexpr int C55_TH = 32, C55_TW = 128, C55_P = 136;

__global__ void __launch_bounds__(256) conv55_c1_tile_kernel(ConvGeom g, const float* __restrict__ x,
                                                             const float* __restrict__ w, const float* __restrict__ b,
                                                             float* __restrict__ y, int act, float alpha) {
    __shared__ __align__(16) float s_in[(C55_TH + 4) * C55_P];          // origin (oy0 - 2, ox0 - 4)
    const int ox0 = blockIdx.x * C55_TW, oy0 = blockIdx.y * C55_TH;
    const float* xim = x + (int64_t)blockIdx.z * g.h * g.w;
    float* yim = y + (int64_t)blockIdx.z * g.h * g.w;
    const uint32_t sbase = static_cast<uint32_t>(__cvta_generic_to_shared(s_in));
    for (int i = threadIdx.x; i < (C55_TH + 4) * (C55_P / 4); i += 256) {
        const int r = i / (C55_P / 4), q = i - r * (C55_P / 4);
        const int gy = oy0 - 2 + r, gx = ox0 - 4 + 4 * q;
        const bool in = (unsigned)gy < (unsigned)g.h && (unsigned)gx < (unsigned)g.w;
        const float* src = in ? xim + (int64_t)gy * g.w + gx : xim;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                     ::"r"(sbase + (uint32_t)(r * C55_P + 4 * q) * 4u), "l"(src), "r"(in ? 16 : 0) : "memory");
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    float wr[25];
#pragma unroll
    for (int i = 0; i < 25; ++i) wr[i] = __ldg(w + i);
    const float bias = g.bias ? __ldg(b) : 0.f;
    __syncthreads();
    for (int item = threadIdx.x; item < (C55_TH / 2) * (C55_TW / 4); item += 256) {
        const int r = (item / (C55_TW / 4)) * 2, c0 = (item % (C55_TW / 4)) * 4;
        float acc[2][4];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[0][j] = acc[1][j] = bias;
#pragma unroll
        for (int rr = 0; rr < 6; ++rr) {
            const float4* row = reinterpret_cast<const float4*>(s_in + (r + rr) * C55_P + c0);
            const float4 u = row[0], v = row[1], t = row[2];
            const float in[8] = {u.z, u.w, v.x, v.y, v.z, v.w, t.x, t.y};        // block columns c0 + 2 .. c0 + 9
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int ky = rr - k;
                if (ky >= 0 && ky < 5) {
#pragma unroll
                    for (int kx = 0; kx < 5; ++kx)
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc[k][j] = fmaf(wr[ky * 5 + kx], in[j + kx], acc[k][j]);
                }
            }
        }
        const int gx = ox0 + c0;
        if (gx < g.w) {
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int gy = oy0 + r + k;
                if (gy < g.h)
                    *reinterpret_cast<float4*>(yim + (int64_t)gy * g.w + gx) =
                        make_float4(apply_act_fast(acc[k][0], act, alpha), apply_act_fast(acc[k][1], act, alpha),
                                    apply_act_fast(acc[k][2], act, alpha), apply_act_fast(acc[k][3], act, alpha));
            }
        }
    }
}

__global__ void __launch_bounds__(256) conv55_c1_ups_tile_kernel(ConvGeom g, const float* __restrict__ x,
                                                                 const float* __restrict__ w, const float* __restrict__ b,
                                                                 float* __restrict__ y, int act, float alpha) {
    constexpr int SH_ = C55_TH / 2 + 2, SP_ = 72;           // low-resolution block: origin (oy0/2 - 1, ox0/2 - 4)
    __shared__ __align__(16) float s_in[SH_ * SP_];
    __shared__ float s_f[36];
    const int ox0 = blockIdx.x * C55_TW, oy0 = blockIdx.y * C55_TH;
    const int hs = g.h / 2, ws = g.w / 2;                   // stored (low-resolution) size
    const float* xim = x + (int64_t)blockIdx.z * hs * ws;
    float* yim = y + (int64_t)blockIdx.z * g.h * g.w;
    const uint32_t sbase = static_cast<uint32_t>(__cvta_generic_to_shared(s_in));
    for (int i = threadIdx.x; i < SH_ * (SP_ / 4); i += 256) {
        const int r = i / (SP_ / 4), q = i - r * (SP_ / 4);
        const int gy = oy0 / 2 - 1 + r, gx = ox0 / 2 - 4 + 4 * q;
        const bool in = (unsigned)gy < (unsigned)hs && (unsigned)gx < (unsigned)ws;
        const float* src = in ? xim + (int64_t)gy * ws + gx : xim;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;"
                     ::"r"(sbase + (uint32_t)(r * SP_ + 4 * q) * 4u), "l"(src), "r"(in ? 16 : 0) : "memory");
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    if (threadIdx.x < 36) {                                 // parity-folded 3 x 3 kernels (see hourglass.cu)
        const int i = threadIdx.x, bb = i % 3, a = (i / 3) % 3, px = (i / 9) % 2, py = i / 18;
        const int ylo = py == 0 ? 2 * a : (a == 0 ? 0 : 2 * a - 1), yhi = py == 0 ? min(2 * a + 1, 4) : (a == 0 ? 0 : 2 * a);
        const int xlo = px == 0 ? 2 * bb : (bb == 0 ? 0 : 2 * bb - 1), xhi = px == 0 ? min(2 * bb + 1, 4) : (bb == 0 ? 0 : 2 * bb);
        float t = 0.f;
        for (int ky = ylo; ky <= yhi; ++ky)
            for (int kx = xlo; kx <= xhi; ++kx) t += __ldg(w + ky * 5 + kx);
        s_f[i] = t;
    }
    const float bias = g.bias ? __ldg(b) : 0.f;
    __syncthreads();
    float wf[36];
#pragma unroll
    for (int i = 0; i < 36; ++i) wf[i] = s_f[i];
    // item = source row j (output rows 2j, 2j + 1) x 2 source cells n0, n0 + 1 (output columns 2 n0 .. 2 n0 + 3)
    for (int item = threadIdx.x; item < (C55_TH / 2) * (C55_TW / 4); item += 256) {
        const int j = item / (C55_TW / 4), n0 = (item % (C55_TW / 4)) * 2;
        float sv[3][4];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float* row = s_in + (j + a) * SP_ + n0 + 3;                   // block column of source column n0 - 1
#pragma unroll
            for (int q = 0; q < 4; ++q) sv[a][q] = row[q];
        }
#pragma unroll
        for (int py = 0; py < 2; ++py) {
            float o[4];
#pragma unroll
            for (int i = 0; i < 2; ++i)
#pragma unroll
                for (int px = 0; px < 2; ++px) {
                    float acc = bias;
#pragma unroll
                    for (int a = 0; a < 3; ++a)
#pragma unroll
                        for (int bb = 0; bb < 3; ++bb) acc = fmaf(wf[((py * 2 + px) * 3 + a) * 3 + bb], sv[a][i + bb], acc);
                    o[2 * i + px] = apply_act_fast(acc, act, alpha);
                }
            const int gy = oy0 + 2 * j + py, gx = ox0 + 2 * n0;
            if (gy < g.h && gx < g.w)
                *reinterpret_cast<float4*>(yim + (int64_t)gy * g.w + gx) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
}

static int conv55_c1_tiled(const ConvGeom& g, int ups, const float* x, const float* w, const float* b, float* y, int act,
                           float alpha, cudaStream_t st) {
    if (g.cin != 1 || g.cout != 1 || g.kh != 5 || g.kw != 5 || g.sh != 1 || g.sw != 1 || g.ph != 2 || g.pw != 2 ||
        g.padding_value != 0.f || g.n > 65535 || ceil_div(g.h, C55_TH) > 65535)
        return UOCR_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) return UOCR_ERR_UNSUPPORTED;
    dim3 grid((unsigned)ceil_div(g.w, C55_TW), (unsigned)ceil_div(g.h, C55_TH), (unsigned)g.n);
    if (ups == 2) {
        if (g.w % 8 || g.h % 2) return UOCR_ERR_UNSUPPORTED;
        conv55_c1_ups_tile_kernel<<<grid, 256, 0, st>>>(g, x, w, b, y, act, alpha);
        UOCR_LAUNCHED("conv55_c1_ups_tile");
    } else {
        if (g.w % 4) return UOCR_ERR_UNSUPPORTED;
        conv55_c1_tile_kernel<<<grid, 256, 0, st>>>(g, x, w, b, y, act, alpha);
        UOCR_LAUNCHED("conv55_c1_tile");
    }
    return UOCR_OK;
}

// ------------------------------------------------------------------------------------------
// Cin = 1 -> Cout = 64 (Char conv_1: 5x3, stride (2, 1)): the layer is bound by its 58.7 MB output write, so the
// kernel is organised around the STORE: lane = (channel quad, pixel), a warp's 128-bit store covers two pixels x
// 64 channels = two fully used 256-byte segments (the generic kernel above wrote 16 bytes per lane at a 1 KB
// stride: half-used sectors, 0.038 ms).  CTA = 128 output pixels of one output row; the KH input rows sit in
// shared memory (read as broadcasts), a thread owns 4 channels x 8 consecutive pixels with its 15 x 4 weights in
// registers.
// ------------------------------------------------------------------------------------------
template <int KH, int KW, int SH, int SW, int RB>
__global__ void __launch_bounds__(256) conv_c1_wide64_kernel(ConvGeom g, const float* __restrict__ x,
                                                             const float* __restrict__ w, const float* __restrict__ b,
                                                             float* __restrict__ y, int act, float alpha) {
    // CTA = 128 output pixels x RB output rows: the weights go to registers and the input rows to shared memory ONCE,
    // then the rows are computed and stored back to back (one CTA per output row spent most of its life in the
    // prologue: load -> barrier -> 480 FMA -> store at 16 warps per SM, 0.027 ms for a 9 us write).
    constexpr int TXB = 128, PXT = 8, NQ = 16;              // pixels per CTA, pixels per thread, channel quads
    constexpr int IW = (TXB - 1) * SW + KW;                  // input columns a CTA needs
    constexpr int NIN = (PXT - 1) * SW + KW;                 // ... a thread needs per row
    constexpr int IH = (RB - 1) * SH + KH;                   // input rows of the RB output rows
    __shared__ float s_in[IH][IW + 1];
    const int ox0 = blockIdx.x * TXB, oy0 = blockIdx.y * RB;
    const int64_t n = blockIdx.z;
    const int iy0 = oy0 * SH - g.ph, ix0 = ox0 * SW - g.pw;
    const float* xim = x + n * g.h * (int64_t)g.w;
    for (int i = threadIdx.x; i < IH * IW; i += 256) {
        const int r = i / IW, c = i - r * IW;
        const int iy = iy0 + r, ix = ix0 + c;
        s_in[r][c] = (iy >= 0 && iy < g.h && ix >= 0 && ix < g.w) ? __ldg(xim + (int64_t)iy * g.w + ix) : g.padding_value;
    }
    const int cq = threadIdx.x % NQ, pg = threadIdx.x / NQ;
    float wr[KH * KW][4];
#pragma unroll
    for (int t = 0; t < KH * KW; ++t) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(w + t * 64) + cq);
        wr[t][0] = v.x; wr[t][1] = v.y; wr[t][2] = v.z; wr[t][3] = v.w;
    }
    float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
    if (g.bias) bias = __ldg(reinterpret_cast<const float4*>(b) + cq);
    __syncthreads();
    const int px0 = pg * PXT;
#pragma unroll 1
    for (int ro = 0; ro < RB; ++ro) {
    const int oy = oy0 + ro;
    if (oy >= g.ho) break;
    float acc[PXT][4];
#pragma unroll
    for (int p = 0; p < PXT; ++p) { acc[p][0] = bias.x; acc[p][1] = bias.y; acc[p][2] = bias.z; acc[p][3] = bias.w; }
#pragma unroll
    for (int ky = 0; ky < KH; ++ky) {
        float in[NIN];
#pragma unroll
        for (int j = 0; j < NIN; ++j) in[j] = s_in[ro * SH + ky][px0 * SW + j];
#pragma unroll
        for (int kx = 0; kx < KW; ++kx)
#pragma unroll
            for (int p = 0; p < PXT; ++p)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[p][c] = fmaf(wr[ky * KW + kx][c], in[p * SW + kx], acc[p][c]);
    }
    float* yrow = y + ((n * g.ho + oy) * (int64_t)g.wo + ox0 + px0) * 64 + cq * 4;
#pragma unroll
    for (int p = 0; p < PXT; ++p) {
        if (ox0 + px0 + p < g.wo)
            *reinterpret_cast<float4*>(yrow + (int64_t)p * 64) =
                make_float4(apply_act_fast(acc[p][0], act, alpha), apply_act_fast(acc[p][1], act, alpha),
                            apply_act_fast(acc[p][2], act, alpha), apply_act_fast(acc[p][3], act, alpha));
    }
    }
}

int conv_fwd_fast(const ConvGeom& g, int ups, int math_mode, const float* x, const float* w,
                  const float* b, float* y, int act, float alpha, cudaStream_t st, const float* w_kmajor) {
    if (math_mode == UOCR_MATH_TF32) {
        int rc = conv_fwd_tc(g, x, w, w_kmajor, b, y, act, alpha, st);
        if (rc != UOCR_ERR_UNSUPPORTED) return rc;
        // 5x5 / stride 1 / Cin = 4 (Line up_*, end): row GEMM with TMEM-resident windows (conv_row_tc.cu)
        if (g.ups == ups) {
            rc = conv55_row_tc(g, x, w, b, y, act, alpha, st);
            if (rc != UOCR_ERR_UNSUPPORTED) return rc;
        }
    }
    if (ups != 1 && ups != 2) return UOCR_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) return UOCR_ERR_UNSUPPORTED;
#define UOCR_SMALL(KH_, KW_, SH_, SW_, CIN_, COUTMOD, COT_, PX_)                                    \
    if (g.kh == KH_ && g.kw == KW_ && g.sh == SH_ && g.sw == SW_ && g.cin == CIN_ &&                 \
        g.cout % COUTMOD == 0 && g.cout >= COT_ && (COT_ != 1 || g.cout == 1) && (COT_ != 2 || g.cout == 2)) \
        return launch_small_fwd<KH_, KW_, SH_, SW_, CIN_, COT_, PX_>(g, ups, x, w, b, y, act, alpha, st);
#define UOCR_C1(KH_, KW_, SH_, SW_, COUTMOD, COT_, PX_)                                              \
    if (g.cin == 1 && g.kh == KH_ && g.kw == KW_ && g.sh == SH_ && g.sw == SW_ && g.cout % COUTMOD == 0 && \
        (COT_ != 1 || g.cout == 1)) {                                                                   \
        const int rc = launch_c1_fwd<KH_, KW_, SH_, SW_, COT_, PX_>(g, ups, x, w, b, y, act, alpha, st); \
        if (rc != UOCR_ERR_UNSUPPORTED) return rc;                                                      \
    }
    {
        const int rc = conv55_c1_tiled(g, ups, x, w, b, y, act, alpha, st);     // Paragraph up_*, end (+ stride-1 dgrads)
        if (rc != UOCR_ERR_UNSUPPORTED) return rc;
    }
    if (g.cin == 1 && g.cout == 64 && g.kh == 5 && g.kw == 3 && g.sh == 2 && g.sw == 1 && ups == 1 && g.n <= 65535 &&
        g.ho <= 65535 && !(reinterpret_cast<uintptr_t>(w) & 15) && !(reinterpret_cast<uintptr_t>(b) & 15)) {     // Char conv_1
        constexpr int RB = 7;                                 // Char: 14 output rows -> 2 row groups, 256 CTAs at batch 64
        dim3 grid((unsigned)ceil_div(g.wo, 128), (unsigned)ceil_div(g.ho, RB), (unsigned)g.n);
        conv_c1_wide64_kernel<5, 3, 2, 1, RB><<<grid, 256, 0, st>>>(g, x, w, b, y, act, alpha);
        UOCR_LAUNCHED("conv_c1_wide64");
        return UOCR_OK;
    }
    UOCR_C1(5, 5, 1, 1, 1, 1, 4)             // Paragraph up_*, end
    UOCR_C1(5, 5, 2, 2, 1, 1, 4)             // Paragraph down_*
    UOCR_C1(5, 5, 2, 2, 4, 4, 4)             // Line down_1
    UOCR_C1(3, 3, 1, 1, 16, 16, 4)           // Monochrome conv_1
    UOCR_C1(5, 3, 2, 1, 16, 16, 4)           // Char conv_1
#undef UOCR_C1
    UOCR_SMALL(3, 3, 1, 1, 1, 16, 16, 4)     // Monochrome conv_1
    UOCR_SMALL(3, 3, 1, 1, 16, 1, 1, 8)      // Monochrome conv_2
    UOCR_SMALL(5, 5, 1, 1, 1, 1, 1, 8)       // Paragraph up_*, end
    UOCR_SMALL(5, 5, 2, 2, 1, 1, 1, 8)       // Paragraph down_*
    UOCR_SMALL(5, 5, 2, 2, 1, 4, 4, 4)       // Line down_1
    UOCR_SMALL(5, 5, 2, 2, 4, 4, 4, 4)       // Line down_2
    UOCR_SMALL(5, 5, 1, 1, 4, 4, 4, 4)       // Line up_*
    UOCR_SMALL(5, 5, 1, 1, 4, 2, 2, 4)       // Line end
    UOCR_SMALL(5, 5, 1, 1, 2, 4, 4, 4)       // dgrad of Line end (2 -> 4 on flipped weights)
    UOCR_SMALL(5, 3, 2, 1, 1, 16, 16, 4)     // Char conv_1 (1 -> 64)
#undef UOCR_SMALL
    return UOCR_ERR_UNSUPPORTED;
}

// ------------------------------------------------------------------------------------------
// Fused pair: 3x3 conv (1 -> C1) + act1 + 3x3 conv (C1 -> 1) + act2, padding 1, stride 1
// (my_model's Monochrome net, model.py:119-122, in inference).  The C1-channel hidden map
// (23 MB per 496x736 tile at C1 = 16) never leaves registers: a thread owns CW output columns and
// streams down R rows; for every hidden row and channel it evaluates the CW + 2 hidden pixels it
// needs (9 FFMA each) and immediately scatters them into the three output rows they touch
// (9 * CW FFMA).  No shared memory traffic except 5 broadcast 128-bit weight loads per channel, no
// barriers.  Algorithmic cost 288 FMA / pixel, executed (1 + 2/CW)(1 + 2/R) * 144 + (1 + 2/R) * 144.
// ------------------------------------------------------------------------------------------
constexpr int PAIR_CW = 8, PAIR_R = 16;

// LMAX: act1 is LeakyRelu with 0 < alpha <= 1, evaluated as max(v, alpha * v) (FMUL + FMNMX instead of
// compare + multiply + select).  ncu showed this kernel issue-bound (issue slots 83 % busy) with a third
// of the slots spent on ALU work around the hidden values, so the activation and the image-border
// masking of the hidden pixels (needed by edge strips only) are kept off the common path.
template <int CW, int R, bool LMAX>
__global__ void __launch_bounds__(128) conv3x3_pair_fwd_kernel(
    const float* __restrict__ x, const float* __restrict__ w1, const float* __restrict__ b1,
    const float* __restrict__ w2, const float* __restrict__ b2, float* __restrict__ y, int n_img, int H,
    int W, int C1, int act1, float alpha1, int act2, float alpha2) {
    extern __shared__ __align__(16) float s_p[];            // per channel: w1[9], b1, w2[9], pad -> 20
    for (int i = threadIdx.x; i < C1 * 20; i += 128) {
        const int c = i / 20, k = i % 20;
        float v = 0.f;
        if (k < 9) v = w1[k * C1 + c];                      // w1 (3,3,1,C1)
        else if (k == 9) v = b1[c];
        else if (k < 19) v = w2[(k - 10) * C1 + c];         // w2 (3,3,C1,1)
        s_p[i] = v;
    }
    __syncthreads();

    const int strips = (W + CW - 1) / CW;
    const int rchunks = (H + R - 1) / R;
    const int64_t idx = (int64_t)blockIdx.x * 128 + threadIdx.x;
    const int strip = (int)(idx % strips);
    const int rc = (int)((idx / strips) % rchunks);
    const int64_t n = idx / ((int64_t)strips * rchunks);
    if (n >= n_img) return;
    const int c0 = strip * CW, r0 = rc * R;
    const float* xim = x + n * (int64_t)H * W;
    float* yim = y + n * (int64_t)H * W;
    const float bias2 = __ldg(b2);

    float xr[3][CW + 4];                                    // x rows hr-1, hr, hr+1; cols c0-2 ..
    float accA[CW], accB[CW], accC[CW];                     // output rows hr-1, hr, hr+1
#pragma unroll
    for (int j = 0; j < CW; ++j) accA[j] = accB[j] = accC[j] = 0.f;

    auto load_row = [&](int row, float* dst) {
        const bool rin = row >= 0 && row < H;
#pragma unroll
        for (int j = 0; j < CW + 4; ++j) {
            const int col = c0 - 2 + j;
            dst[j] = (rin && col >= 0 && col < W) ? __ldg(xim + (int64_t)row * W + col) : 0.f;
        }
    };
    load_row(r0 - 2, xr[0]);
    load_row(r0 - 1, xr[1]);

    const int r_end = min(r0 + R, H);
    // does any strip of this warp touch the left / right image border?  (warp-uniform)
    const bool warp_has_edge = __any_sync(__activemask(), (c0 == 0) || (c0 + CW >= W));
    for (int hr = r0 - 1; hr <= r_end; ++hr) {
        load_row(hr + 1, xr[2]);
        if (hr >= 0 && hr < H) {
            // two copies of the channel loop: warps that contain an image-border strip mask the
            // out-of-image hidden columns (conv_2's zero padding); all other warps skip that work
#define UOCR_PAIR_CHANNEL_LOOP(MASKED)                                                                  \
            for (int c = 0; c < C1; ++c) {                                                              \
                const float4* pw = reinterpret_cast<const float4*>(s_p + c * 20);                      \
                const float4 q0 = pw[0], q1 = pw[1], q2 = pw[2], q3 = pw[3], q4 = pw[4];               \
                const float k1[9] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x};            \
                const float bb = q2.y;                                                                  \
                const float k2[9] = {q2.z, q2.w, q3.x, q3.y, q3.z, q3.w, q4.x, q4.y, q4.z};            \
                float h[CW + 2];                                                                        \
                _Pragma("unroll") for (int j = 0; j < CW + 2; ++j) {                                    \
                    float v = bb;                                                                       \
                    _Pragma("unroll") for (int ky = 0; ky < 3; ++ky)                                    \
                        _Pragma("unroll") for (int kx = 0; kx < 3; ++kx)                                \
                            v = fmaf(k1[ky * 3 + kx], xr[ky][j + kx], v);                               \
                    h[j] = LMAX ? fmaxf(v, alpha1 * v) : apply_act_fast(v, act1, alpha1);               \
                    if (MASKED) {                                                                       \
                        const int col = c0 - 1 + j;                                                     \
                        if (col < 0 || col >= W) h[j] = 0.f;                                            \
                    }                                                                                   \
                }                                                                                       \
                _Pragma("unroll") for (int j = 0; j < CW; ++j) {                                        \
                    _Pragma("unroll") for (int kx = 0; kx < 3; ++kx) {                                  \
                        accA[j] = fmaf(k2[6 + kx], h[j + kx], accA[j]); /* ky = 2 -> output row hr - 1 */ \
                        accB[j] = fmaf(k2[3 + kx], h[j + kx], accB[j]); /* ky = 1 -> output row hr     */ \
                        accC[j] = fmaf(k2[kx], h[j + kx], accC[j]);     /* ky = 0 -> output row hr + 1 */ \
                    }                                                                                   \
                }                                                                                       \
            }
            if (warp_has_edge) { UOCR_PAIR_CHANNEL_LOOP(true) } else { UOCR_PAIR_CHANNEL_LOOP(false) }
#undef UOCR_PAIR_CHANNEL_LOOP
        }
        const int orow = hr - 1;
        if (orow >= r0 && orow < r_end) {
            float* yp = yim + (int64_t)orow * W + c0;
            if (c0 + CW <= W && (W & 3) == 0) {
#pragma unroll
                for (int j = 0; j < CW; j += 4) {
                    float4 t;
                    t.x = apply_act_fast(accA[j] + bias2, act2, alpha2);
                    t.y = apply_act_fast(accA[j + 1] + bias2, act2, alpha2);
                    t.z = apply_act_fast(accA[j + 2] + bias2, act2, alpha2);
                    t.w = apply_act_fast(accA[j + 3] + bias2, act2, alpha2);
                    *reinterpret_cast<float4*>(yp + j) = t;
                }
            } else {
#pragma unroll
                for (int j = 0; j < CW; ++j)
                    if (c0 + j < W) yp[j] = apply_act_fast(accA[j] + bias2, act2, alpha2);
            }
        }
#pragma unroll
        for (int j = 0; j < CW; ++j) { accA[j] = accB[j]; accB[j] = accC[j]; accC[j] = 0.f; }
#pragma unroll
        for (int j = 0; j < CW + 4; ++j) { xr[0][j] = xr[1][j]; xr[1][j] = xr[2][j]; }
    }
}

int conv3x3_pair_fwd(const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                     float* y, int64_t n, int64_t h, int64_t w, int c1, int act1, float alpha1, int act2,
                     float alpha2, cudaStream_t st) {
    const int64_t strips = ceil_div(w, PAIR_CW), rchunks = ceil_div(h, PAIR_R);
    const int64_t blocks = ceil_div(n * strips * rchunks, 128);
    if (blocks > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    if (act1 == UOCR_ACT_LEAKY && alpha1 > 0.f && alpha1 <= 1.f)
        conv3x3_pair_fwd_kernel<PAIR_CW, PAIR_R, true><<<(unsigned)blocks, 128, sizeof(float) * 20 * c1, st>>>(
            x, w1, b1, w2, b2, y, (int)n, (int)h, (int)w, c1, act1, alpha1, act2, alpha2);
    else
        conv3x3_pair_fwd_kernel<PAIR_CW, PAIR_R, false><<<(unsigned)blocks, 128, sizeof(float) * 20 * c1, st>>>(
            x, w1, b1, w2, b2, y, (int)n, (int)h, (int)w, c1, act1, alpha1, act2, alpha2);
    UOCR_LAUNCHED("conv3x3_pair_fwd");
    return UOCR_OK;
}

}  // namespace uocr

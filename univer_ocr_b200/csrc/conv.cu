// Convolutional2D forward / dgrad / wgrad -- the general FP32-FFMA path ("check mode").
//
// Reference semantics (nn/layers/convolutional.py):
//   fwd   :62-99    y = bias*b + sum_k w[ky,kx,ci,co] * Xpad[n, oy*sh+ky, ox*sw+kx, ci]
//   dgrad :129-142  dX = scatter of dy . w^T over the padded input, cropped by the padding
//   wgrad :121-139  dW += Xpad^T . dy  (the padded border holds `padding_value` and takes part),
//                   db += bias * sum(dy)
// These kernels handle EVERY geometry (any kernel size / padding / stride / channel count);
// the shape-specialised fast paths (conv_fast.cu, tc_gemm.cu) are validated against them.
#include <stdlib.h>

#include "common.cuh"
#include "conv_common.cuh"

namespace uocr {

// ------------------------------------------------------------------ forward
// one thread = one output pixel x COT consecutive output channels; item index runs
// (pixel, channel-chunk) with the chunk fastest, so a warp writes contiguous NHWC memory.
template <int COT>
__global__ void __launch_bounds__(kThreads) conv_fwd_direct_kernel(ConvGeom g, const float* __restrict__ x,
                                                                   const float* __restrict__ w,
                                                                   const float* __restrict__ b,
                                                                   float* __restrict__ y, int act,
                                                                   float alpha) {
    const int chunks = g.cout / COT;
    const int64_t items = (int64_t)g.n * g.ho * g.wo * chunks;
    for (int64_t it = (int64_t)blockIdx.x * kThreads + threadIdx.x; it < items;
         it += (int64_t)gridDim.x * kThreads) {
        const int chunk = (int)(it % chunks);
        int64_t pix = it / chunks;
        const int ox = (int)(pix % g.wo);
        const int oy = (int)((pix / g.wo) % g.ho);
        const int n = (int)(pix / ((int64_t)g.wo * g.ho));
        const int co0 = chunk * COT;
        float acc[COT];
#pragma unroll
        for (int j = 0; j < COT; ++j) acc[j] = 0.f;
        const int iy0 = oy * g.sh - g.ph, ix0 = ox * g.sw - g.pw;
        for (int ky = 0; ky < g.kh; ++ky) {
            const int iy = iy0 + ky;
            const bool yin = iy >= 0 && iy < g.h;
            for (int kx = 0; kx < g.kw; ++kx) {
                const int ix = ix0 + kx;
                const bool in = yin && ix >= 0 && ix < g.w;
                const float* xp = x + (((int64_t)n * (g.h / g.ups) + iy / g.ups) * (g.w / g.ups) + ix / g.ups) * g.cin;
                const float* wp = w + ((int64_t)(ky * g.kw + kx) * g.cin) * g.cout + co0;
                for (int ci = 0; ci < g.cin; ++ci) {
                    const float xv = in ? __ldg(xp + ci) : g.padding_value;
#pragma unroll
                    for (int j = 0; j < COT; ++j) acc[j] = fmaf(xv, __ldg(wp + j), acc[j]);
                    wp += g.cout;
                }
            }
        }
        float* yp = y + pix * g.cout + co0;
#pragma unroll
        for (int j = 0; j < COT; ++j) {
            float v = acc[j] + (g.bias ? __ldg(b + co0 + j) : 0.f);
            yp[j] = apply_act(v, act, alpha);
        }
    }
}

// ------------------------------------------------------------------ dgrad (gather form)
// one thread = one input pixel x CIT consecutive input channels
template <int CIT>
__global__ void __launch_bounds__(kThreads) conv_dgrad_direct_kernel(ConvGeom g,
                                                                     const float* __restrict__ dy,
                                                                     const float* __restrict__ w,
                                                                     float* __restrict__ dx) {
    const int chunks = g.cin / CIT;
    const int64_t items = (int64_t)g.n * g.h * g.w * chunks;
    for (int64_t it = (int64_t)blockIdx.x * kThreads + threadIdx.x; it < items;
         it += (int64_t)gridDim.x * kThreads) {
        const int chunk = (int)(it % chunks);
        int64_t pix = it / chunks;
        const int ix = (int)(pix % g.w);
        const int iy = (int)((pix / g.w) % g.h);
        const int n = (int)(pix / ((int64_t)g.w * g.h));
        const int ci0 = chunk * CIT;
        float acc[CIT];
#pragma unroll
        for (int j = 0; j < CIT; ++j) acc[j] = 0.f;
        for (int ky = 0; ky < g.kh; ++ky) {
            const int ty = iy + g.ph - ky;
            if (ty < 0 || ty % g.sh != 0) continue;
            const int oy = ty / g.sh;
            if (oy >= g.ho) continue;
            for (int kx = 0; kx < g.kw; ++kx) {
                const int tx = ix + g.pw - kx;
                if (tx < 0 || tx % g.sw != 0) continue;
                const int ox = tx / g.sw;
                if (ox >= g.wo) continue;
                const float* gp = dy + (((int64_t)n * g.ho + oy) * g.wo + ox) * g.cout;
                const float* wp = w + ((int64_t)(ky * g.kw + kx) * g.cin + ci0) * g.cout;
                for (int co = 0; co < g.cout; ++co) {
                    const float gv = __ldg(gp + co);
#pragma unroll
                    for (int j = 0; j < CIT; ++j)
                        acc[j] = fmaf(gv, __ldg(wp + (int64_t)j * g.cout + co), acc[j]);
                }
            }
        }
        float* dp = dx + pix * g.cin + ci0;
#pragma unroll
        for (int j = 0; j < CIT; ++j) dp[j] = acc[j];
    }
}

// ------------------------------------------------------------------ wgrad
// dWb[k, co] = sum_m A[m, k] * dy[m, co],  m = (n, oy, ox),  k = (ky, kx, ci) plus one extra
// row k == K whose A column is the constant `bias` flag (that row is db) -- the same
// [patch, 1] trick the reference uses (convolutional.py:124-128).
// CTA tile: KT x CT outputs, reduction over its slice of m in steps of MT pixels staged in smem;
// partial tiles go to workspace[split][K+1][cout], summed by wgrad_reduce_kernel
// (deterministic: no atomics).
constexpr int WG_MT = 32;

template <int KT, int CT, int RK, int RC>
__global__ void __launch_bounds__((KT / RK) * (CT / RC)) conv_wgrad_tile_kernel(
    ConvGeom g, const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ ws,
    int64_t m_per_split) {
    constexpr int NT = (KT / RK) * (CT / RC);
    __shared__ float s_a[WG_MT][KT + 1];
    __shared__ float s_d[WG_MT][CT + 1];
    __shared__ int s_ky[KT], s_kx[KT], s_ci[KT];            // s_ci < 0: -1 = bias row, -2 = beyond K
    __shared__ int s_iy0[WG_MT], s_ix0[WG_MT];
    __shared__ int64_t s_base[WG_MT];                        // n * H * W, or -1 beyond M

    const int tid = threadIdx.x;
    const int K = g.kh * g.kw * g.cin;
    const int k0 = blockIdx.x * KT, c0 = blockIdx.y * CT;
    const int64_t M = (int64_t)g.n * g.ho * g.wo;
    const int64_t m_begin = (int64_t)blockIdx.z * m_per_split;
    const int64_t m_end = min(M, m_begin + m_per_split);

    for (int k = tid; k < KT; k += NT) {
        const int kk = k0 + k;
        if (kk < K) {
            s_ci[k] = kk % g.cin;
            s_kx[k] = (kk / g.cin) % g.kw;
            s_ky[k] = kk / (g.cin * g.kw);
        } else {
            s_ci[k] = (kk == K) ? -1 : -2;
            s_kx[k] = s_ky[k] = 0;
        }
    }

    const int tk = (tid % (KT / RK)) * RK;      // k fastest across threads
    const int tc = (tid / (KT / RK)) * RC;
    float acc[RK][RC];
#pragma unroll
    for (int i = 0; i < RK; ++i)
#pragma unroll
        for (int j = 0; j < RC; ++j) acc[i][j] = 0.f;

    for (int64_t m0 = m_begin; m0 < m_end; m0 += WG_MT) {
        __syncthreads();                          // previous tile consumed (and tables ready)
        for (int mm = tid; mm < WG_MT; mm += NT) {
            const int64_t m = m0 + mm;
            if (m < m_end) {
                const int ox = (int)(m % g.wo);
                const int oy = (int)((m / g.wo) % g.ho);
                const int64_t n = m / ((int64_t)g.wo * g.ho);
                s_iy0[mm] = oy * g.sh - g.ph;
                s_ix0[mm] = ox * g.sw - g.pw;
                s_base[mm] = n * g.h * g.w;
            } else {
                s_base[mm] = -1;
                s_iy0[mm] = s_ix0[mm] = 0;
            }
        }
        __syncthreads();
        for (int e = tid; e < WG_MT * KT; e += NT) {
            const int mm = e / KT, k = e % KT;
            float v = 0.f;
            const int64_t base = s_base[mm];
            const int ci = s_ci[k];
            if (base >= 0 && ci != -2) {
                if (ci == -1) {
                    v = g.bias ? 1.f : 0.f;
                } else {
                    const int iy = s_iy0[mm] + s_ky[k], ix = s_ix0[mm] + s_kx[k];
                    v = (iy >= 0 && iy < g.h && ix >= 0 && ix < g.w)
                            ? __ldg(x + (base + (int64_t)iy * g.w + ix) * g.cin + ci)
                            : g.padding_value;
                }
            }
            s_a[mm][k] = v;
        }
        for (int e = tid; e < WG_MT * CT; e += NT) {
            const int mm = e / CT, c = e % CT;
            const int64_t m = m0 + mm;
            s_d[mm][c] = (m < m_end && c0 + c < g.cout) ? __ldg(dy + m * g.cout + c0 + c) : 0.f;
        }
        __syncthreads();
#pragma unroll 4
        for (int mm = 0; mm < WG_MT; ++mm) {
            float a[RK], d[RC];
#pragma unroll
            for (int i = 0; i < RK; ++i) a[i] = s_a[mm][tk + i];
#pragma unroll
            for (int j = 0; j < RC; ++j) d[j] = s_d[mm][tc + j];
#pragma unroll
            for (int i = 0; i < RK; ++i)
#pragma unroll
                for (int j = 0; j < RC; ++j) acc[i][j] = fmaf(a[i], d[j], acc[i][j]);
        }
    }

    float* out = ws + (int64_t)blockIdx.z * (K + 1) * g.cout;
#pragma unroll
    for (int i = 0; i < RK; ++i) {
        const int kk = k0 + tk + i;
        if (kk > K) continue;
#pragma unroll
        for (int j = 0; j < RC; ++j) {
            const int cc = c0 + tc + j;
            if (cc < g.cout) out[(int64_t)kk * g.cout + cc] = acc[i][j];
        }
    }
}

// dw[i] (+)= sum_s ws[s][i]  for i < K*cout ; db[c] (+)= sum_s ws[s][K*cout + c]
__global__ void __launch_bounds__(kThreads) conv_wgrad_reduce_kernel(const float* __restrict__ ws,
                                                                     int splits, int64_t kc, int cout,
                                                                     float* __restrict__ dw,
                                                                     float* __restrict__ db,
                                                                     int accumulate) {
    const int64_t total = kc + cout;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < total;
         i += (int64_t)gridDim.x * kThreads) {
        float s = 0.f;
        for (int sp = 0; sp < splits; ++sp) s += ws[(int64_t)sp * total + i];
        float* dst = (i < kc) ? dw + i : db + (i - kc);
        *dst = accumulate ? *dst + s : s;
    }
}

struct WgradPlan {
    int kt, ct, ktiles, ctiles, splits;
    int64_t m_per_split;
};

static WgradPlan plan_wgrad(const ConvGeom& g) {
    WgradPlan p;
    if (g.cout >= 32) { p.kt = 64; p.ct = 64; }
    else if (g.cout >= 9) { p.kt = 64; p.ct = 16; }
    else { p.kt = 32; p.ct = 8; }
    const int K1 = g.kh * g.kw * g.cin + 1;
    p.ktiles = (K1 + p.kt - 1) / p.kt;
    p.ctiles = (g.cout + p.ct - 1) / p.ct;
    const int64_t M = (int64_t)g.n * g.ho * g.wo;
    const int64_t tiles = (int64_t)p.ktiles * p.ctiles;
    int64_t splits = (148 * 4 + tiles - 1) / tiles;           // ~4 CTAs per SM in flight
    const int64_t max_splits = (M + WG_MT * 8 - 1) / (WG_MT * 8);   // >= 8 smem tiles per CTA
    if (splits > max_splits) splits = max_splits;
    if (splits < 1) splits = 1;
    if (splits > 4096) splits = 4096;
    int64_t mps = (M + splits - 1) / splits;
    mps = (mps + WG_MT - 1) / WG_MT * WG_MT;
    p.m_per_split = mps;
    p.splits = (int)((M + mps - 1) / mps);
    return p;
}

template <int COT>
static int launch_fwd(const ConvGeom& g, const float* x, const float* w, const float* b, float* y,
                      int act, float alpha, cudaStream_t st) {
    const int64_t items = (int64_t)g.n * g.ho * g.wo * (g.cout / COT);
    int64_t blocks = ceil_div(items, kThreads);
    if (blocks > 148 * 32) blocks = 148 * 32;
    conv_fwd_direct_kernel<COT><<<(int)blocks, kThreads, 0, st>>>(g, x, w, b, y, act, alpha);
    UOCR_LAUNCHED("conv2d_fwd_direct");
    return UOCR_OK;
}

template <int CIT>
static int launch_dgrad(const ConvGeom& g, const float* dy, const float* w, float* dx, cudaStream_t st) {
    const int64_t items = (int64_t)g.n * g.h * g.w * (g.cin / CIT);
    int64_t blocks = ceil_div(items, kThreads);
    if (blocks > 148 * 32) blocks = 148 * 32;
    conv_dgrad_direct_kernel<CIT><<<(int)blocks, kThreads, 0, st>>>(g, dy, w, dx);
    UOCR_LAUNCHED("conv2d_dgrad_direct");
    return UOCR_OK;
}

int conv_fwd_general(const ConvGeom& g, const float* x, const float* w, const float* b, float* y,
                     int act, float alpha, cudaStream_t st) {
    if (g.cout % 16 == 0) return launch_fwd<16>(g, x, w, b, y, act, alpha, st);
    if (g.cout % 8 == 0) return launch_fwd<8>(g, x, w, b, y, act, alpha, st);
    if (g.cout % 4 == 0) return launch_fwd<4>(g, x, w, b, y, act, alpha, st);
    if (g.cout % 2 == 0) return launch_fwd<2>(g, x, w, b, y, act, alpha, st);
    return launch_fwd<1>(g, x, w, b, y, act, alpha, st);
}

int conv_dgrad_general(const ConvGeom& g, const float* dy, const float* w, float* dx, cudaStream_t st) {
    if (g.cin % 8 == 0) return launch_dgrad<8>(g, dy, w, dx, st);
    if (g.cin % 4 == 0) return launch_dgrad<4>(g, dy, w, dx, st);
    if (g.cin % 2 == 0) return launch_dgrad<2>(g, dy, w, dx, st);
    return launch_dgrad<1>(g, dy, w, dx, st);
}

size_t conv_wgrad_general_workspace(const ConvGeom& g) {
    const WgradPlan p = plan_wgrad(g);
    return (size_t)p.splits * ((size_t)g.kh * g.kw * g.cin + 1) * g.cout * sizeof(float);
}

int conv_wgrad_general(const ConvGeom& g, const float* x, const float* dy, float* dw, float* db,
                       int accumulate, float* ws, cudaStream_t st) {
    const WgradPlan p = plan_wgrad(g);
    dim3 grid(p.ktiles, p.ctiles, p.splits);
    if (p.ct == 64) {
        conv_wgrad_tile_kernel<64, 64, 4, 4><<<grid, 256, 0, st>>>(g, x, dy, ws, p.m_per_split);
    } else if (p.ct == 16) {
        conv_wgrad_tile_kernel<64, 16, 4, 1><<<grid, 256, 0, st>>>(g, x, dy, ws, p.m_per_split);
    } else {
        conv_wgrad_tile_kernel<32, 8, 1, 1><<<grid, 256, 0, st>>>(g, x, dy, ws, p.m_per_split);
    }
    UOCR_LAUNCHED("conv2d_wgrad_tile");
    const int64_t kc = (int64_t)g.kh * g.kw * g.cin * g.cout;
    conv_wgrad_reduce_kernel<<<ew_grid(kc + g.cout, 1), kThreads, 0, st>>>(ws, p.splits, kc, g.cout, dw,
                                                                           db, accumulate);
    UOCR_LAUNCHED("conv2d_wgrad_reduce");
    return UOCR_OK;
}

}  // namespace uocr

using namespace uocr;

static int make_geom(const uocr_conv2d_desc* d, ConvGeom* g) {
    UOCR_REQUIRE(d, "descriptor is NULL");
    UOCR_REQUIRE(d->n > 0 && d->h > 0 && d->w > 0 && d->cin > 0 && d->cout > 0,
                 "non-positive tensor dimension");
    UOCR_REQUIRE(d->kh > 0 && d->kw > 0 && d->sh > 0 && d->sw > 0, "non-positive kernel/stride");
    UOCR_REQUIRE(d->ph >= 0 && d->pw >= 0, "padding cannot be negative");
    UOCR_REQUIRE(d->h + 2 * d->ph >= d->kh && d->w + 2 * d->pw >= d->kw,
                 "kernel larger than the padded input");
    UOCR_REQUIRE(d->n < (1 << 30) && d->h < (1 << 30) && d->w < (1 << 30) && d->cin < (1 << 20) &&
                     d->cout < (1 << 20), "dimension too large");
    g->n = (int)d->n; g->h = (int)d->h; g->w = (int)d->w; g->cin = (int)d->cin; g->cout = (int)d->cout;
    g->kh = d->kh; g->kw = d->kw; g->ph = d->ph; g->pw = d->pw; g->sh = d->sh; g->sw = d->sw;
    g->ho = (g->h + 2 * g->ph - g->kh) / g->sh + 1;
    g->wo = (g->w + 2 * g->pw - g->kw) / g->sw + 1;
    g->padding_value = d->padding_value;
    g->bias = d->bias ? 1 : 0;
    g->ups = d->in_upsample >= 2 ? d->in_upsample : 1;
    UOCR_REQUIRE(g->ups <= 2 && g->h % g->ups == 0 && g->w % g->ups == 0,
                 "in_upsample must be 0, 1 or 2 and divide H and W");
    return UOCR_OK;
}

extern "C" {

int uocr_conv2d_out_hw(const uocr_conv2d_desc* d, int64_t* ho, int64_t* wo) {
    UOCR_REQUIRE(ho && wo, "NULL pointer");
    ConvGeom g;
    int rc = make_geom(d, &g);
    if (rc) return rc;
    *ho = g.ho;
    *wo = g.wo;
    return UOCR_OK;
}

static int conv2d_fwd_impl(const uocr_conv2d_desc* d, const float* x, const float* w, const float* w_kmajor,
                           const float* b, float* y, int act, float alpha, void* stream) {
    ConvGeom g;
    int rc = make_geom(d, &g);
    if (rc) return rc;
    UOCR_REQUIRE(x && w && b && y, "NULL pointer");
    UOCR_REQUIRE(act >= UOCR_ACT_NONE && act <= UOCR_ACT_SIGMOID, "unknown activation %d", act);
    cudaStream_t st = as_stream(stream);
    rc = conv_fwd_fast(g, g.ups, d->math_mode, x, w, b, y, act, alpha, st, w_kmajor);
    if (rc != UOCR_ERR_UNSUPPORTED) return rc;
    return conv_fwd_general(g, x, w, b, y, act, alpha, st);
}

int uocr_conv2d_fwd(const uocr_conv2d_desc* d, const float* x, const float* w, const float* b,
                    float* y, int act, float alpha, void* stream) {
    return conv2d_fwd_impl(d, x, w, nullptr, b, y, act, alpha, stream);
}

int uocr_conv2d_fwd_kmajor(const uocr_conv2d_desc* d, const float* x, const float* w, const float* w_kmajor,
                           const float* b, float* y, int act, float alpha, void* stream) {
    return conv2d_fwd_impl(d, x, w, w_kmajor, b, y, act, alpha, stream);
}

int uocr_conv3x3_pair_fwd(const float* x, const float* w1, const float* b1, const float* w2,
                          const float* b2, float* y, int64_t n, int64_t h, int64_t w, int32_t c_mid,
                          int act1, float alpha1, int act2, float alpha2, int math_mode, void* stream) {
    UOCR_REQUIRE(x && w1 && b1 && w2 && b2 && y, "NULL pointer");
    UOCR_REQUIRE(n > 0 && h > 0 && w > 0 && c_mid > 0 && c_mid <= 256, "bad dimension");
    UOCR_REQUIRE(h < (1 << 30) && w < (1 << 30), "dimension too large");
    UOCR_REQUIRE(act1 >= UOCR_ACT_NONE && act1 <= UOCR_ACT_SIGMOID && act2 >= UOCR_ACT_NONE &&
                     act2 <= UOCR_ACT_SIGMOID, "unknown activation");
    // TF32 mode, c_mid == 16: on the tensor cores.  First the persistent warp-specialised kernel whose GEMM 1 reads the
    // image rows in shared memory through overlapping descriptor rows (conv_pair_rows_tc.cu); where that one has no
    // kernel (w % 4 != 0, w < 8, unaligned x, ...), the one that stores both convolutions' windows to tensor memory
    // (conv_pair_tc.cu).  FP32 mode and every other shape: the CUDA-core pair kernel.
    if (math_mode == UOCR_MATH_TF32) {
        int rc = conv3x3_pair_rows(x, w1, b1, w2, b2, y, n, h, w, c_mid, act1, alpha1, act2, alpha2, as_stream(stream));
        if (rc == UOCR_ERR_UNSUPPORTED)
            rc = conv3x3_pair_tmem(x, w1, b1, w2, b2, y, n, h, w, c_mid, act1, alpha1, act2, alpha2, as_stream(stream));
        if (rc != UOCR_ERR_UNSUPPORTED) return rc;
    }
    return conv3x3_pair_fwd(x, w1, b1, w2, b2, y, n, h, w, c_mid, act1, alpha1, act2, alpha2,
                            as_stream(stream));
}

int uocr_conv3x3_pair_bwd_workspace(int64_t n, int64_t h, int64_t w, int32_t c_mid, size_t* bytes) {
    UOCR_REQUIRE(bytes && n > 0 && h > 0 && w > 0 && c_mid > 0, "bad argument");
    *bytes = conv3x3_pair_bwd_workspace(n, h, w, c_mid);
    return UOCR_OK;
}

static int pair_bwd_impl(const float* x, const float* w1, const float* b1, const float* w2, const float* dy,
                         float* dx, float* dw1, float* db1, float* dw2, float* db2, int64_t n, int64_t h,
                         int64_t w, int32_t c_mid, int act1, float alpha1, int accumulate, void* workspace,
                         size_t workspace_bytes, int math_mode, void* stream);

int uocr_conv3x3_pair_bwd(const float* x, const float* w1, const float* b1, const float* w2, const float* dy,
                          float* dx, float* dw1, float* db1, float* dw2, float* db2, int64_t n, int64_t h,
                          int64_t w, int32_t c_mid, int act1, float alpha1, int accumulate, void* workspace,
                          size_t workspace_bytes, void* stream) {
    return pair_bwd_impl(x, w1, b1, w2, dy, dx, dw1, db1, dw2, db2, n, h, w, c_mid, act1, alpha1, accumulate, workspace,
                         workspace_bytes, UOCR_MATH_FP32, stream);
}

int uocr_conv3x3_pair_bwd_mode(const float* x, const float* w1, const float* b1, const float* w2, const float* dy,
                               float* dx, float* dw1, float* db1, float* dw2, float* db2, int64_t n, int64_t h,
                               int64_t w, int32_t c_mid, int act1, float alpha1, int accumulate, void* workspace,
                               size_t workspace_bytes, int math_mode, void* stream) {
    return pair_bwd_impl(x, w1, b1, w2, dy, dx, dw1, db1, dw2, db2, n, h, w, c_mid, act1, alpha1, accumulate, workspace,
                         workspace_bytes, math_mode, stream);
}

static int pair_bwd_impl(const float* x, const float* w1, const float* b1, const float* w2, const float* dy,
                         float* dx, float* dw1, float* db1, float* dw2, float* db2, int64_t n, int64_t h,
                         int64_t w, int32_t c_mid, int act1, float alpha1, int accumulate, void* workspace,
                         size_t workspace_bytes, int math_mode, void* stream) {
    UOCR_REQUIRE(x && w1 && b1 && w2 && dy && dw1 && db1 && dw2 && db2, "NULL pointer");
    UOCR_REQUIRE(n > 0 && h > 0 && w > 0 && c_mid > 0 && c_mid <= 256, "bad dimension");
    UOCR_REQUIRE(h < (1 << 30) && w < (1 << 30), "dimension too large");
    UOCR_REQUIRE(act1 == UOCR_ACT_NONE || (act1 == UOCR_ACT_LEAKY && alpha1 > 0.f),
                 "the middle activation must be LeakyRelu (alpha > 0) or none");
    const size_t need = conv3x3_pair_bwd_workspace(n, h, w, c_mid);
    if (!workspace || workspace_bytes < need) {
        set_error("pair backward workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return UOCR_ERR_WORKSPACE;
    }
    return conv3x3_pair_bwd(x, w1, b1, w2, dy, dx, dw1, db1, dw2, db2, n, h, w, c_mid, act1, alpha1, accumulate,
                            (float*)workspace, as_stream(stream), math_mode);
}

int uocr_conv2d_dgrad(const uocr_conv2d_desc* d, const float* dy, const float* w, float* dx,
                      void* stream) {
    ConvGeom g;
    int rc = make_geom(d, &g);
    if (rc) return rc;
    UOCR_REQUIRE(dy && w && dx, "NULL pointer");
    UOCR_REQUIRE(g.ups == 1, "in_upsample is a forward-only fusion");
    cudaStream_t st = as_stream(stream);
    rc = conv_dgrad_fast(g, d->math_mode, dy, w, dx, st);
    if (rc != UOCR_ERR_UNSUPPORTED) return rc;
    return conv_dgrad_general(g, dy, w, dx, st);
}

int uocr_conv2d_wgrad_workspace(const uocr_conv2d_desc* d, size_t* bytes) {
    UOCR_REQUIRE(bytes, "NULL pointer");
    ConvGeom g;
    int rc = make_geom(d, &g);
    if (rc) return rc;
    size_t fast = conv_wgrad_fast_workspace(g, d->math_mode);
    size_t gen = conv_wgrad_general_workspace(g);
    *bytes = fast > gen ? fast : gen;
    return UOCR_OK;
}

int uocr_conv2d_wgrad(const uocr_conv2d_desc* d, const float* x, const float* dy, float* dw,
                      float* db, int accumulate, void* workspace, size_t workspace_bytes,
                      void* stream) {
    ConvGeom g;
    int rc = make_geom(d, &g);
    if (rc) return rc;
    UOCR_REQUIRE(x && dy && dw && db, "NULL pointer");
    size_t need = 0;
    uocr_conv2d_wgrad_workspace(d, &need);
    if (need > 0 && (!workspace || workspace_bytes < need)) {
        set_error("wgrad workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return UOCR_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    rc = conv_wgrad_fast(g, d->math_mode, x, dy, dw, db, accumulate, (float*)workspace, st);
    if (rc != UOCR_ERR_UNSUPPORTED) return rc;
    // x stored at half resolution (in_upsample == 2) is only understood by the 5x5 / 1 -> 1 / stride 1 kernel
    UOCR_REQUIRE(g.ups == 1, "in_upsample == 2: no weight-gradient kernel for this geometry");
    return conv_wgrad_general(g, x, dy, dw, db, accumulate, (float*)workspace, st);
}

}  // extern "C"

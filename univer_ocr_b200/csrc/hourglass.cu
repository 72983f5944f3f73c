// Fused single-channel "hourglass" forward (inference): the whole Paragraph network in one kernel.
//
//   x -> conv5x5 s2 + act -> conv5x5 s2 + act -> up x2, conv5x5 + act -> up x2, conv5x5 + act -> conv5x5 + act_end -> y
//        (down_1)            (down_2)            (up_2)                  (up_1)                  (end)
//   replaces, for make_paragraph (my_model/model.py:137-190, channels = 1): five Convolutional2D._forward calls
//   (convolutional.py:62-99), two Upsample2D._forward (upsample.py:21-39) and five LeakyRelu / Sigmoid._forward
//   (layers.py:390-415), i.e. 12 layer calls that move 18.6 MB per 496 x 736 tile between them; fused, a tile is
//   read once and written once (2.92 MB, SURVEY.md 8d).
//
// One CTA produces a TH x TW block of the output.  Working backwards through the five 5 x 5 convolutions gives
// the region of every intermediate map the block depends on (receptive field 29 + the stride-2 alignment):
//   X  (TH + 25) x (TW + 25)   full resolution, origin (oy0 - 14, ox0 - 14)
//   D1 (TH/2 + 11) x (TW/2 + 11)   half,    origin (oy0/2 - 6, ..)       D2 (TH/4 + 4) x (TW/4 + 4)  quarter, origin (oy0/4 - 2, ..)
//   U2 (TH/2 + 4) x (TW/2 + 4)     half,    origin (oy0/2 - 2, ..)       U1 (TH + 4) x (TW + 4)      full,    origin (oy0 - 2, ..)
// all of which live in shared memory (70 KB for 32 x 128 blocks, 3 CTAs per SM); halo recomputation costs 22 % extra
// FMAs.  Values outside an intermediate map's image are stored as 0 -- they are the next convolution's zero padding.
// With these origins every level reads its source at (2 r + ky, 2 c + kx) or (r + ky, c + kx): no index arithmetic.
//
// A 5 x 5 convolution over a x2 nearest-upsampled map only ever sees 3 x 3 distinct source pixels: for output row
// parity 0 the kernel rows {0,1}, {2,3}, {4} hit source rows m-1, m, m+1, for parity 1 the rows {0}, {1,2}, {3,4};
// same for columns.  The two "up" levels therefore run as four parity-specific 3 x 3 convolutions on the low-resolution
// map with pre-summed weights (9 FMA per output instead of 25; the upsampled map is never materialised).
// Register tiling: a thread computes 4 (stride-2 levels) or 8 (stride-1 / up levels) outputs of a row from 64-bit
// shared loads, weights in registers.
#include "conv_common.cuh"
#include "tc_ptx.cuh"

namespace uocr {

struct HourglassParams {
    const float* x; float* y;
    const float* w[5]; const float* b[5];       // down_1, down_2, up_2, up_1, end : (5,5,1,1) + (1)
    int H, W;
    float alpha;                                 // LeakyReLU slope of the four inner activations
    int act_end; float alpha_end;
};

// a level's 25 weights + bias in shared memory: 28 floats, so that every level's slot is 16-byte aligned and a thread
// fetches it with 7 vector loads (scalar loads of weights were a quarter of the kernel's shared-memory wavefronts)
constexpr int HG_WSLOT = 28;

template <int TH, int TW>
struct HG {
    // X block: origin column ox0 - 16 (16-byte aligned rows; the convolution reads from column 2 on), two spare rows
    // for the last 4-row strip of D1
    static constexpr int XH = TH + 25, XW = TW + 27, XP = (XW + 1 + 3) & ~3, XROWS = XH + 2;
    static constexpr int D1H = TH / 2 + 11, D1W = TW / 2 + 11, D1P = (D1W + 3 + 3) & ~3;
    static constexpr int D2H = TH / 4 + 4, D2W = TW / 4 + 4, D2P = (D2W + 2 + 3 + 3) & ~3;
    static constexpr int U2H = TH / 2 + 4, U2W = TW / 2 + 4, U2P = (U2W + 3 + 3) & ~3;
    static constexpr int U1H = TH + 4, U1W = TW + 4, U1P = (U1W + 3 + 3) & ~3;
    // the U1 block lives in the x block, which is dead after down_1 -- 54.6 KB, 4 CTAs / SM
    static constexpr int FLOATS = XROWS * XP + D1H * D1P + D2H * D2P + U2H * U2P + 5 * HG_WSLOT + 2 * 36 + 6;
    static_assert(U1H * U1P <= XROWS * XP, "U1 fits into the x block");
};

constexpr int HG_THREADS = 256;
// 64-row blocks run with 512 threads (2 CTAs / SM = the same 32 warps): 7 % fewer halo FMAs, half the prologues
__host__ __device__ constexpr int hg_threads(int th) { return th >= 64 ? 512 : HG_THREADS; }

template <int N4>
__device__ __forceinline__ void hg_load_weights(const float* __restrict__ src, float* w) {
#pragma unroll
    for (int i = 0; i < N4; ++i) {
        const float4 v = reinterpret_cast<const float4*>(src)[i];
        w[4 * i] = v.x; w[4 * i + 1] = v.y; w[4 * i + 2] = v.z; w[4 * i + 3] = v.w;
    }
}

// dst (DH x DW, origin (gy0, gx0) at its resolution, image hl x wl) = act(conv5x5 stride 2 (src) + b); src(2r+ky, 2c+kx).
// Thread = one output column x R rows: neighbouring lanes read neighbouring 8-byte words (no bank conflicts).  R = 4
// for the large level; the small one (12 x 36) uses R = 2 so that seven warps share its 222 strips instead of four
// warps carrying 111 (the level is latency-, not throughput-bound: ncu showed the other warps parked at the barrier).
template <int DH, int DW, int DP, int SP, int R, int NT>
__device__ __forceinline__ void hg_down(const float* __restrict__ src, float* __restrict__ dst, const float* __restrict__ wb,
                                        int gy0, int gx0, int hl, int wl, float alpha) {
    float w[28];
    hg_load_weights<7>(wb, w);
    const float bias = w[25];
    constexpr int STRIPS = (DH + R - 1) / R;
    for (int item = threadIdx.x; item < STRIPS * DW; item += NT) {
        const int s = item / DW, c = item - s * DW, r0 = R * s;
        float acc[R];
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j] = bias;
#pragma unroll
        for (int rr = 0; rr < 2 * R + 3; ++rr) {
            const float2* row = reinterpret_cast<const float2*>(src + (2 * r0 + rr) * SP + 2 * c);
            const float2 a = row[0], b = row[1], e = row[2];
            const float in[5] = {a.x, a.y, b.x, b.y, e.x};
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const int ky = rr - 2 * j;
                if (ky >= 0 && ky < 5) {
#pragma unroll
                    for (int kx = 0; kx < 5; ++kx) acc[j] = fmaf(w[ky * 5 + kx], in[kx], acc[j]);
                }
            }
        }
        const bool colin = (unsigned)(gx0 + c) < (unsigned)wl;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            const float v = fmaxf(acc[j], acc[j] * alpha);
            if (r0 + j < DH) dst[(r0 + j) * DP + c] = (colin && (unsigned)(gy0 + r0 + j) < (unsigned)hl) ? v : 0.f;
        }
    }
}

// The large stride-2 level (x block -> D1) with 16-byte loads: thread = D1 columns (2 p - 1, 2 p) x R rows.  Column j reads
// block columns 2 + 2 j + kx (the block starts 16 columns left of the output block, the convolution 14), so the pair's
// eight inputs are block columns 4 p .. 4 p + 7: two aligned 128-bit loads per input row at lane stride 16 bytes
// (conflict-free), 2.6 input floats per FMA-column instead of 6 with the one-column-per-thread form above.  R = 5: the
// 27 x 75 block is 6 strips x 38 pairs = 228 items, one pass of the 256 threads (R = 4 needs a second pass for 10 items).
// The last strip's rows past DH read beyond the x block's spare rows into the D1 block; they are not stored.
template <int DH, int DW, int DP, int SP, int R, int NT>
__device__ __forceinline__ void hg_down_pairs(const float* __restrict__ src, float* __restrict__ dst, const float* __restrict__ wb,
                                              int gy0, int gx0, int hl, int wl, float alpha) {
    float w[28];
    hg_load_weights<7>(wb, w);
    const float bias = w[25];
    constexpr int STRIPS = (DH + R - 1) / R, PAIRS = DW / 2 + 1;
    for (int item = threadIdx.x; item < STRIPS * PAIRS; item += NT) {
        const int s = item / PAIRS, pr = item - s * PAIRS, r0 = R * s;
        float acc[R][2];
#pragma unroll
        for (int j = 0; j < R; ++j) acc[j][0] = acc[j][1] = bias;
#pragma unroll
        for (int rr = 0; rr < 2 * R + 3; ++rr) {
            const float4* row = reinterpret_cast<const float4*>(src + (2 * r0 + rr) * SP + 4 * pr);
            const float4 u = row[0], v = row[1];
            const float in[8] = {u.x, u.y, u.z, u.w, v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < R; ++j) {
                const int ky = rr - 2 * j;
                if (ky >= 0 && ky < 5) {
#pragma unroll
                    for (int kx = 0; kx < 5; ++kx) {
                        acc[j][0] = fmaf(w[ky * 5 + kx], in[kx], acc[j][0]);
                        acc[j][1] = fmaf(w[ky * 5 + kx], in[2 + kx], acc[j][1]);
                    }
                }
            }
        }
        const int c1 = 2 * pr, c0 = c1 - 1;
        const bool in0 = pr > 0 && (unsigned)(gx0 + c0) < (unsigned)wl, in1 = c1 < DW && (unsigned)(gx0 + c1) < (unsigned)wl;
#pragma unroll
        for (int j = 0; j < R; ++j) {
            if (r0 + j < DH) {
                const bool rowin = (unsigned)(gy0 + r0 + j) < (unsigned)hl;
                const float v0 = fmaxf(acc[j][0], acc[j][0] * alpha), v1 = fmaxf(acc[j][1], acc[j][1] * alpha);
                if (pr > 0) dst[(r0 + j) * DP + c0] = (rowin && in0) ? v0 : 0.f;
                if (c1 < DW) dst[(r0 + j) * DP + c1] = (rowin && in1) ? v1 : 0.f;
            }
        }
    }
}

// dst (DH x DW at 2x the source resolution, origin (gy0, gx0) even) = act(conv5x5(upsample2(src)) + b) through the four
// parity-folded 3 x 3 kernels wf[py][px][a][b]; output rows (2j, 2j+1) x columns (2n, 2n+1) read src(j + a, n + b).
// Thread = 2 source cells = a 2 x 4 output block (8-byte loads, 16-byte stores at lane stride: conflict-free).
template <int DH, int DW, int DP, int SP, int NT>
__device__ __forceinline__ void hg_up(const float* __restrict__ src, float* __restrict__ dst, const float* __restrict__ wf,
                                      float bias, int gy0, int gx0, int hl, int wl, float alpha) {
    float w[36];
    hg_load_weights<9>(wf, w);
    constexpr int GROUPS = (DW + 3) / 4;
    for (int item = threadIdx.x; item < (DH / 2) * GROUPS; item += NT) {
        const int j = item / GROUPS, n0 = (item - j * GROUPS) * 2;
        float s[3][4];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const float2* row = reinterpret_cast<const float2*>(src + (j + a) * SP + n0);
            const float2 u = row[0], v = row[1];
            s[a][0] = u.x; s[a][1] = u.y; s[a][2] = v.x; s[a][3] = v.y;
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
                        for (int b = 0; b < 3; ++b) acc = fmaf(w[((py * 2 + px) * 3 + a) * 3 + b], s[a][i + b], acc);
                    o[2 * i + px] = fmaxf(acc, acc * alpha);
                }
            const bool rowin = (unsigned)(gy0 + 2 * j + py) < (unsigned)hl;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (!(rowin && (unsigned)(gx0 + 2 * n0 + k) < (unsigned)wl)) o[k] = 0.f;
            *reinterpret_cast<float4*>(dst + (2 * j + py) * DP + 2 * n0) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
}

// wf[py][px][a][b] = sum of the 5 x 5 weights whose row / column lands on source offset a / b for that parity
template <int NT>
__device__ __forceinline__ void hg_fold(const float* __restrict__ w25, float* __restrict__ wf) {
    for (int i = threadIdx.x; i < 36; i += NT) {
        const int b = i % 3, a = (i / 3) % 3, px = (i / 9) % 2, py = i / 18;
        // parity 0: kernel indices {0,1} {2,3} {4};  parity 1: {0} {1,2} {3,4}
        const int ylo = py == 0 ? 2 * a : (a == 0 ? 0 : 2 * a - 1), yhi = py == 0 ? min(2 * a + 1, 4) : (a == 0 ? 0 : 2 * a);
        const int xlo = px == 0 ? 2 * b : (b == 0 ? 0 : 2 * b - 1), xhi = px == 0 ? min(2 * b + 1, 4) : (b == 0 ? 0 : 2 * b);
        float s = 0.f;
        for (int ky = ylo; ky <= yhi; ++ky)
            for (int kx = xlo; kx <= xhi; ++kx) s += w25[ky * 5 + kx];
        wf[i] = s;
    }
}

template <int TH, int TW>
__global__ void __launch_bounds__(hg_threads(TH), TH >= 64 ? 2 : 4) hourglass1_fwd_kernel(const HourglassParams p,
                                                                       const __grid_constant__ CUtensorMap map_x) {
    using G = HG<TH, TW>;
    constexpr int NT = hg_threads(TH);
    extern __shared__ __align__(128) float hg_smem[];
    float* sX = hg_smem;
    float* sD1 = sX + G::XROWS * G::XP;
    float* sD2 = sD1 + G::D1H * G::D1P;
    float* sU2 = sD2 + G::D2H * G::D2P;
    float* sU1 = sX;                                 // over the x block (dead after down_1)
    float* sW = sU2 + G::U2H * G::U2P;               // 5 x (25 weights + bias)
    float* sF = sW + 5 * HG_WSLOT;                   // folded kernels of up_2, up_1

    const int ox0 = blockIdx.x * TW, oy0 = blockIdx.y * TH;
    float* yim = p.y + (int64_t)blockIdx.z * p.H * p.W;
    const int tid = threadIdx.x;

    // ---- level 0: x block -> shared memory.  ONE thread issues one 3-D TMA box (XP x XH x 1 at (ox0 - 16, oy0 - 14,
    // image)); out-of-image elements arrive as zeros (= the padding), completion on an mbarrier.  A per-thread cp.async
    // fill (zero fill through src-size 0) spent 18 % of the kernel's instructions on addresses and bounds (ncu source view).
    uint64_t* bar = reinterpret_cast<uint64_t*>(sF + 2 * 36);          // 8-byte aligned: all segment sizes are even
    if (tid == 0) {
        mbar_init(smem_u32(bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_arrive_expect_tx(smem_u32(bar), (uint32_t)(G::XH * G::XP * sizeof(float)));
        tma_load_3d(smem_u32(sX), &map_x, smem_u32(bar), ox0 - 16, oy0 - 14, (int)blockIdx.z);
    }
    // weights: static level index (a runtime index into p.w[] forces the whole parameter block into local memory)
    if (tid < 26) {
#pragma unroll
        for (int l = 0; l < 5; ++l) sW[l * HG_WSLOT + tid] = tid < 25 ? __ldg(p.w[l] + tid) : __ldg(p.b[l]);
    }
    // the two spare rows the last strip of D1 reads must be finite
    for (int i = tid; i < 2 * G::XP; i += NT) sX[G::XH * G::XP + i] = 0.f;
    __syncthreads();
    mbar_wait(smem_u32(bar), 0);
    hg_fold<NT>(sW + 2 * HG_WSLOT, sF);
    hg_fold<NT>(sW + 3 * HG_WSLOT, sF + 36);
    const int hy0 = oy0 / 2, hx0 = ox0 / 2, qy0 = oy0 / 4, qx0 = ox0 / 4;
    hg_down_pairs<G::D1H, G::D1W, G::D1P, G::XP, 5, NT>(sX, sD1, sW, hy0 - 6, hx0 - 6, p.H / 2, p.W / 2, p.alpha);
    __syncthreads();
    hg_down<G::D2H, G::D2W, G::D2P, G::D1P, (G::D2H % 2 == 0) ? 2 : 4, NT>(sD1, sD2, sW + HG_WSLOT, qy0 - 2, qx0 - 2, p.H / 4, p.W / 4, p.alpha);
    __syncthreads();
    hg_up<G::U2H, G::U2W, G::U2P, G::D2P, NT>(sD2, sU2, sF, sW[2 * HG_WSLOT + 25], hy0 - 2, hx0 - 2, p.H / 2, p.W / 2, p.alpha);
    __syncthreads();
    hg_up<G::U1H, G::U1W, G::U1P, G::U2P, NT>(sU2, sU1, sF + 36, sW[3 * HG_WSLOT + 25], oy0 - 2, ox0 - 2, p.H, p.W, p.alpha);
    __syncthreads();
    // ---- end: y(r, c) = act_end(conv5x5(U1)(r + ky, c + kx) + b); thread = 4 rows x 4 columns (16-byte loads at lane
    // stride: conflict-free; 8 input rows x 32 bytes per 16 outputs, was 6 x 32 per 8), one pass of the 256 threads
    {
        float w[28];
        hg_load_weights<7>(sW + 4 * HG_WSLOT, w);
        const float bias = w[25];
        constexpr int GROUPS = TW / 4, RE = 4;
        for (int item = tid; item < (TH / RE) * GROUPS; item += NT) {
            const int r = (item / GROUPS) * RE, c0 = (item - (item / GROUPS) * GROUPS) * 4;
            float acc[RE][4];
#pragma unroll
            for (int k = 0; k < RE; ++k)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[k][j] = bias;
#pragma unroll
            for (int rr = 0; rr < RE + 4; ++rr) {
                const float4* row = reinterpret_cast<const float4*>(sU1 + (r + rr) * G::U1P + c0);
                const float4 u = row[0], v = row[1];
                const float in[8] = {u.x, u.y, u.z, u.w, v.x, v.y, v.z, v.w};
#pragma unroll
                for (int k = 0; k < RE; ++k) {
                    const int ky = rr - k;
                    if (ky >= 0 && ky < 5) {
#pragma unroll
                        for (int kx = 0; kx < 5; ++kx)
#pragma unroll
                            for (int j = 0; j < 4; ++j) acc[k][j] = fmaf(w[ky * 5 + kx], in[j + kx], acc[k][j]);
                    }
                }
            }
            const int gx = ox0 + c0;
            if (gx < p.W) {                                              // W % 4 == 0: float4 granularity
#pragma unroll
                for (int k = 0; k < RE; ++k) {
                    const int gy = oy0 + r + k;
                    if (gy < p.H)
                        *reinterpret_cast<float4*>(yim + (int64_t)gy * p.W + gx) =
                            make_float4(apply_act_fast(acc[k][0], p.act_end, p.alpha_end),
                                        apply_act_fast(acc[k][1], p.act_end, p.alpha_end),
                                        apply_act_fast(acc[k][2], p.act_end, p.alpha_end),
                                        apply_act_fast(acc[k][3], p.act_end, p.alpha_end));
                }
            }
        }
    }
}

static int hourglass1_unsupported() {
    set_error("hourglass1_fwd: unsupported geometry (H, W must be multiples of 4)");
    return UOCR_ERR_UNSUPPORTED;
}

template <int TH>
static int hourglass1_launch(const HourglassParams& p, const float* x, int64_t n, int64_t h, int64_t wd, cudaStream_t st) {
    constexpr int TW = 128;
    using G = HG<TH, TW>;
    const uint64_t dims[3] = {(uint64_t)wd, (uint64_t)h, (uint64_t)n};
    const uint64_t strides[2] = {(uint64_t)wd * 4, (uint64_t)wd * h * 4};
    const uint32_t box[3] = {(uint32_t)G::XP, (uint32_t)G::XH, 1};
    CUtensorMap map{};
    const int rc = make_tmap_plain_f32(&map, x, 3, dims, strides, box);
    if (rc != UOCR_OK) return rc;
    const size_t smem = sizeof(float) * G::FLOATS;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(hourglass1_fwd_kernel<TH, TW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
        configured = true;
    }
    dim3 grid((unsigned)ceil_div(wd, TW), (unsigned)ceil_div(h, TH), (unsigned)n);
    if (grid.y > 65535) return hourglass1_unsupported();
    hourglass1_fwd_kernel<TH, TW><<<grid, hg_threads(TH), smem, st>>>(p, map);
    UOCR_LAUNCHED("hourglass1_fwd");
    return UOCR_OK;
}

// The kernel is the same in both math modes: its FFMA levels are exact FP32.  A tensor map that cannot be built
// returns its own error and message.
int hourglass1_fwd(const float* x, const float* const* w, const float* const* b, float* y, int64_t n, int64_t h,
                   int64_t wd, float alpha, int act_end, float alpha_end, cudaStream_t st) {
    if (h % 4 || wd % 4 || n > 65535 || alpha < 0.f || alpha > 1.f) return hourglass1_unsupported();
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) return hourglass1_unsupported();
    HourglassParams p{};
    p.x = x; p.y = y;
    for (int l = 0; l < 5; ++l) { p.w[l] = w[l]; p.b[l] = b[l]; }
    p.H = (int)h; p.W = (int)wd; p.alpha = alpha; p.act_end = act_end; p.alpha_end = alpha_end;
    // 64-row blocks with 512 threads where they still fill the machine twice over (2 CTAs / SM): 7 % fewer halo FMAs
    // and half as many block prologues, 115.7 -> 111.6 us per 64 tiles.
    const int64_t blocks64 = n * ceil_div(h, 64) * ceil_div(wd, 128);
    if (blocks64 >= 148 * 2 * 2) return hourglass1_launch<64>(p, x, n, h, wd, st);
    return hourglass1_launch<32>(p, x, n, h, wd, st);
}

}  // namespace uocr

static int hourglass1_entry(const float* x, const float* const* weights, const float* const* biases, float* y, int64_t n,
                            int64_t h, int64_t w, float alpha, int act_end, float alpha_end, int math_mode, void* stream) {
    using namespace uocr;
    UOCR_REQUIRE(x && y && weights && biases, "NULL pointer");
    for (int l = 0; l < 5; ++l) UOCR_REQUIRE(weights[l] && biases[l], "NULL weight pointer (level %d)", l);
    UOCR_REQUIRE(n > 0 && h > 0 && w > 0 && h < (1 << 30) && w < (1 << 30), "bad dimension");
    UOCR_REQUIRE(act_end >= UOCR_ACT_NONE && act_end <= UOCR_ACT_SIGMOID, "unknown activation %d", act_end);
    UOCR_REQUIRE(math_mode == UOCR_MATH_FP32 || math_mode == UOCR_MATH_TF32, "unknown math mode %d", math_mode);
    return hourglass1_fwd(x, weights, biases, y, n, h, w, alpha, act_end, alpha_end, as_stream(stream));
}

extern "C" int uocr_hourglass1_fwd(const float* x, const float* const* weights, const float* const* biases, float* y,
                                   int64_t n, int64_t h, int64_t w, float alpha, int act_end, float alpha_end,
                                   void* stream) {
    return hourglass1_entry(x, weights, biases, y, n, h, w, alpha, act_end, alpha_end, UOCR_MATH_FP32, stream);
}

extern "C" int uocr_hourglass1_fwd_mode(const float* x, const float* const* weights, const float* const* biases, float* y,
                                        int64_t n, int64_t h, int64_t w, float alpha, int act_end, float alpha_end,
                                        int math_mode, void* stream) {
    return hourglass1_entry(x, weights, biases, y, n, h, w, alpha, act_end, alpha_end, math_mode, stream);
}

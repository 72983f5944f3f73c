// 5 x 5 / stride 1 / padding 2 convolutions with 4 input channels on the tensor cores (Line up_2, up_1, end:
// Cin = 4, Cout = 4 or 2, optionally reading their input through a folded Upsample2D(2)).
//
//   replaces: Convolutional2D._forward (convolutional.py:62-99) [+ Upsample2D._forward (upsample.py:21-39) in front,
//   + LeakyRelu / Sigmoid._forward (layers.py:390-415) behind] for make_line's up and end blocks (my_model/model.py:192-248).
//
// As an implicit GEMM these layers have N = Cout = 4: useless for tcgen05.  Like the Monochrome pair kernel
// (conv_pair_tc.cu) this one contracts over what a thread already holds and keeps N full:
//
//   GEMM   Z[r'][c, (ky, co)] = sum_{kx, ci} x[r', c + kx - 2, ci] . w[ky, kx, ci, co]     for every INPUT row r'
//          M = 128 pixels of the row, K = 5 x 4 (+ a constant 1 that carries the bias in the ky = 2 block) = 24,
//          N = 5 x Cout = 20 (10) -> 32 (16)
//   shift  y[r, c, co] = act(sum_ky Z[r + ky - 2][c, (ky, co)])                            vertical only: registers
//
// i.e. the horizontal taps and the input channels are the contraction, the vertical taps ride along as extra output
// columns and are summed while the thread walks down the rows (4 rolling partial sums x Cout).  Three tcgen05.mma
// (128 x 32 x 8, kind::tf32) per 128 pixels replace 128 x 400 FFMA.  lane = pixel: a thread loads the five 16-byte
// pixels of its window straight from global memory and tcgen05.st's them into its TMEM lane (the A operand never
// touches shared memory), the MMA leaves Z in TMEM, the thread tcgen05.ld's its 20 values back.  Only the 3 KB weight
// operand sits in shared memory (K-major, no swizzle: one 16-byte chunk = the 4 input channels of one kx).
//
// Numerics: activations are consumed as TF32 by truncation inside the tensor core, made unbiased by scaling the
// weights (not the bias) with (1 + 2^-11); weights rounded to nearest; FP32 accumulation.
#include "conv_common.cuh"
#include "tc_ptx.cuh"

namespace uocr {

constexpr int RT_THREADS = 128;
constexpr int RT_R = 2;                       // input rows per pipeline step (128 TMEM columns: 4 CTAs per SM)
constexpr int RT_SLOT = 64;                   // TMEM columns per row in flight: A at +0 (24), Z at +32 (32)

struct RowTcParams {
    const float* x; const float* w; const float* b; float* y;
    int H, W;                                 // logical (upsampled) input size = output size
    int strips, bands, rb;
    int64_t items;
    int steps;
    int act; float alpha;
};

__device__ __forceinline__ void rt_st4(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void rt_ld4(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void rt_ld2(uint32_t taddr, uint32_t* r) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ bool rt_elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void rt_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity), "r"(20000u) : "memory");
    } while (!done);
}

template <int COUT, bool UPS>
__global__ void __launch_bounds__(RT_THREADS, 4) conv55_row_tc_kernel(const RowTcParams p) {
    constexpr int NPAD = COUT == 4 ? 32 : 16;
    constexpr int NZ = 5 * COUT;                          // useful Z columns
    __shared__ __align__(128) float s_b[6 * NPAD * 4];    // chunk kq (= kx, 5 = bias): NPAD rows (n) x 4 floats (ci)
    __shared__ __align__(8) uint64_t s_bar[2];
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);

    for (int i = tid; i < 6 * NPAD * 4; i += RT_THREADS) {
        const int kq = i / (NPAD * 4), n = (i / 4) % NPAD, kk = i & 3;
        const int ky = n / COUT, co = n - ky * COUT;
        float v = 0.f;
        if (n < NZ) {
            if (kq < 5) v = __ldg(p.w + ((ky * 5 + kq) * 4 + kk) * COUT + co) * (1.f + 1.f / 2048.f);
            else if (kk == 0 && ky == 2 && p.b) v = __ldg(p.b + co);   // A column 20 is the constant 1
        }
        s_b[i] = round_tf32(v);
    }
    if (tid == 0) {
        mbar_init(smem_u32(&s_bar[0]), RT_THREADS);       // windows stored by every thread
        mbar_init(smem_u32(&s_bar[1]), 1);                // MMAs committed
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(&s_tmem)), "r"((uint32_t)(RT_R * RT_SLOT)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tlane = s_tmem + ((uint32_t)(warp * 32) << 16);
    {   // A columns 20 .. 23 = {1, 0, 0, 0}: written once, the windows only ever overwrite columns 0 .. 19
        const uint32_t one[4] = {__float_as_uint(1.f), 0u, 0u, 0u};
#pragma unroll
        for (int r = 0; r < RT_R; ++r) rt_st4(tlane + (uint32_t)(RT_SLOT * r + 20), one);
        tc_wait_st();
    }

    int64_t item = (int64_t)blockIdx.x * 4 + warp;
    const bool active = item < p.items;
    if (!active) item = p.items - 1;
    const int strip = (int)(item % p.strips);
    const int64_t rest = item / p.strips;
    const int band = (int)(rest % p.bands);
    const int64_t img = rest / p.bands;
    const int c = strip * 32 + lane;                      // output column = centre of the window
    const bool colvalid = active && c < p.W;
    const int oy0 = band * p.rb;
    const int nrows = min(p.H - oy0, p.rb);
    const int sW = UPS ? p.W / 2 : p.W, sH = UPS ? p.H / 2 : p.H;       // stored size
    const float4* xim = reinterpret_cast<const float4*>(p.x) + img * (int64_t)sH * sW;
    // &y[output row completed by the band's first input row = oy0 - 4] (stores are predicated)
    float* yout = p.y + ((img * p.H + oy0 - 4) * (int64_t)p.W + c) * COUT;
    bool cok[5];
    int coff[5];
#pragma unroll
    for (int kx = 0; kx < 5; ++kx) {
        const int cc = c + kx - 2;
        cok[kx] = active && cc >= 0 && cc < p.W;
        coff[kx] = UPS ? (cc >> 1) : cc;
    }

    uint32_t xq[RT_R][5][4];                               // windows of the step's input rows (prefetched)
    auto load_rows = [&](int k) {
#pragma unroll
        for (int r = 0; r < RT_R; ++r) {
            const int ri = oy0 - 2 + RT_R * k + r;
            const bool rowok = ri >= 0 && ri < p.H;
            const float4* row = xim + (int64_t)(rowok ? (UPS ? ri >> 1 : ri) : 0) * sW;
#pragma unroll
            for (int kx = 0; kx < 5; ++kx) {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (rowok && cok[kx]) v = __ldg(row + coff[kx]);
                xq[r][kx][0] = __float_as_uint(v.x); xq[r][kx][1] = __float_as_uint(v.y);
                xq[r][kx][2] = __float_as_uint(v.z); xq[r][kx][3] = __float_as_uint(v.w);
            }
        }
    };
    load_rows(0);

    float S[4][COUT];
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int co = 0; co < COUT; ++co) S[j][co] = 0.f;
    const uint32_t bars = smem_u32(&s_bar[0]);
    const uint32_t sb = smem_u32(s_b);
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(NPAD >> 3) << 17) | ((128u >> 4) << 24);

#pragma unroll 1
    for (int k = 0; k < p.steps; ++k) {
        const uint32_t par = (uint32_t)(k & 1);
        // ---- phase A: windows -> TMEM
#pragma unroll
        for (int r = 0; r < RT_R; ++r)
#pragma unroll
            for (int kx = 0; kx < 5; ++kx) rt_st4(tlane + (uint32_t)(RT_SLOT * r + 4 * kx), xq[r][kx]);
        tc_wait_st();
        tc_fence_before();
        mbar_arrive(bars);
        if (k + 1 < p.steps) load_rows(k + 1);             // in flight while the MMAs run
        if (warp == 0) {
            rt_wait(bars, par);
            tc_fence_after();
            if (rt_elect_one()) {
                uint32_t tb;
                asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tb) : "r"(smem_u32(&s_tmem)));
#pragma unroll
                for (int r = 0; r < RT_R; ++r)
#pragma unroll
                    for (int m = 0; m < 3; ++m)
                        tc_mma_tf32_ts(tb + (uint32_t)(RT_SLOT * r + 32), tb + (uint32_t)(RT_SLOT * r + 8 * m),
                                       make_kmajor_nosw_desc(sb + (uint32_t)(2 * m) * (NPAD * 16), NPAD * 16, 128), idesc, m);
                tc_commit(bars + 8);
            }
            __syncwarp();
        }
        // ---- phase C: Z -> rolling vertical sums -> output rows
        rt_wait(bars + 8, par);
        tc_fence_after();
#pragma unroll
        for (int r = 0; r < RT_R; ++r) {
            uint32_t z[NZ];
            const uint32_t tz = tlane + (uint32_t)(RT_SLOT * r + 32);
            if (COUT == 4) { tc_ld16_nowait(tz, z); rt_ld4(tz + 16, z + 16); }
            else { tc_ld8_nowait(tz, z); rt_ld2(tz + 8, z + 8); }
            tc_wait_ld();
            const int orow = RT_R * k + r - 4;             // output row (within the band) completed by this input row
            float v[COUT];
#pragma unroll
            for (int co = 0; co < COUT; ++co) {
                v[co] = apply_act_fast(S[0][co] + __uint_as_float(z[4 * COUT + co]), p.act, p.alpha);
                S[0][co] = S[1][co] + __uint_as_float(z[3 * COUT + co]);
                S[1][co] = S[2][co] + __uint_as_float(z[2 * COUT + co]);
                S[2][co] = S[3][co] + __uint_as_float(z[1 * COUT + co]);
                S[3][co] = __uint_as_float(z[co]);
            }
            if (colvalid && orow >= 0 && orow < nrows) {
                float* dst = yout + (int64_t)(RT_R * k + r) * p.W * COUT;
                if (COUT == 4) *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
                else *reinterpret_cast<float2*>(dst) = make_float2(v[0], v[1]);
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                     ::"r"(s_tmem), "r"((uint32_t)(RT_R * RT_SLOT)) : "memory");
    }
}

int conv55_row_tc(const ConvGeom& g, const float* x, const float* w, const float* b, float* y, int act, float alpha,
                  cudaStream_t st) {
    if (g.kh != 5 || g.kw != 5 || g.sh != 1 || g.sw != 1 || g.ph != 2 || g.pw != 2 || g.cin != 4) return UOCR_ERR_UNSUPPORTED;
    if ((g.cout != 4 && g.cout != 2) || g.padding_value != 0.f || (g.ups != 1 && g.ups != 2))
        return UOCR_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) return UOCR_ERR_UNSUPPORTED;
    // output rows per band: tall bands amortise the 4 halo rows, short ones give enough CTAs for a few waves
    // (4 resident per SM); measured on the Line shapes: 12 rows beat 28 and 60 there
    RowTcParams p{};
    p.x = x; p.w = w; p.b = g.bias ? b : nullptr; p.y = y;          // no bias: the stride-1 dgrad on flipped weights
    p.H = g.h; p.W = g.w;
    p.strips = (int)ceil_div(g.w, 32);
    int rb = 12;
    for (int cand : {60, 28}) {
        if ((int64_t)g.n * ceil_div(g.h, cand) * p.strips / 4 >= 3 * 4 * 148) { rb = cand; break; }
    }
    p.rb = g.h < rb ? g.h : rb;
    p.bands = (int)ceil_div(g.h, p.rb);
    p.items = (int64_t)g.n * p.bands * p.strips;
    p.steps = (p.rb + 4 + RT_R - 1) / RT_R;
    p.act = act; p.alpha = alpha;
    const int64_t ctas = ceil_div(p.items, 4);
    if (ctas > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    const unsigned grid = (unsigned)ctas;
    if (g.cout == 4) {
        if (g.ups == 2) conv55_row_tc_kernel<4, true><<<grid, RT_THREADS, 0, st>>>(p);
        else conv55_row_tc_kernel<4, false><<<grid, RT_THREADS, 0, st>>>(p);
    } else {
        if (g.ups == 2) conv55_row_tc_kernel<2, true><<<grid, RT_THREADS, 0, st>>>(p);
        else conv55_row_tc_kernel<2, false><<<grid, RT_THREADS, 0, st>>>(p);
    }
    UOCR_LAUNCHED("conv55_row_tc");
    return UOCR_OK;
}

}  // namespace uocr

// Monochrome conv pair on the tensor cores, both convolutions, operands resident in TENSOR MEMORY.
//
//   y = act2(conv3x3(act1(conv3x3(x, w1) + b1), w2) + b2)        1 -> 16 -> 1 channels, padding 1, stride 1
//   replaces: make_monochrome's conv_1 -> leaky_relu_1 -> conv_2 -> sigmoid (my_model/model.py:119-122), i.e.
//   Convolutional2D._forward (convolutional.py:62-99) twice + LeakyRelu/Sigmoid._forward (layers.py:390-415).
//
// The pair costs 288 FMA per pixel; on the CUDA cores (conv_fast.cu) that is FFMA-issue bound (0.44 ms for 64
// tiles of 496 x 736, FMA pipe 62 % busy).  The obvious implicit GEMM (M = pixels, K = taps x channels, N = Cout)
// wastes the tensor core because Cout = 1.  This kernel turns BOTH convolutions into GEMMs whose N dimension is
// full, by contracting over what is small and shifting afterwards:
//
//   GEMM 1   H[p, c]  = sum_t X9[p, t] . w1[t, c]          M = 128 hidden pixels, K = 16 (9 taps of the 3 x 3
//                                                          window of x around p, a constant 1 that carries b1,
//                                                          6 zeros), N = 16 hidden channels
//   act1     A2[p, c] = max(H, alpha H)                     (LeakyReLU, in registers)
//   GEMM 2   Z[p, t]  = sum_c A2[p, c] . w2[t, c]          K = 16 channels, N = 16 (9 taps used): the
//                                                          contribution of hidden pixel p to its 9 neighbours
//   shift    y[q]     = act2(b2 + sum_t Z[q + off(t), t])   9 adds per pixel instead of 144 FMA
//
// Four tcgen05.mma (128 x 16 x 8, kind::tf32, 8 cycles each) per 128 hidden pixels replace 128 x 288 FFMA.  The A
// operands never touch shared memory: lane = hidden pixel, so each thread writes the 3 x 3 window it already holds
// in registers into its own TMEM lane with tcgen05.st, GEMM 1 reads A from TMEM and leaves H in TMEM, the thread
// reads its H row back with tcgen05.ld, applies act1, stores A2 in place, GEMM 2 reads it from TMEM and writes Z
// over the dead X9 columns (32 TMEM columns per hidden row in flight).  B operands (w1 + b1, w2: 2 x 1 KB) sit in
// shared memory in the K-major no-swizzle layout.
//
// Geometry: a warp owns a strip of 32 hidden columns (30 output columns + 1 halo column each side) and streams
// down a band of RB output rows; the vertical part of the shift is a rolling set of 3 x 3 partial sums in
// registers, the horizontal part two warp shuffles per output pixel.  The four warps of a CTA (4 strips, together
// the M = 128 rows of one MMA) advance in lock step, PM_R = 4 hidden rows per pipeline step:
//   st X9 -> [barA] -> MMA1 -> [barD1] -> ld H, act, st A2 -> [barA2] -> MMA2 -> [barD2] -> ld Z, shift, store
// Each hop costs ~500 cycles (measured, tools/tmem_probe.cu), so latency is hidden by occupancy: 4 CTAs per SM x
// 128 TMEM columns = all 512 columns, 16 hidden rows in flight per SM (TMEM capacity is what bounds it).
//
// Numerics: x and the weights are rounded to TF32 (cvt.rna); H is consumed as TF32 by truncation inside the
// tensor core, made unbiased by scaling w1 and b1 with (1 + 2^-11) when the B operand is built (act1 is positively
// homogeneous); accumulation is FP32.  Tolerance in tests: 1e-3 of the output range (TF32 mode).
#include "conv_common.cuh"
#include "tc_ptx.cuh"

namespace uocr {

constexpr int PM_OUT = 30;            // output columns per warp strip
constexpr int PM_THREADS = 160;       // 4 compute warps = the 128 rows of one UMMA, + 1 MMA-issuing warp
constexpr int PM_R = 4;               // hidden rows per pipeline step
constexpr int PM_NS = PM_R + 2;       // x rows live during a step = ring slots
constexpr int PM_TMEM_COLS = 32 * PM_R;   // per hidden row in flight: 16 columns X9 / Z + 16 columns H / A2

struct PairTcParams {
    const float* x; const float* w1; const float* b1; const float* w2; const float* b2; float* y;
    int H, W;
    int strips, bands, rb;            // strips per image row, bands per image, output rows per band
    int64_t items;                    // n * bands * strips
    int steps;                        // ceil((rb + 2) / PM_R)
    float alpha1, alpha2;
};

// Per-thread state.  The x window is a ring of PM_NS image rows; a slot holds {x[., hc-1], x[., hc], x[., hc+1],
// one} as one register quad, so the 3 x 3 window of a hidden row goes to TMEM as three tcgen05.st.x4 (columns
// 4a .. 4a+3 for window row a) without any register shuffling.  `one` (1 for a hidden pixel inside the image,
// else 0) multiplies b1 in B1's row k = 3; rows k = 7, 11 .. 15 of B1 are zero.
struct PairTcState {
    uint32_t xw[PM_NS][4];
    float acc[3][3];                  // rolling partial sums: [output row % 3][kx]
};

// ring slot <- x[xr, hc - 1 .. hc + 1] (xrow = &x[xr, hc]); zero outside the image / for idle lanes
__device__ __forceinline__ void pm_load_row(const float* __restrict__ xrow, bool rowok, bool c0, bool c1, bool c2,
                                            uint32_t* dst) {
    dst[0] = (rowok && c0) ? __float_as_uint(__ldg(xrow - 1)) : 0u;
    dst[1] = (rowok && c1) ? __float_as_uint(__ldg(xrow)) : 0u;
    dst[2] = (rowok && c2) ? __float_as_uint(__ldg(xrow + 1)) : 0u;
}
// FP32 -> TF32 round to nearest: the tensor core ignores the low 13 mantissa bits, so adding half an ulp is enough
// (volatile: keeps the add where it is written -- hoisted next to the prefetching load it would stall the warp)
__device__ __forceinline__ void pm_round_row(uint32_t* q) {
    asm volatile("add.u32 %0, %0, 0x1000;\n\tadd.u32 %1, %1, 0x1000;\n\tadd.u32 %2, %2, 0x1000;"
                 : "+r"(q[0]), "+r"(q[1]), "+r"(q[2]));
}
__device__ __forceinline__ void tc_st4_nowait(uint32_t taddr, const uint32_t* r) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}
__device__ __forceinline__ void tc_st16_zero(uint32_t taddr) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
        ::"r"(taddr), "r"(0u) : "memory");
}
__device__ __forceinline__ uint32_t pm_tmem_base(uint32_t slot_addr) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(slot_addr));
    return v;
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// mbarrier wait whose failed probes sleep in hardware (suspend-time hint) instead of spinning through issue slots
__device__ __forceinline__ void mbar_wait_sleepy(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity), "r"(20000u) : "memory");
    } while (!done);
}

// Barriers, per half h of a step (rows 2h, 2h + 1): [0] windows stored (128 arrivals), [1] MMA1 committed,
// [2] A2 stored (128 arrivals), [3] MMA2 committed.  Every barrier completes once per step: parity = k & 1.
__device__ __forceinline__ uint32_t pm_bar(uint32_t bars, int half, int which) { return bars + (uint32_t)(half * 4 + which) * 8u; }

// One pipeline step = hidden rows i0 = PM_R k .. i0 + PM_R - 1 of the band, as TWO half-steps (rows 0-1, rows 2-3)
// whose phases are interleaved so that a warp computes on one half while the other half's MMAs are in flight:
//   A(0) A(1) | B(0) B(1) | C(0) C(1)        (A: windows -> TMEM, B: H -> act -> A2, C: Z -> shift-add -> output)
// The MMAs are issued by a dedicated fifth warp (pm_issuer), so no compute warp ever waits for the other three.
// PX = i0 % PM_NS (x ring phase) and PH = i0 % 3 (partial-sum ring phase) are compile-time: static register indices.
template <int PX, int PH, bool LEAKY, bool SIGMOID>
__device__ __forceinline__ void pm_step(const PairTcParams& p, PairTcState& s, int k, const float* __restrict__& xnext,
                                        float* __restrict__& ynext, int hr0, int nrows, bool c0, bool c1, bool c2,
                                        bool store_lane, uint32_t tlane, uint32_t bars, float bias2) {
    const uint32_t par = (uint32_t)(k & 1);
    const int i0 = PM_R * k;
    // ---------------- phase A: 3 x 3 windows -> TMEM (GEMM 1's A operand)
#pragma unroll
    for (int half = 0; half < 2; ++half) {
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int r = 2 * half + rr;
            const int hr = hr0 + i0 + r;
            const uint32_t tx = tlane + (uint32_t)(32 * r);
            if (hr >= 0 && hr < p.H) {                    // warp-uniform
#pragma unroll
                for (int a = 0; a < 3; ++a) tc_st4_nowait(tx + 4 * a, s.xw[(PX + r + a) % PM_NS]);
            } else {                                      // hidden rows outside the image are conv_2's zero padding
                tc_st16_zero(tx);
            }
        }
        tc_wait_st();
        tc_fence_before();
        mbar_arrive(pm_bar(bars, half, 0));
    }
    // Prefetch the PM_R x rows the NEXT step adds to the window, straight into the ring slots that died with this
    // step's stores; their latency hides behind this step's waits; they are rounded to TF32 at the end of phase C.
#pragma unroll
    for (int j = 0; j < PM_R; ++j) {
        const int xr = hr0 - 1 + i0 + PM_NS + j;
        pm_load_row(xnext, xr >= 0 && xr < p.H, c0, c1, c2, s.xw[(PX + j) % PM_NS]);
        xnext += p.W;
    }
    // ---------------- phase B: H -> act1 -> A2 (in place)
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        mbar_wait_sleepy(pm_bar(bars, half, 1), par);
        tc_fence_after();
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int r = 2 * half + rr;
            uint32_t h[16];
            tc_ld16_nowait(tlane + (uint32_t)(32 * r + 16), h);
            tc_wait_ld();
            if (LEAKY) {                                   // max(h, alpha h): packed multiply (FMUL2) + FMNMX
                const uint32_t ab = __float_as_uint(p.alpha1);
#pragma unroll
                for (int c = 0; c < 16; c += 2) {
                    uint32_t t0, t1;
                    asm("{\n\t.reg .b64 x, y, r;\n\tmov.b64 x, {%2, %3};\n\tmov.b64 y, {%4, %4};\n\t"
                        "mul.rn.f32x2 r, x, y;\n\tmov.b64 {%0, %1}, r;\n\t}"
                        : "=r"(t0), "=r"(t1) : "r"(h[c]), "r"(h[c + 1]), "r"(ab));
                    h[c] = __float_as_uint(fmaxf(__uint_as_float(h[c]), __uint_as_float(t0)));
                    h[c + 1] = __float_as_uint(fmaxf(__uint_as_float(h[c + 1]), __uint_as_float(t1)));
                }
            }
            tc_st16_nowait(tlane + (uint32_t)(32 * r + 16), h);
        }
        tc_wait_st();
        tc_fence_before();
        mbar_arrive(pm_bar(bars, half, 2));
    }
    // ---------------- phase C: Z -> rolling shift-and-add -> output rows
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        mbar_wait_sleepy(pm_bar(bars, half, 3), par);
        tc_fence_after();
#pragma unroll
        for (int rr = 0; rr < 2; ++rr) {
            const int r = 2 * half + rr;
            const int ph = (PH + r) % 3;
            uint32_t z[9];
            tc_ld8_nowait(tlane + (uint32_t)(32 * r), z);
            tc_ld1_nowait(tlane + (uint32_t)(32 * r + 8), z + 8);
            tc_wait_ld();
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                s.acc[(ph + 2) % 3][kx] = __uint_as_float(z[kx]);             // ky = 0: opens output row i + 2
                s.acc[(ph + 1) % 3][kx] += __uint_as_float(z[3 + kx]);        // ky = 1: output row i + 1
                s.acc[ph][kx] += __uint_as_float(z[6 + kx]);                  // ky = 2: completes output row i
            }
            // y[oy, ox] = b2 + Z-sum of hidden columns ox - 1 (kx = 0), ox (kx = 1), ox + 1 (kx = 2)
            const float left = __shfl_up_sync(0xffffffffu, s.acc[ph][0], 1);
            const float right = __shfl_down_sync(0xffffffffu, s.acc[ph][2], 1);
            float v = s.acc[ph][1] + left + right + bias2;
            if (SIGMOID) v = __fdividef(1.f, 1.f + __expf(-v));
            else if (p.alpha2 != 1.f) v = v >= 0.f ? v : v * p.alpha2;        // LeakyReLU; alpha2 == 1: no activation
            const int orow = i0 + r - 2;                  // output row of the band completed by hidden row i
            if (store_lane && orow >= 0 && orow < nrows) ynext[(int64_t)r * p.W] = v;
        }
    }
    ynext += (int64_t)PM_R * p.W;
#pragma unroll
    for (int j = 0; j < PM_R; ++j) pm_round_row(s.xw[(PX + j) % PM_NS]);
}

// The fifth warp: waits for each half's operands and issues its MMAs (one elected lane).
__device__ __forceinline__ void pm_issuer(int steps, uint32_t tmem_base, uint32_t bars, uint32_t sb1, uint32_t sb2) {
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((16u >> 3) << 17) | ((128u >> 4) << 24);
#pragma unroll 1
    for (int k = 0; k < steps; ++k) {
        const uint32_t par = (uint32_t)(k & 1);
#pragma unroll
        for (int g = 0; g < 2; ++g) {                     // g = 0: GEMM 1 (windows -> H), g = 1: GEMM 2 (A2 -> Z)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                mbar_wait_sleepy(pm_bar(bars, half, g == 0 ? 0 : 2), par);
                tc_fence_after();
                if (elect_one()) {
#pragma unroll
                    for (int rr = 0; rr < 2; ++rr) {
                        const uint32_t t = tmem_base + (uint32_t)(32 * (2 * half + rr));
#pragma unroll
                        for (int m = 0; m < 2; ++m) {
                            if (g == 0)
                                tc_mma_tf32_ts(t + 16, t + (uint32_t)(8 * m),
                                               make_kmajor_nosw_desc(sb1 + (uint32_t)(2 * m) * 256u, 256, 128), idesc, m);
                            else
                                tc_mma_tf32_ts(t, t + (uint32_t)(16 + 8 * m),
                                               make_kmajor_nosw_desc(sb2 + (uint32_t)(2 * m) * 256u, 256, 128), idesc, m);
                        }
                    }
                    tc_commit(pm_bar(bars, half, g == 0 ? 1 : 3));
                }
                __syncwarp();
            }
        }
    }
}

template <bool LEAKY, bool SIGMOID>
__global__ void __launch_bounds__(PM_THREADS, 4) conv3x3_pair_tmem_kernel(const PairTcParams p) {
    __shared__ __align__(128) float s_b1[256];          // chunk kq: 16 rows (n = channel) x 4 floats (k = 4 kq + kk)
    __shared__ __align__(128) float s_b2[256];          // chunk kq: 16 rows (n = tap) x 4 floats (k = channel)
    __shared__ __align__(8) uint64_t s_bar[8];
    __shared__ uint32_t s_tmem;
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);      // warp-uniform for the compiler

    for (int i = tid; i < 256; i += PM_THREADS) {
        const int kq = i >> 6, n = (i & 63) >> 2, kk = i & 3;
        // B1[n = channel][k = 4 a + b]: window row a = kq < 3, column b < 3; k = 3 carries b1; scaled so that the
        // tensor core's truncation of H to TF32 is unbiased
        float v = 0.f;
        if (kq < 3 && kk < 3) v = __ldg(p.w1 + (kq * 3 + kk) * 16 + n);
        if (kq == 0 && kk == 3) v = __ldg(p.b1 + n);
        s_b1[i] = round_tf32(v * (1.f + 1.f / 2048.f));
        s_b2[i] = n < 9 ? round_tf32(__ldg(p.w2 + n * 16 + kq * 4 + kk)) : 0.f;
    }
    if (tid == 0) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            mbar_init(smem_u32(&s_bar[half * 4 + 0]), 128);      // windows stored by every compute thread
            mbar_init(smem_u32(&s_bar[half * 4 + 1]), 1);        // MMA1 committed
            mbar_init(smem_u32(&s_bar[half * 4 + 2]), 128);      // A2 stored
            mbar_init(smem_u32(&s_bar[half * 4 + 3]), 1);        // MMA2 committed
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // s_b1 / s_b2 are read by the async proxy
    if (warp == 4) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(&s_tmem)), "r"((uint32_t)PM_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t bars = smem_u32(&s_bar[0]);

    if (warp == 4) {
        pm_issuer(p.steps, s_tmem, bars, smem_u32(s_b1), smem_u32(s_b2));
    } else {
        const uint32_t tlane = s_tmem + ((uint32_t)(warp * 32) << 16);
        // columns 12 .. 15 of every X block are never stored by phase A (zero weights) but must hold finite numbers
#pragma unroll
        for (int r = 0; r < PM_R; ++r) tc_st16_zero(tlane + (uint32_t)(32 * r));
        tc_wait_st();

        // work item of this warp: (image, band, strip); warps past the end run on zeros and store nothing
        int64_t item = (int64_t)blockIdx.x * 4 + warp;
        const bool active = item < p.items;
        if (!active) item = p.items - 1;
        const int strip = (int)(item % p.strips);
        const int64_t rest = item / p.strips;
        const int band = (int)(rest % p.bands);
        const int64_t img = rest / p.bands;
        const int hc = strip * PM_OUT - 1 + lane;       // hidden column of this lane
        const bool c1 = active && hc >= 0 && hc < p.W;  // hidden pixels outside the image are zero padding
        const bool c0 = c1 && hc - 1 >= 0, c2 = c1 && hc + 1 < p.W;
        const bool store_lane = c1 && lane >= 1 && lane <= PM_OUT;
        const int hr0 = band * p.rb - 1;                // first hidden row of the band
        const int nrows = min(p.H - band * p.rb, p.rb); // output rows of the band
        const float bias2 = __ldg(p.b2);
        // &x[first x row of the band = hr0 - 1, hc] (never dereferenced outside the image)
        const float* xnext = p.x + (img * p.H + (hr0 - 1)) * p.W + hc;
        // ynext = &y[output row completed by the step's first hidden row = band row - 2, hc] (stores are predicated)
        float* ynext = p.y + (img * p.H + (hr0 - 1)) * p.W + hc;

        PairTcState s;
#pragma unroll
        for (int a = 0; a < 3; ++a)
#pragma unroll
            for (int b = 0; b < 3; ++b) s.acc[a][b] = 0.f;
#pragma unroll
        for (int a = 0; a < PM_NS; ++a) {
            const int xr = hr0 - 1 + a;
            pm_load_row(xnext, xr >= 0 && xr < p.H, c0, c1, c2, s.xw[a]);
            // (blockIdx.y is 0, which the compiler cannot know: one physical register per slot instead of one shared
            // register, so that every quad is contiguous for tcgen05.st.x4 without moves)
            s.xw[a][3] = (c1 ? __float_as_uint(1.f) : 0u) ^ (blockIdx.y * (uint32_t)(a + 1));
            xnext += p.W;
        }
#pragma unroll
        for (int a = 0; a < PM_NS; ++a) pm_round_row(s.xw[a]);

#define PM_STEP(PX, PH, K) \
        pm_step<PX, PH, LEAKY, SIGMOID>(p, s, K, xnext, ynext, hr0, nrows, c0, c1, c2, store_lane, tlane, bars, bias2)
        static_assert(PM_R == 4 && PM_NS == 6, "the unrolled phases below are (4k) % 6 and (4k) % 3");
#pragma unroll 1
        for (int k = 0; k < p.steps; k += 3) {
            PM_STEP(0, 0, k);
            if (k + 1 < p.steps) PM_STEP(4, 1, k + 1);
            if (k + 2 < p.steps) PM_STEP(2, 2, k + 2);
        }
#undef PM_STEP
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                     ::"r"(s_tmem), "r"((uint32_t)PM_TMEM_COLS) : "memory");
    }
}

int conv3x3_pair_tmem(const float* x, const float* w1, const float* b1, const float* w2, const float* b2, float* y,
                      int64_t n, int64_t h, int64_t w, int c1, int act1, float alpha1, int act2, float alpha2,
                      cudaStream_t st) {
    if (c1 != 16) return UOCR_ERR_UNSUPPORTED;
    const bool leaky = act1 == UOCR_ACT_LEAKY;
    if (!(act1 == UOCR_ACT_NONE || (leaky && alpha1 >= 0.f && alpha1 <= 1.f))) return UOCR_ERR_UNSUPPORTED;
    // output rows per band: a multiple of PM_R minus the 2 halo rows keeps every step full
    // (measured on 64 tiles of 496 x 736: 126-row bands 0.133 ms, 62 rows 0.139, 30 rows 0.155; shorter bands only
    // when there would otherwise be fewer than ~2 waves of CTAs, 4 resident per SM)
    PairTcParams p{};
    p.x = x; p.w1 = w1; p.b1 = b1; p.w2 = w2; p.b2 = b2; p.y = y;
    p.H = (int)h; p.W = (int)w;
    p.strips = (int)ceil_div(w, PM_OUT);
    int rb = 126;
    while (rb > 14 && n * ceil_div(h, rb) * p.strips / 4 < 2 * 4 * 148) rb = rb / 2 - 1;    // 126, 62, 30, 14
    p.rb = (int)(h < rb ? h : rb);
    p.bands = (int)ceil_div(h, p.rb);
    p.items = n * p.bands * p.strips;
    p.steps = (p.rb + 2 + PM_R - 1) / PM_R;
    p.alpha1 = alpha1;
    p.alpha2 = act2 == UOCR_ACT_LEAKY ? alpha2 : 1.f;
    const int64_t ctas = ceil_div(p.items, 4);
    if (ctas > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    const unsigned grid = (unsigned)ctas;
    if (act2 == UOCR_ACT_SIGMOID) {
        if (leaky) conv3x3_pair_tmem_kernel<true, true><<<grid, PM_THREADS, 0, st>>>(p);
        else conv3x3_pair_tmem_kernel<false, true><<<grid, PM_THREADS, 0, st>>>(p);
    } else {
        if (leaky) conv3x3_pair_tmem_kernel<true, false><<<grid, PM_THREADS, 0, st>>>(p);
        else conv3x3_pair_tmem_kernel<false, false><<<grid, PM_THREADS, 0, st>>>(p);
    }
    UOCR_LAUNCHED("conv3x3_pair_tmem");
    return UOCR_OK;
}

}  // namespace uocr

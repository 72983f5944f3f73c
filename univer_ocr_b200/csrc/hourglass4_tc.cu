// Fused four-channel "hourglass" forward (inference, TF32 mode): the whole Line network in one kernel on the tensor
// cores.
//
//   x (1 ch) -> conv5x5 s2 + act -> conv5x5 s2 + act -> up x2, conv5x5 + act -> up x2, conv5x5 + act -> conv5x5 + act_end -> y (2 ch)
//               (down_1, 1 -> 4)    (down_2, 4 -> 4)    (up_2, 4 -> 4)          (up_1, 4 -> 4)          (end, 4 -> 2)
//   replaces, for make_line (my_model/model.py:194-248, channels = 4): five Convolutional2D._forward calls
//   (convolutional.py:62-99), two Upsample2D._forward (upsample.py:21-39) and five LeakyRelu / Sigmoid._forward
//   (layers.py:390-415) -- five launches of 15-35 us at batch 64 before.
//
// One CTA produces a 16 x 128 block of the output; the blocks of the intermediate maps it depends on (same geometry as
// hourglass.cu) live in shared memory as channels-last pixels of 16 bytes.  Every level is a handful of
// tcgen05.mma (128 x 16 x 8, TF32, FP32 accumulators in tensor memory) whose A operand is the previous level's block
// read IN PLACE: K-major, no swizzle, 8 rows of a core matrix 16 bytes apart -- row m of the operand is "position" m of
// the block in linear pixel order, its K = 8 floats are that pixel and the next one, and the next K chunk is simply
// the descriptor advanced by two pixels.  The rows of the operand overlap in memory; nothing is gathered or copied.
// A tile of 128 positions runs across block rows (the positions in the halo columns compute garbage that is never
// stored), a vertical tap is the descriptor advanced by one block row.
//   down_1  x block as two row-parity planes (two TMA boxes through tensor maps with a doubled row stride), position =
//           4 input columns = 2 output pixels: N = 2 pixels x 4 channels, one MMA per kernel row           (5 per tile)
//   down_2  the down_1 epilogue scatters its pixels into 4 (row, column)-parity planes, which turns the stride-2
//           convolution into four stride-1 convolutions with 3x3 / 3x2 / 2x3 / 2x2 taps                   (15 per tile)
//   up_2, up_1   a 5 x 5 convolution over a x2 nearest-upsampled map sees 3 x 3 distinct source pixels with
//           parity-specific pre-summed weights (hourglass.cu): M = SOURCE position, N = 2 x 2 parities x 4
//           channels = 16, so one accumulator row holds the 2 x 2 output pixels of its source pixel      (6 per tile)
//   end     M = the 128 output columns of one block row, N = 8 output rows x 2 channels: the MMA of input row j
//           carries the weights of kernel row j - i in the columns of output row i, so 12 input rows x 3 K chunks
//           produce 8 output rows (4.5 MMAs per output row instead of 15).  The 36 B tiles are windows of one
//           weight strip (tile j starts 2 rows before tile j + 1)                                         (36 per 8 rows)
// Epilogues: tcgen05.ld (lane = position), + bias, LeakyReLU, zero outside the image (= the next level's padding),
// round to TF32, 16-byte stores into the next block.  ~160 MMAs and ~20 tensor-memory loads per warp replace 0.9 MFMA.
#include "conv_common.cuh"
#include "tc_ptx.cuh"

namespace uocr {
namespace {

constexpr int H4_TH = 16, H4_TW = 128, H4_THREADS = 256;
constexpr int H4_XP = 156;                        // x block pitch (floats) = 39 positions of 4 columns
constexpr int H4_POS = 39;                        // positions per row of down_1 = pixel pitch of the D1 planes and of D2
constexpr int H4_XE_ROWS = 21, H4_XO_ROWS = 20;   // even / odd rows of the 41-row x block
constexpr int H4_D1H = 19, H4_D1W = 75;
constexpr int H4_P0_ROWS = 10, H4_P1_ROWS = 9;    // rows of the even- / odd-row planes of D1
constexpr int H4_D2H = 8, H4_D2W = 36;
constexpr int H4_U2H = 12, H4_U2W = 68, H4_PU2 = 68;
constexpr int H4_U1H = 20, H4_U1W = 132, H4_PU1 = 132;
constexpr int H4_T1 = 6, H4_T2 = 3, H4_T3 = 2, H4_T4 = 6, H4_T5 = 1;      // M tiles per level
static_assert(H4_D1H * H4_POS <= H4_T1 * 128 && H4_D2H * H4_POS <= H4_T2 * 128, "tiles cover the positions");
static_assert((H4_U2H / 2) * H4_POS <= H4_T3 * 128 && (H4_U1H / 2) * H4_PU2 <= H4_T4 * 128, "tiles cover the positions");

// B operand image (floats): [level 1: 5 tiles][level 2: 13][level 3: 5][level 4: 5][level 5: strip 3 x 2 x 70 x 4]
constexpr int H4_B1 = 0, H4_B2 = 5 * 128, H4_B3 = H4_B2 + 13 * 128, H4_B4 = H4_B3 + 5 * 128, H4_B5 = H4_B4 + 5 * 128;
constexpr int H4_SROWS = 70;                      // 32 tile rows + 2 * 19 window positions
constexpr int H4_BFLOATS = H4_B5 + 3 * 2 * H4_SROWS * 4;                   // 5264

// shared memory (bytes)
constexpr int OFF_XE = 0;
constexpr int OFF_XO = 13184;                     // 21 * 624 = 13104, rounded up to 128
constexpr int OFF_P00 = 25728;                    // 13184 + 20 * 624 = 25664, rounded up to 128
constexpr int P0_BYTES = H4_P0_ROWS * H4_POS * 16, P1_BYTES = H4_P1_ROWS * H4_POS * 16;
constexpr int OFF_P10 = OFF_P00 + 2 * P0_BYTES;
constexpr int OFF_R0_END = OFF_P10 + 2 * P1_BYTES;                         // 49440
// D2, U2 and U1 alias the x block and the D1 planes: a level's epilogue starts only after all of the level's MMAs have
// completed, so the block a level WRITES may overwrite the block it READ (and everything older).  70 KB: 3 CTAs / SM.
constexpr int OFF_U1 = 0, OFF_D2 = 0, OFF_U2 = 0;
constexpr int U1_BYTES = H4_U1H * H4_PU1 * 16;
constexpr int D2_BYTES = H4_D2H * H4_POS * 16;
constexpr int U2_BYTES = H4_U2H * H4_PU2 * 16;
static_assert(OFF_U1 + U1_BYTES + 64 <= OFF_R0_END, "U1 fits over the x block and the D1 planes");
constexpr int OFF_B = OFF_R0_END;
constexpr int OFF_BIAS = OFF_B + H4_BFLOATS * 4;
constexpr int OFF_BAR = OFF_BIAS + 96;
constexpr int OFF_TMEM = OFF_BAR + 64;
constexpr int OFF_EXT = OFF_BIAS + 72;            // ragged batches: the image's extent (int2) after the 18 biases
constexpr int H4_SMEM = OFF_TMEM + 16;
static_assert(OFF_XO % 128 == 0 && OFF_P00 % 16 == 0 && OFF_D2 % 16 == 0 && OFF_U2 % 16 == 0 && OFF_B % 16 == 0 &&
              OFF_BAR % 8 == 0, "alignment");

struct Hourglass4Params {
    float* y;
    const float* bimg;                            // H4_BFLOATS B-operand floats (hourglass4_prep_kernel)
    const float* b[5];
    int H, W;
    float alpha;
    int act_end; float alpha_end;
    const int32_t* ext;                           // ragged batches: (N, 2) extents (h_i, w_i) on the device
};

// ---- B operand image.  Every MMA tile is K-major [chunk c: 2][n: 16][e: 4] (k = 4 c + e); weights are (5,5,Cin,Cout).
__device__ __forceinline__ bool fold_hit(int parity, int slot, int k) {
    // kernel index k lands on source offset `slot` for this output parity: parity 0: {0,1} {2,3} {4}; 1: {0} {1,2} {3,4}
    return parity == 0 ? (k >> 1) == slot : ((k + 1) >> 1) == slot;
}

__global__ void __launch_bounds__(256) hourglass4_prep_kernel(const float* __restrict__ w1, const float* __restrict__ w2,
                                                              const float* __restrict__ w3, const float* __restrict__ w4,
                                                              const float* __restrict__ w5, float* __restrict__ bimg) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= H4_BFLOATS) return;
    float v = 0.f;
    if (i < H4_B5) {
        const int tile = i >> 7, c = (i >> 6) & 1, n = (i >> 2) & 15, e = i & 3;
        if (i < H4_B2) {                          // down_1: tile = ky, k = x column inside the position, n = (pixel jj, co)
            const int ky = tile, jj = n >> 2, co = n & 3, kx = 4 * c + e - 2 * jj;
            if (n < 8 && kx >= 0 && kx < 5) v = w1[(ky * 5 + kx) * 4 + co];
        } else if (i < H4_B3) {
            // down_2: a K chunk is one pixel of one parity plane = (row parity pr, row tap a, column parity pc, column
            // tap b), kernel tap (2 a + pr, 2 b + pc).  Tiles 2 g, 2 g + 1 of group g = (pr, a): chunks (pc 0, b 0 | pc 0,
            // b 1) and (pc 0, b 2 | pc 1, b 0); the five left-over chunks (pc 1, b 1) share tiles 10-12 in pairs.
            const int t = tile - 5;
            int g, pc, b;
            if (t < 10) { g = t >> 1; pc = (t & 1) & c; b = (t & 1) ? (c ? 0 : 2) : c; }
            else { g = 2 * (t - 10) + c; pc = 1; b = 1; }
            if (g < 5) {
                const int pr = g < 3 ? 0 : 1, a = pr ? g - 3 : g, ky = 2 * a + pr, kx = 2 * b + pc;
                if (n < 4) v = w2[((ky * 5 + kx) * 4 + e) * 4 + n];
            }
        } else {
            // up_2 / up_1: a K chunk = source pixel (row a, column b); tiles 0-2: (a, 0 | a, 1), tile 3: (0, 2 | 1, 2),
            // tile 4: (2, 2 | nothing); n = (py, px, co), weights pre-summed per output parity
            const bool l4 = i >= H4_B4;
            const float* w = l4 ? w4 : w3;
            const int t = tile - (l4 ? 23 : 18);
            const int a = t < 3 ? t : t == 3 ? c : 2, b = t < 3 ? c : 2;
            const int py = n >> 3, px = (n >> 2) & 1, co = n & 3;
            if (!(t == 4 && c == 1))
                for (int ky = 0; ky < 5; ++ky)
                    for (int kx = 0; kx < 5; ++kx)
                        if (fold_hit(py, a, ky) && fold_hit(px, b, kx)) v += w[((ky * 5 + kx) * 4 + e) * 4 + co];
        }
    } else {
        // end: strip [k'][c][row v][ci], row v = kernel row 19 - v / 2, channel v & 1; the tile of input row j is the
        // 32-row window from row 38 - 2 j.  Block [2][1] repeats block [2][0] (kx = 4): the MMA that pairs the kx = 4
        // chunks of rows j and j + 1 reads its second chunk's window 2 rows lower, i.e. at a positive offset from the first
        const int s = i - H4_B5, e = s & 3, vrow = (s >> 2) % H4_SROWS, c = (s / (4 * H4_SROWS)) & 1, kq = s / (8 * H4_SROWS);
        const int ky = 19 - (vrow >> 1), kx = kq == 2 ? 4 : 2 * kq + c;
        if (ky >= 0 && ky < 5) v = w5[((ky * 5 + kx) * 4 + e) * 2 + (vrow & 1)];
    }
    bimg[i] = round_tf32(v);
}

__device__ __forceinline__ bool h4_elect() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// the block just written through the generic proxy becomes an MMA operand; the accumulators just read become free
__device__ __forceinline__ void h4_level_sync() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
}

// + bias, LeakyReLU, round to TF32 (round to nearest, ties away: add half an ulp of the 10-bit mantissa and cut; the mask
// doubles as the "inside the image" select), as one 16-byte shared-memory store.  Branch-free: the first version (a
// conditional around every value, biases read from shared memory) spent 8 k cycles in up_1's epilogue alone.
__device__ __forceinline__ void h4_store4(uint32_t addr, const uint32_t* v, const float4 b, float alpha, bool in) {
    const uint32_t msk = in ? 0xffffe000u : 0u;
    const float t0 = __uint_as_float(v[0]) + b.x, t1 = __uint_as_float(v[1]) + b.y;
    const float t2 = __uint_as_float(v[2]) + b.z, t3 = __uint_as_float(v[3]) + b.w;
    const uint32_t o0 = (__float_as_uint(fmaxf(t0, t0 * alpha)) + 0x1000u) & msk;
    const uint32_t o1 = (__float_as_uint(fmaxf(t1, t1 * alpha)) + 0x1000u) & msk;
    const uint32_t o2 = (__float_as_uint(fmaxf(t2, t2 * alpha)) + 0x1000u) & msk;
    const uint32_t o3 = (__float_as_uint(fmaxf(t3, t3 * alpha)) + 0x1000u) & msk;
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(o0), "r"(o1), "r"(o2), "r"(o3) : "memory");
}
__device__ __forceinline__ void h4_zero16(uint32_t addr) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(addr), "r"(0u) : "memory");
}
// a ragged CTA outside its image: zeros over its 16 x 128 output block (out of line: inlined, it costs the kernel spills)
__device__ __noinline__ void h4_zero_block(const Hourglass4Params& p, int img, int oy0, int ox0) {
    const int gx = ox0 + (threadIdx.x & (H4_TW - 1));
    if (gx < p.W)
        for (int r = threadIdx.x / H4_TW; r < H4_TH && oy0 + r < p.H; r += H4_THREADS / H4_TW)
            *reinterpret_cast<float2*>(p.y + (((int64_t)img * p.H + oy0 + r) * p.W + gx) * 2) = make_float2(0.f, 0.f);
}

// the image's extent (h, w) for the "inside the image" tests: the canvas size, or in a ragged batch the image's own
// extent, parked in shared memory and re-read where it is used (kept in registers it pushes the kernel into spills)
template <bool RAGGED>
__device__ __forceinline__ int2 h4_extent(uint32_t sm, const Hourglass4Params& p) {
    if constexpr (!RAGGED) return make_int2(p.H, p.W);
    int2 e;
    asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(e.x), "=r"(e.y) : "r"(sm + OFF_EXT));
    return e;
}
__device__ __forceinline__ float4 h4_lds4(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
    return r;
}

// RAGGED: x and y are canvases of a ragged batch (uocr.h); every "inside the image" test uses image img's own extent
// extent instead of the canvas size (h4_extent), while addresses keep the canvas pitch.
template <bool RAGGED>
__global__ void __launch_bounds__(H4_THREADS, 3) hourglass4_fwd_kernel(const Hourglass4Params p,
                                                                       const __grid_constant__ CUtensorMap map_even,
                                                                       const __grid_constant__ CUtensorMap map_odd) {
    extern __shared__ __align__(128) uint8_t h4_smem[];
    const uint32_t sm = smem_u32(h4_smem);
    float* sBias = reinterpret_cast<float*>(h4_smem + OFF_BIAS);         // b1[4] b2[4] b3[4] b4[4] b5[2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(h4_smem + OFF_TMEM);
    const uint32_t bar = sm + OFF_BAR;                                   // bar + 8 l: level l (0 = the x block's TMA)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, quarter = warp & 3;
    const int ox0 = blockIdx.x * H4_TW, oy0 = blockIdx.y * H4_TH, img = blockIdx.z;
    const int hy0 = oy0 / 2, hx0 = ox0 / 2, qy0 = oy0 / 4, qx0 = ox0 / 4;
    if constexpr (RAGGED) {
        int eh = min(max(__ldg(p.ext + 2 * img), 0), p.H), ew = min(max(__ldg(p.ext + 2 * img + 1), 0), p.W);
        if ((eh | ew) & 3) eh = ew = 0;                                  // not a multiple of 4: no image, zeros only
        if (oy0 >= eh || ox0 >= ew) {
            // the block lies wholly outside the image: its zeros, then exit before any barrier, TMA copy or tensor
            // memory exists (a CTA that exits with a TMA copy in flight faults, DESIGN.md §3)
            h4_zero_block(p, img, oy0, ox0);
            return;
        }
        if (tid == 0) *reinterpret_cast<int2*>(h4_smem + OFF_EXT) = make_int2(eh, ew);
    }

    if (tid == 0) {
#pragma unroll
        for (int l = 0; l < 6; ++l) mbar_init(bar + 8 * l, l == 0 ? 1u : (uint32_t)(l == 1 ? H4_T1 : l == 2 ? H4_T2 : l == 3 ? H4_T3 : l == 4 ? H4_T4 : H4_T5));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_arrive_expect_tx(bar, (uint32_t)((H4_XE_ROWS + H4_XO_ROWS) * H4_XP * 4 + H4_BFLOATS * 4));
        // block row 2 i (+ 1) = row (oy0 - 14) / 2 + i of the even- (odd-) row view of the image; zeros outside it.
        // The box starts at column ox0 - 16: a TMA box has to start on a 16-byte boundary of the tensor.
        tma_load_3d(sm + OFF_XE, &map_even, bar, ox0 - 16, (oy0 - 14) / 2, img);
        tma_load_3d(sm + OFF_XO, &map_odd, bar, ox0 - 16, (oy0 - 14) / 2, img);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(sm + OFF_B), "l"(p.bimg), "r"((uint32_t)(H4_BFLOATS * 4)), "r"(bar) : "memory");
    }
    __syncwarp();
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sm + OFF_TMEM), "r"(128u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    {   // biases; the gaps that valid rows' zero-weight K lanes reach must hold finite numbers
        if (tid < 4) {                                                   // static level index: keeps p in constant memory
#pragma unroll
            for (int l = 0; l < 4; ++l) sBias[4 * l + tid] = __ldg(p.b[l] + tid);
            if (tid < 2) sBias[16 + tid] = __ldg(p.b[4] + tid);
        }
        if (tid >= 32 && tid < 37) h4_zero16(sm + OFF_XO - 80 + 16 * (tid - 32));
        if (tid >= 64 && tid < 68) h4_zero16(sm + OFF_P00 - 64 + 16 * (tid - 64));
    }
    h4_level_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((16u >> 3) << 17) | ((128u >> 4) << 24);
    // descriptors count in 16-byte units = pixels (positions for the x planes)
    const uint64_t dA0 = make_kmajor_nosw_desc(sm, 16, 128);             // + byte offset / 16
    const uint64_t dB0 = make_kmajor_nosw_desc(sm + OFF_B, 256, 128);    // + 32 per tile
    const uint32_t my_tmem = tmem + ((uint32_t)(quarter * 32) << 16);

    // ================= down_1: x planes -> D1 parity planes
    if (warp < H4_T1) {
        if (h4_elect()) {
            mbar_wait(bar, 0);
            const uint64_t ae = dA0 + (uint64_t)(OFF_XE / 16 + 128 * warp), ao = dA0 + (uint64_t)(OFF_XO / 16 + 128 * warp);
#pragma unroll
            for (int ky = 0; ky < 5; ++ky)
                tc_mma_tf32(tmem + 16u * warp, ((ky & 1) ? ao : ae) + (uint64_t)((ky >> 1) * H4_POS),
                            dB0 + (uint64_t)(H4_B1 / 4 + 32 * ky), idesc, ky > 0);
            tc_commit(bar + 8);
        }
        __syncwarp();
    }
    mbar_wait(bar + 8, 0);
    tc_fence_after();
    float4 bias = h4_lds4(sm + OFF_BIAS);
    for (int t = warp >> 2; t < H4_T1; t += 2) {
        uint32_t v[8];
        tc_ld8_nowait(my_tmem + 16u * t, v);
        tc_wait_ld();
        const int m = t * 128 + quarter * 32 + lane, r = m / H4_POS, q = m - r * H4_POS;
        if (r < H4_D1H) {
            const int2 e = h4_extent<RAGGED>(sm, p);
            const bool rowin = (unsigned)(hy0 - 6 + r) < (unsigned)(e.x / 2);
            const uint32_t plane = sm + ((r & 1) ? OFF_P10 : OFF_P00) + ((r >> 1) * H4_POS + q) * 16;
            const uint32_t pbytes = (r & 1) ? P1_BYTES : P0_BYTES;
            // position q = block columns 4 q .. 4 q + 3 = D1 columns 2 q - 1 (odd: plane 1, column q - 1) and 2 q (even:
            // plane 0, column q)
            const int col = 2 * q - 1;
            const bool in0 = rowin && col >= 0 && (unsigned)(hx0 - 6 + col) < (unsigned)(e.y / 2);
            const bool in1 = rowin && col + 1 < H4_D1W && (unsigned)(hx0 - 6 + col + 1) < (unsigned)(e.y / 2);
            if (q > 0) h4_store4(plane + pbytes - 16, v, bias, p.alpha, in0);
            h4_store4(plane, v + 4, bias, p.alpha, in1);
            if (q == H4_POS - 1) h4_zero16(plane + pbytes);
        }
    }
    h4_level_sync();

    // ================= down_2: D1 planes -> D2
    if (warp < H4_T2) {
        if (h4_elect()) {
            const uint32_t d = tmem + 16u * warp;
            const uint32_t t0 = sm + 128 * 16 * warp;                    // this tile's first position
            // group (pr, a): (pc 0: b 0 | b 1), (pc 0: b 2 | pc 1: b 0) -- the second chunk sits in the other plane
#pragma unroll
            for (int g = 0; g < 5; ++g) {
                const int pr = g < 3 ? 0 : 1, a = pr ? g - 3 : g;
                const uint32_t base = t0 + (pr ? OFF_P10 : OFF_P00) + a * H4_POS * 16, pbytes = pr ? P1_BYTES : P0_BYTES;
                tc_mma_tf32(d, make_kmajor_nosw_desc(base, 16, 128), dB0 + (uint64_t)(H4_B2 / 4 + 32 * (2 * g)), idesc, g > 0);
                tc_mma_tf32(d, make_kmajor_nosw_desc(base + 32, pbytes - 32, 128), dB0 + (uint64_t)(H4_B2 / 4 + 32 * (2 * g + 1)), idesc, 1);
            }
            // the left-over chunks (pc 1, b 1) of the five groups, two per MMA
            constexpr int L0 = OFF_P00 + P0_BYTES + 16, L1 = OFF_P10 + P1_BYTES + 16;       // plane pc 1, pixel c + 1
            tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + L0, H4_POS * 16, 128), dB0 + (uint64_t)(H4_B2 / 4 + 32 * 10), idesc, 1);
            tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + L0 + 2 * H4_POS * 16, L1 - (L0 + 2 * H4_POS * 16), 128),
                        dB0 + (uint64_t)(H4_B2 / 4 + 32 * 11), idesc, 1);
            tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + L1 + H4_POS * 16, 16, 128), dB0 + (uint64_t)(H4_B2 / 4 + 32 * 12), idesc, 1);
            tc_commit(bar + 16);
        }
        __syncwarp();
    }
    mbar_wait(bar + 16, 0);
    tc_fence_after();
    bias = h4_lds4(sm + OFF_BIAS + 16);
    for (int t = warp >> 2; t < H4_T2; t += 2) {
        uint32_t v[4];
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(my_tmem + 16u * t) : "memory");
        tc_wait_ld();
        const int m = t * 128 + quarter * 32 + lane, r = m / H4_POS, c = m - r * H4_POS;
        if (r < H4_D2H) {
            const int2 e = h4_extent<RAGGED>(sm, p);
            const bool in = c < H4_D2W && (unsigned)(qy0 - 2 + r) < (unsigned)(e.x / 4) && (unsigned)(qx0 - 2 + c) < (unsigned)(e.y / 4);
            h4_store4(sm + OFF_D2 + m * 16, v, bias, p.alpha, in);
        }
    }
    h4_level_sync();

    // ================= up_2: D2 -> U2 (source position (j, n) -> pixels (2 j + py, 2 n + px))
    if (warp < H4_T3) {
        if (h4_elect()) {
            const uint32_t d = tmem + 16u * warp, t0 = sm + OFF_D2 + 128 * 16 * warp;
            // source pixels (a, 0 | a, 1) for the three rows, then the third column: (0, 2 | 1, 2) one row apart, (2, 2 | -)
#pragma unroll
            for (int a = 0; a < 3; ++a)
                tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + a * H4_POS * 16, 16, 128), dB0 + (uint64_t)(H4_B3 / 4 + 32 * a), idesc, a > 0);
            tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + 32, H4_POS * 16, 128), dB0 + (uint64_t)(H4_B3 / 4 + 32 * 3), idesc, 1);
            tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + 2 * H4_POS * 16 + 32, 16, 128), dB0 + (uint64_t)(H4_B3 / 4 + 32 * 4), idesc, 1);
            tc_commit(bar + 24);
        }
        __syncwarp();
    }
    mbar_wait(bar + 24, 0);
    tc_fence_after();
    bias = h4_lds4(sm + OFF_BIAS + 32);
    for (int t = warp >> 2; t < H4_T3; t += 2) {
        uint32_t v[16];
        tc_ld16_nowait(my_tmem + 16u * t, v);
        tc_wait_ld();
        const int m = t * 128 + quarter * 32 + lane, j = m / H4_POS, n = m - j * H4_POS;
        if (j < H4_U2H / 2 && n < H4_U2W / 2) {
            const int2 e = h4_extent<RAGGED>(sm, p);
#pragma unroll
            for (int py = 0; py < 2; ++py) {
                const bool rowin = (unsigned)(hy0 - 2 + 2 * j + py) < (unsigned)(e.x / 2);
#pragma unroll
                for (int px = 0; px < 2; ++px) {
                    const bool in = rowin && (unsigned)(hx0 - 2 + 2 * n + px) < (unsigned)(e.y / 2);
                    h4_store4(sm + OFF_U2 + ((2 * j + py) * H4_PU2 + 2 * n + px) * 16, v + 4 * (2 * py + px), bias, p.alpha, in);
                }
            }
        }
    }
    h4_level_sync();

    // ================= up_1: U2 -> U1
    if (warp < H4_T4) {
        if (h4_elect()) {
            const uint32_t d = tmem + 16u * warp, t0 = sm + OFF_U2 + 128 * 16 * warp;
            // source pixels (a, 0 | a, 1) for the three rows, then the third column: (0, 2 | 1, 2) one row apart, (2, 2 | -)
#pragma unroll
            for (int a = 0; a < 3; ++a)
                tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + a * H4_PU2 * 16, 16, 128), dB0 + (uint64_t)(H4_B4 / 4 + 32 * a), idesc, a > 0);
            tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + 32, H4_PU2 * 16, 128), dB0 + (uint64_t)(H4_B4 / 4 + 32 * 3), idesc, 1);
            tc_mma_tf32(d, make_kmajor_nosw_desc(t0 + 2 * H4_PU2 * 16 + 32, 16, 128), dB0 + (uint64_t)(H4_B4 / 4 + 32 * 4), idesc, 1);
            tc_commit(bar + 32);
        }
        __syncwarp();
    }
    mbar_wait(bar + 32, 0);
    tc_fence_after();
    bias = h4_lds4(sm + OFF_BIAS + 48);
    for (int t = warp >> 2; t < H4_T4; t += 2) {
        uint32_t v[16];
        tc_ld16_nowait(my_tmem + 16u * t, v);
        tc_wait_ld();
        const int m = t * 128 + quarter * 32 + lane, j = m / H4_PU2, n = m - j * H4_PU2;
        if (j < H4_U1H / 2 && n < H4_U1W / 2) {
            const int2 e = h4_extent<RAGGED>(sm, p);
#pragma unroll
            for (int py = 0; py < 2; ++py) {
                const bool rowin = (unsigned)(oy0 - 2 + 2 * j + py) < (unsigned)e.x;
#pragma unroll
                for (int px = 0; px < 2; ++px) {
                    const bool in = rowin && (unsigned)(ox0 - 2 + 2 * n + px) < (unsigned)e.y;
                    h4_store4(sm + OFF_U1 + ((2 * j + py) * H4_PU1 + 2 * n + px) * 16, v + 4 * (2 * py + px), bias, p.alpha, in);
                }
            }
        }
    }
    h4_level_sync();

    // ================= end: U1 -> y; tile g = output rows 8 g .. 8 g + 7, lane = output column
    if (warp < H4_T5) {
        if (h4_elect()) {
            // one accumulator of N = 16 output rows x 2 channels; input row j: pixels (c, c+1), (c+2, c+3) against the
            // strip windows of row j, and pixel c + 4 of rows j and j + 1 together (chunks one block row apart)
            const uint32_t idesc32 = (1u << 4) | (2u << 7) | (2u << 10) | ((32u >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t sS = sm + OFF_B + H4_B5 * 4;
#pragma unroll
            for (int j = 0; j < 20; ++j) {
                const uint32_t row = sm + OFF_U1 + j * H4_PU1 * 16;
#pragma unroll
                for (int kq = 0; kq < 2; ++kq)
                    tc_mma_tf32(tmem, make_kmajor_nosw_desc(row + 32 * kq, 16, 128),
                                make_kmajor_nosw_desc(sS + (2 * kq * H4_SROWS + 38 - 2 * j) * 16, H4_SROWS * 16, 128), idesc32, (j | kq) != 0);
                if (!(j & 1))
                    tc_mma_tf32(tmem, make_kmajor_nosw_desc(row + 64, H4_PU1 * 16, 128),
                                make_kmajor_nosw_desc(sS + (4 * H4_SROWS + 38 - 2 * j) * 16, H4_SROWS * 16 - 32, 128), idesc32, 1);
            }
            tc_commit(bar + 40);
        }
        __syncwarp();
    }
    mbar_wait(bar + 40, 0);
    tc_fence_after();
    {
        const int g = warp >> 2, c = quarter * 32 + lane;
        uint32_t v[16];
        tc_ld16_nowait(my_tmem + 16u * g, v);
        tc_wait_ld();
        const int gx = ox0 + c;
        const float b0 = sBias[16], b1 = sBias[17];
        float o[16];
        if (p.act_end == UOCR_ACT_SIGMOID) {                              // one branch, not one per value
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = apply_act_fast(__uint_as_float(v[i]) + ((i & 1) ? b1 : b0), UOCR_ACT_SIGMOID, 0.f);
        } else {
            const float a = p.act_end == UOCR_ACT_LEAKY ? p.alpha_end : 1.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float t = __uint_as_float(v[i]) + ((i & 1) ? b1 : b0);
                o[i] = t > 0.f ? t : t * a;
            }
        }
        if constexpr (RAGGED) {                                          // the canvas outside the extent gets zeros
            const int2 e = h4_extent<RAGGED>(sm, p);
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (gx >= e.y || oy0 + 8 * g + i >= e.x) o[2 * i] = o[2 * i + 1] = 0.f;
        }
        if (gx < p.W) {
            float* dst = p.y + (((int64_t)img * p.H + oy0 + 8 * g) * p.W + gx) * 2;
#pragma unroll
            for (int i = 0; i < 8; ++i)
                if (oy0 + 8 * g + i < p.H) *reinterpret_cast<float2*>(dst + (int64_t)i * p.W * 2) = make_float2(o[2 * i], o[2 * i + 1]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(128u) : "memory");
}

}  // namespace

static int hourglass4_pack(const float* const* w, float* packed, cudaStream_t st) {
    hourglass4_prep_kernel<<<(H4_BFLOATS + 255) / 256, 256, 0, st>>>(w[0], w[1], w[2], w[3], w[4], packed);
    UOCR_LAUNCHED("hourglass4_prep");
    return UOCR_OK;
}

static int hourglass4_run(const float* x, const float* packed, const float* const* b, float* y, int64_t n, int64_t h,
                          int64_t wd, float alpha, int act_end, float alpha_end, cudaStream_t st,
                          const int32_t* extents = nullptr) {
    if (h % 4 || wd % 4 || n > 65535 || alpha < 0.f || alpha > 1.f) return UOCR_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(packed)) & 15)
        return UOCR_ERR_UNSUPPORTED;
    CUtensorMap map_even{}, map_odd{};
    const uint64_t dims[3] = {(uint64_t)wd, (uint64_t)(h / 2), (uint64_t)n};         // the even / odd rows of the image
    const uint64_t strides[2] = {(uint64_t)wd * 8, (uint64_t)wd * h * 4};
    const uint32_t box_e[3] = {(uint32_t)H4_XP, (uint32_t)H4_XE_ROWS, 1}, box_o[3] = {(uint32_t)H4_XP, (uint32_t)H4_XO_ROWS, 1};
    int rc = make_tmap_plain_tf32(&map_even, x, 3, dims, strides, box_e);
    if (rc == UOCR_OK) rc = make_tmap_plain_tf32(&map_odd, x + wd, 3, dims, strides, box_o);
    if (rc != UOCR_OK) return rc;
    static bool configured = false;
    if (!configured) {
        for (const void* kernel : {(const void*)hourglass4_fwd_kernel<false>, (const void*)hourglass4_fwd_kernel<true>}) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, H4_SMEM);
            if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
        }
        configured = true;
    }
    Hourglass4Params p{};
    p.y = y; p.bimg = packed;
    for (int l = 0; l < 5; ++l) p.b[l] = b[l];
    p.H = (int)h; p.W = (int)wd; p.alpha = alpha; p.act_end = act_end; p.alpha_end = alpha_end; p.ext = extents;
    dim3 grid((unsigned)ceil_div(wd, H4_TW), (unsigned)ceil_div(h, H4_TH), (unsigned)n);
    if (grid.y > 65535) return UOCR_ERR_UNSUPPORTED;
    if (extents) {
        hourglass4_fwd_kernel<true><<<grid, H4_THREADS, H4_SMEM, st>>>(p, map_even, map_odd);
        UOCR_LAUNCHED("hourglass4_fwd_ragged");
    } else {
        hourglass4_fwd_kernel<false><<<grid, H4_THREADS, H4_SMEM, st>>>(p, map_even, map_odd);
        UOCR_LAUNCHED("hourglass4_fwd");
    }
    return UOCR_OK;
}

}  // namespace uocr

using namespace uocr;

static int hourglass4_check(const void* x, const void* y, const float* const* biases, int64_t n, int64_t h, int64_t w,
                            int act_end) {
    UOCR_REQUIRE(x && y && biases, "NULL pointer");
    for (int l = 0; l < 5; ++l) UOCR_REQUIRE(biases[l], "NULL bias pointer (level %d)", l);
    UOCR_REQUIRE(n > 0 && h > 0 && w > 0 && h < (1 << 30) && w < (1 << 30), "bad dimension");
    UOCR_REQUIRE(act_end >= UOCR_ACT_NONE && act_end <= UOCR_ACT_SIGMOID, "unknown activation %d", act_end);
    return UOCR_OK;
}

extern "C" int uocr_hourglass4_packed_floats(int64_t* floats) {
    UOCR_REQUIRE(floats, "NULL pointer");
    *floats = H4_BFLOATS;
    return UOCR_OK;
}

extern "C" int uocr_hourglass4_pack(const float* const* weights, float* packed, void* stream) {
    UOCR_REQUIRE(weights && packed, "NULL pointer");
    for (int l = 0; l < 5; ++l) UOCR_REQUIRE(weights[l], "NULL weight pointer (level %d)", l);
    return hourglass4_pack(weights, packed, as_stream(stream));
}

extern "C" int uocr_hourglass4_fwd_packed(const float* x, const float* packed, const float* const* biases, float* y,
                                          int64_t n, int64_t h, int64_t w, float alpha, int act_end, float alpha_end,
                                          void* stream) {
    UOCR_REQUIRE(packed, "NULL pointer");
    int rc = hourglass4_check(x, y, biases, n, h, w, act_end);
    if (rc != UOCR_OK) return rc;
    rc = hourglass4_run(x, packed, biases, y, n, h, w, alpha, act_end, alpha_end, as_stream(stream));
    if (rc == UOCR_ERR_UNSUPPORTED) set_error("hourglass4_fwd: unsupported geometry (H, W must be multiples of 4)");
    return rc;
}

extern "C" int uocr_hourglass4_fwd_packed_ragged(const float* x, const float* packed, const float* const* biases, float* y,
                                                 const int32_t* extents, int64_t n, int64_t h, int64_t w, float alpha,
                                                 int act_end, float alpha_end, void* stream) {
    UOCR_REQUIRE(packed && extents, "NULL pointer");
    int rc = hourglass4_check(x, y, biases, n, h, w, act_end);
    if (rc != UOCR_OK) return rc;
    rc = hourglass4_run(x, packed, biases, y, n, h, w, alpha, act_end, alpha_end, as_stream(stream), extents);
    if (rc == UOCR_ERR_UNSUPPORTED)
        set_error("hourglass4_fwd_packed_ragged: unsupported geometry (H, W and every extent must be multiples of 4)");
    return rc;
}

extern "C" int uocr_hourglass4_fwd(const float* x, const float* const* weights, const float* const* biases, float* y,
                                   int64_t n, int64_t h, int64_t w, float alpha, int act_end, float alpha_end,
                                   void* stream) {
    UOCR_REQUIRE(weights, "NULL pointer");
    for (int l = 0; l < 5; ++l) UOCR_REQUIRE(weights[l], "NULL weight pointer (level %d)", l);
    int rc = hourglass4_check(x, y, biases, n, h, w, act_end);
    if (rc != UOCR_OK) return rc;
    Scratch packed(as_stream(stream));
    rc = packed.alloc(H4_BFLOATS * sizeof(float));
    if (rc != UOCR_OK) return rc;
    hourglass4_pack(weights, static_cast<float*>(packed.ptr), as_stream(stream));
    rc = hourglass4_run(x, static_cast<const float*>(packed.ptr), biases, y, n, h, w, alpha, act_end, alpha_end, as_stream(stream));
    if (rc == UOCR_ERR_UNSUPPORTED) set_error("hourglass4_fwd: unsupported geometry (H, W must be multiples of 4)");
    return rc;
}

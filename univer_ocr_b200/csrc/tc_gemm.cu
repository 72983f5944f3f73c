// tcgen05 (5th-generation tensor core) TF32 kernels: the dense contractions of the path
// (SURVEY.md 8d: Char conv_2 / conv_3 and the three FullyConnected GEMMs).
//
//   D[M, N] (+)= A[M, K] . B[N, K]^T        TF32 inputs, FP32 accumulation in TMEM
//
// One CTA = one 128 x NT output tile (cta_group::1, UMMA M = 128, N = NT <= 256, K = 8 per
// instruction).  Warp roles (192 threads):
//   warp 0    TMA producer: one elected lane streams 128B-swizzled K-major tiles
//             (A: 128 rows x 32 floats, B: NT rows x 32 floats per stage) into a ring of shared
//             memory stages, signalling `full[s]` through mbarrier complete_tx
//   warp 1    allocates TMEM, then one elected lane issues tcgen05.mma (4 per stage) and releases
//             the stage with tcgen05.commit -> `empty[s]`; the last commit raises `tmem_full`
//   warps 2-5 epilogue: tcgen05.ld the accumulator (lane = row, column = n), add the bias row,
//             apply the activation, store to global memory
// A tiles come either from a plain row-major matrix (2-D tensor map) or -- implicit GEMM for
// Convolutional2D with Cin % 32 == 0 and stride_w == 1 -- straight from the NHWC activation
// tensor through a 4-D tensor map: the tile for kernel tap (ky, kx) is the box
// [32 channels x 128 consecutive pixels] at (x0 + kx - pw, oy * sh + ky - ph); TMA's
// out-of-bounds zero fill IS the zero padding, so no im2col buffer ever exists.
//
// Operands must be K-major; weight matrices that are stored N-major ((kh,kw,Cin,Cout) conv
// weights, (n_in+1, n_out) FC weights) are transposed into a stream-ordered scratch buffer first
// (<= 2 MB, microseconds).  FP32 bit patterns would be TRUNCATED to TF32 by the tensor core
// (biased); the tensor maps therefore use the TFLOAT32 data type, which makes TMA round to
// nearest while copying.
#include <cuda.h>

#include <mutex>

#include "conv_common.cuh"
#include "gemm_common.cuh"
#include "tc_ptx.cuh"

namespace uocr {

// ------------------------------------------------------------------ driver entry point (no -lcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

// rank-`rank` fp32 tensor, dims innermost first.  The three flavours differ only in data type, swizzle and L2 promotion.
static int encode_tmap(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                       const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box, CUtensorMapDataType dtype,
                       CUtensorMapSwizzle swizzle, CUtensorMapL2promotion l2) {
    EncodeTiledFn fn = encode_tiled();
    if (!fn) { set_error("cuTensorMapEncodeTiled is unavailable"); return UOCR_ERR_UNSUPPORTED; }
    cuuint64_t gd[5]; cuuint64_t gs[4]; cuuint32_t bx[5]; cuuint32_t es[5];
    for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
    CUresult r = fn(map, dtype, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle, l2, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return UOCR_ERR_UNSUPPORTED; }
    return UOCR_OK;
}

// 128-byte swizzled tcgen05 operand boxes, rounded to TF32 by the TMA unit.  MN-major 32-bit operands must use the
// 32-byte-atom flavour of the 128B swizzle (UMMA layout SWIZZLE_128B_BASE32B); K-major operands the plain 16-byte one.
static int make_tmap(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box, bool mn_major = false) {
    return encode_tmap(map, base, rank, dims, strides_bytes, box, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32,
                       mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                       CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
}

// plain (no swizzle, raw FP32) boxes: kernels that stage an image block for the CUDA cores (hourglass.cu)
int make_tmap_plain_f32(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                        const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box) {
    return encode_tmap(map, base, rank, dims, strides_bytes, box, CU_TENSOR_MAP_DATA_TYPE_FLOAT32,
                       CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
}

// plain (no swizzle) boxes whose elements the TMA unit rounds to TF32 (round to nearest): image rows that a tcgen05.mma
// reads directly as its A operand (conv_pair_rows_tc.cu)
int make_tmap_plain_tf32(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                         const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box) {
    return encode_tmap(map, base, rank, dims, strides_bytes, box, CU_TENSOR_MAP_DATA_TYPE_TFLOAT32,
                       CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B);
}

constexpr int TC_BM = 128;           // UMMA M
constexpr int TC_BK = 32;            // contraction elements per stage
constexpr int TC_THREADS = 192;
constexpr int TC_BLK = 32 * 32 * 4;  // one MN-major 32 x 32 float block (4 KB)

enum { TC_GEMM = 0, TC_CONV_FWD = 1, TC_CONV_DGRAD = 2, TC_GEMM_MN = 3, TC_CONV_WGRAD = 4 };

struct TcParams {
    float* C; int64_t ldc;
    int64_t M, N;
    int num_kb;                       // K blocks of 32 (modes 0, 1; total for mode 3)
    int nt;                           // N tile (multiple of 16 / 32 for MN-major, <= 256)
    int stages;
    const float* bias;                // length N or NULL
    int act; float alpha;
    int accumulate;                   // C += (plain read-modify-write)
    int atomic;                       // C += through atomicAdd (split-K CTAs share the tile)
    // implicit-GEMM convolution
    int ho, wo, sh, ph, pw, kh, kw;
    int cblocks;                      // channel blocks of 32 along the contraction (fwd: Cin, dgrad: Cout)
    int xtiles;                       // ceil(row width / 128)
    int h_in, w_in, cin;              // dgrad / wgrad: input tensor geometry
    // split-K
    int kb_per_split;
    // conv wgrad
    int ntaps, taps_per_cta, kbx, rows_total, rows_per_split;
    // persistent GEMM with the A operand gathered as sliding windows (Conv2DToBatchedFixedWidthed + Flatten folded
    // into the FullyConnected that follows): row (n, wi) of A, K index (k, ch) = x[n, wi + k - win_half, ch]
    int win_w, win_cblocks, win_half, win_tiles_per_img;
};

template <int MODE>
__global__ void __launch_bounds__(TC_THREADS, 2) tc_gemm_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                const __grid_constant__ CUtensorMap map_b,
                                                                const TcParams p) {
    constexpr bool MN = (MODE == TC_GEMM_MN || MODE == TC_CONV_WGRAD);
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t a_bytes = TC_BM * TC_BK * 4;
    const uint32_t b_bytes = (uint32_t)p.nt * TC_BK * 4;
    const uint32_t stage_bytes = a_bytes + ((b_bytes + 1023) & ~1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + p.stages;
    uint64_t* tmem_full = bars + 2 * p.stages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // ---- tile coordinates and this CTA's K-block list
    int64_t m0 = 0;                   // first output row of this tile (row index into C)
    int64_t m_rows = 0;               // valid rows in this tile
    int cn = 0, crow = 0, cx0 = 0;    // conv: image, row (oy for fwd, iy for dgrad), first column
    int num_kb = 0, kb0 = 0;
    uint32_t ky_mask = 0;             // dgrad: kernel rows that hit this input row
    int tap0 = 0, r0 = 0;             // wgrad
    float* cbase = p.C;
    const int n0 = blockIdx.y * p.nt;
    if (MODE == TC_GEMM) {
        m0 = (int64_t)blockIdx.x * TC_BM;
        m_rows = min((int64_t)TC_BM, p.M - m0);
        num_kb = p.num_kb;
    } else if (MODE == TC_CONV_FWD) {
        const int xt = blockIdx.x % p.xtiles, row = blockIdx.x / p.xtiles;     // row = n * ho + oy
        crow = row % p.ho; cn = row / p.ho; cx0 = xt * TC_BM;
        m0 = (int64_t)row * p.wo + cx0;
        m_rows = min(TC_BM, p.wo - cx0);
        num_kb = p.num_kb;
    } else if (MODE == TC_CONV_DGRAD) {
        const int xt = blockIdx.x % p.xtiles, row = blockIdx.x / p.xtiles;     // row = n * h_in + iy
        crow = row % p.h_in; cn = row / p.h_in; cx0 = xt * TC_BM;
        m0 = (int64_t)row * p.w_in + cx0;
        m_rows = min(TC_BM, p.w_in - cx0);
        int nky = 0;
        for (int ky = 0; ky < p.kh; ++ky) {
            const int ty = crow + p.ph - ky;
            if (ty >= 0 && ty % p.sh == 0 && ty / p.sh < p.ho) { ky_mask |= 1u << ky; ++nky; }
        }
        num_kb = nky * p.kw * p.cblocks;
    } else if (MODE == TC_GEMM_MN) {
        m0 = (int64_t)blockIdx.x * TC_BM;
        m_rows = min((int64_t)TC_BM, p.M - m0);
        kb0 = blockIdx.z * p.kb_per_split;
        num_kb = min(p.kb_per_split, p.num_kb - kb0);
    } else {
        tap0 = blockIdx.x * p.taps_per_cta;
        m_rows = min(TC_BM, (p.ntaps - tap0) * p.cin);
        cbase = p.C + (int64_t)tap0 * p.cin * p.ldc;
        r0 = blockIdx.z * p.rows_per_split;
        num_kb = min(p.rows_per_split, p.rows_total - r0) * p.kbx;
    }

    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < p.nt) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(smem_u32(&full[s]), 1);
            mbar_init(smem_u32(&empty[s]), 1);
        }
        mbar_init(smem_u32(tmem_full), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int d_ky = -1, d_left = 0;                       // dgrad: walk the set bits of ky_mask
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % p.stages;
                const uint32_t phase = (kb / p.stages) & 1;
                mbar_wait(smem_u32(&empty[s]), phase ^ 1);
                const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
                const uint32_t sb = sa + a_bytes;
                const uint32_t bar = smem_u32(&full[s]);
                if (MODE == TC_GEMM) {
                    mbar_arrive_expect_tx(bar, a_bytes + b_bytes);
                    tma_load_2d(sa, &map_a, bar, kb * TC_BK, (int)m0);
                    tma_load_2d(sb, &map_b, bar, kb * TC_BK, n0);
                } else if (MODE == TC_CONV_FWD) {
                    mbar_arrive_expect_tx(bar, a_bytes + b_bytes);
                    const int tap = kb / p.cblocks, cb = kb % p.cblocks;
                    const int ky = tap / p.kw, kx = tap % p.kw;
                    tma_load_4d(sa, &map_a, bar, cb * TC_BK, cx0 + kx - p.pw, crow * p.sh + ky - p.ph, cn);
                    tma_load_2d(sb, &map_b, bar, kb * TC_BK, n0);
                } else if (MODE == TC_CONV_DGRAD) {
                    mbar_arrive_expect_tx(bar, a_bytes + b_bytes);
                    if (d_left == 0) {                       // next kernel row with the right parity
                        do { ++d_ky; } while (!((ky_mask >> d_ky) & 1u));
                        d_left = p.kw * p.cblocks;
                    }
                    const int within = p.kw * p.cblocks - d_left;
                    --d_left;
                    const int kx = within / p.cblocks, cb = within % p.cblocks;
                    const int oy = (crow + p.ph - d_ky) / p.sh;
                    // A: dy[n, oy, ix + pw - kx, co-block];  B: w[ky, kx, :, co-block] as (Cin rows, 32 cols)
                    tma_load_4d(sa, &map_a, bar, cb * TC_BK, cx0 + p.pw - kx, oy, cn);
                    tma_load_2d(sb, &map_b, bar, cb * TC_BK, (d_ky * p.kw + kx) * p.cin);
                } else if (MODE == TC_GEMM_MN) {
                    const int k = (kb0 + kb) * TC_BK;
                    int nblk = 0;
                    for (int i = 0; i < TC_BM / 32; ++i) nblk += (m0 + 32 * i < p.M);
                    for (int j = 0; j < p.nt / 32; ++j) nblk += (n0 + 32 * j < p.N);
                    mbar_arrive_expect_tx(bar, (uint32_t)nblk * TC_BLK);
                    for (int i = 0; i < TC_BM / 32; ++i)
                        if (m0 + 32 * i < p.M) tma_load_2d(sa + i * TC_BLK, &map_a, bar, (int)m0 + 32 * i, k);
                    for (int j = 0; j < p.nt / 32; ++j)
                        if (n0 + 32 * j < p.N) tma_load_2d(sb + j * TC_BLK, &map_b, bar, n0 + 32 * j, k);
                } else {
                    const int row = r0 + kb / p.kbx, ox0 = (kb % p.kbx) * TC_BK;      // row = n * ho + oy
                    const int oy = row % p.ho, n = row / p.ho;
                    const int cbl = p.cin / 32;
                    int nblk = p.nt / 32;
                    for (int i = 0; i < TC_BM / 32; ++i) nblk += (tap0 + i / cbl < p.ntaps);
                    mbar_arrive_expect_tx(bar, (uint32_t)nblk * TC_BLK);
                    for (int i = 0; i < TC_BM / 32; ++i) {
                        const int tap = tap0 + i / cbl;
                        if (tap >= p.ntaps) continue;
                        const int ky = tap / p.kw, kx = tap % p.kw;
                        tma_load_4d(sa + i * TC_BLK, &map_a, bar, (i % cbl) * 32, ox0 + kx - p.pw,
                                    oy * p.sh + ky - p.ph, n);
                    }
                    for (int j = 0; j < p.nt / 32; ++j) tma_load_4d(sb + j * TC_BLK, &map_b, bar, j * 32, ox0, oy, n);
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            // instruction descriptor: D = F32, A = B = TF32, N >> 3, M >> 4, major bits for MN-major operands
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (MN ? (1u << 15) | (1u << 16) : 0u) |
                                   ((uint32_t)(p.nt >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            for (int kb = 0; kb < num_kb; ++kb) {
                const int s = kb % p.stages;
                const uint32_t phase = (kb / p.stages) & 1;
                mbar_wait(smem_u32(&full[s]), phase);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
                if (!MN) {
                    const uint64_t da = make_kmajor_sw128_desc(sa);
                    const uint64_t db = make_kmajor_sw128_desc(sa + a_bytes);
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k)      // +32 bytes inside the swizzled 128-byte row
                        tc_mma_tf32(tmem_base, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc,
                                    (kb > 0 || k > 0) ? 1u : 0u);
                } else {
                    const uint64_t da = make_mnmajor_sw128_desc(sa, TC_BLK);
                    const uint64_t db = make_mnmajor_sw128_desc(sa + a_bytes, TC_BLK);
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k)      // next 8 K-rows = next 1024-byte atom
                        tc_mma_tf32(tmem_base, da + (uint64_t)(k * 64), db + (uint64_t)(k * 64), idesc,
                                    (kb > 0 || k > 0) ? 1u : 0u);
                }
                tc_commit(smem_u32(&empty[s]));             // frees the stage when these MMAs retire
            }
            if (num_kb > 0) tc_commit(smem_u32(tmem_full)); // accumulator complete
        }
    } else {
        // ===================== epilogue (warps 2..5) =====================
        const int q = warp & 3;                              // TMEM lane quarter this warp may read
        if (num_kb > 0) {
            mbar_wait(smem_u32(tmem_full), 0);
            tc_fence_after();
        }
        const int r = q * 32 + lane;                         // row within the tile
        const bool row_ok = r < m_rows;
        float* crow_ptr = cbase + (m0 + r) * p.ldc + n0;
        for (int c0 = 0; c0 < p.nt; c0 += 32) {
            float v[32];
            if (num_kb > 0) {
                tc_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = 0.f;     // no tap reaches this row (dgrad)
            }
            if (!row_ok) continue;
            const int ncols = (int)min((int64_t)32, p.N - n0 - c0);
            if (ncols <= 0) continue;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                if (j < ncols) {
                    float t = v[j] + (p.bias ? __ldg(p.bias + n0 + c0 + j) : 0.f);
                    v[j] = apply_act(t, p.act, p.alpha);
                }
            }
            // (every loop over v[] is fully unrolled with predicates: a runtime index would push the
            // accumulator fragment into local memory -- that made the epilogue the bottleneck)
            float* dst = crow_ptr + c0;
            if (p.atomic) {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (j < ncols) atomicAdd(dst + j, v[j]);
            } else if (ncols == 32 && !p.accumulate && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0)) {
#pragma unroll
                for (int j = 0; j < 32; j += 4)
                    *reinterpret_cast<float4*>(dst + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (j < ncols) dst[j] = p.accumulate ? dst[j] + v[j] : v[j];
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

static int pick_stages(int nt, size_t* smem_bytes) {
    const size_t a_bytes = TC_BM * TC_BK * 4;
    const size_t b_bytes = (((size_t)nt * TC_BK * 4) + 1023) & ~(size_t)1023;
    // 70 KB: ~3 CTAs / SM, so that their prologues and epilogues overlap other CTAs' main loops
    const size_t budget = (size_t)70 * 1024;
    int stages = (int)((budget - 2048) / (a_bytes + b_bytes));
    if (stages > 8) stages = 8;
    if (stages < 2) stages = 2;
    *smem_bytes = (size_t)stages * (a_bytes + b_bytes) + 1024 /* align slack */ + (2 * stages + 2) * 8 + 64;
    return stages;
}

template <int MODE>
static int launch_tc(const CUtensorMap& ma, const CUtensorMap& mb, TcParams& p, dim3 grid, cudaStream_t st) {
    size_t smem = 0;
    p.stages = pick_stages(p.nt, &smem);
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(tc_gemm_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             227 * 1024);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
        configured = true;
    }
    tc_gemm_kernel<MODE><<<grid, TC_THREADS, smem, st>>>(ma, mb, p);
    UOCR_LAUNCHED("tc_gemm_tf32");
    return UOCR_OK;
}

static int pick_nt(int64_t n) {
    if (n >= 64) return 64;                   // full-rate N; wider tiles amortise the A reads
    return (int)(((n + 15) / 16) * 16);
}

static int tc_gemm_tn_persistent(const float* A, int64_t lda, const float* Bt, int64_t ldb, float* C, int64_t ldc,
                                 int64_t M, int64_t N, int64_t K, const float* bias, int act, float alpha,
                                 int accumulate, cudaStream_t st);

// D[M,N] = act(A[M,K] . Bt[N,K]^T + bias); A, Bt K-major (rows contiguous in K)
int tc_gemm_tn(const float* A, int64_t lda, const float* Bt, int64_t ldb, float* C, int64_t ldc, int64_t M,
               int64_t N, int64_t K, const float* bias, int act, float alpha, int accumulate, cudaStream_t st) {
    if ((lda % 4) || (ldb % 4) || ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(Bt)) & 15))
        return UOCR_ERR_UNSUPPORTED;            // TMA: 16-byte aligned base and row pitch
    if (M <= 0 || N <= 0 || K <= 0 || M > 0x7fffffff || K > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    {
        // enough 128 x NT tiles to keep most SMs busy (dense_2: 128 tiles, 46 -> 34 us): >= 96, ~2/3 of the SMs
        const int64_t nt = N >= 256 ? 256 : ((N + 15) / 16) * 16;
        if (N >= 128 && ceil_div(M, TC_BM) * ceil_div(N, nt) >= 96) {
            const int rc = tc_gemm_tn_persistent(A, lda, Bt, ldb, C, ldc, M, N, K, bias, act, alpha, accumulate, st);
            if (rc != UOCR_ERR_UNSUPPORTED) return rc;
        }
    }
    TcParams p{};
    p.C = C; p.ldc = ldc; p.M = M; p.N = N; p.num_kb = (int)ceil_div(K, TC_BK);
    p.nt = pick_nt(N);
    p.bias = bias; p.act = act; p.alpha = alpha; p.accumulate = accumulate;
    CUtensorMap ma, mb;
    const uint64_t da[2] = {(uint64_t)K, (uint64_t)M}, sa[1] = {(uint64_t)lda * 4};
    const uint32_t ba[2] = {TC_BK, TC_BM};
    int rc = make_tmap(&ma, A, 2, da, sa, ba);
    if (rc) return rc;
    const uint64_t db[2] = {(uint64_t)K, (uint64_t)N}, sb[1] = {(uint64_t)ldb * 4};
    const uint32_t bb[2] = {TC_BK, (uint32_t)p.nt};
    rc = make_tmap(&mb, Bt, 2, db, sb, bb);
    if (rc) return rc;
    dim3 grid((unsigned)ceil_div(M, TC_BM), (unsigned)ceil_div(N, p.nt));
    return launch_tc<TC_GEMM>(ma, mb, p, grid, st);
}

// ------------------------------------------------------------------------------------------
// Persistent variant for the large K-major GEMMs (FullyConnected forward / dgrad at batch >= ~10k rows).
// One CTA per SM loops over 128 x NT output tiles (NT up to 256: 43.7 flop per L2 byte instead of 21.8
// for the 128 x 64 tiles above, which ncu showed L2-bandwidth bound).  The accumulator is DOUBLE
// BUFFERED in TMEM (2 x NT columns): while the four epilogue warps drain tile i (tcgen05.ld -> bias ->
// activation -> global), the MMA warp already accumulates tile i + 1 and the TMA warp runs further ahead
// through the shared-memory ring, so neither the pipeline fill nor the epilogue is exposed per tile.
//   full[s] / empty[s]          : TMA <-> MMA, per shared-memory stage
//   tmem_full[b] / tmem_empty[b]: MMA <-> epilogue, per accumulator buffer (empty: 4 arrivals, one per warp)
// Tiles are walked n-tile-major so the ~148 CTAs working at the same time share one B tile in L2.
// ------------------------------------------------------------------------------------------

constexpr int TCP_THREADS = 64 + 8 * 32;   // TMA warp, MMA warp, 8 epilogue warps (2 per TMEM lane quarter)

// PAIR: two CTAs of a cluster (one TPC) share every tile: UMMA M = 256 with cta_group::2.  CTA r stages rows
// [128 r, 128 r + 128) of A and rows [nt/2 r, ..) of the B tile (32 KB per stage instead of 48 KB), the leader issues
// the MMAs for both tensor cores, every CTA drains its own 128 accumulator rows.  Shared-memory traffic per MMA drops
// from 12 KB read + 12 KB written to 8 + 8 KB per SM, which is what capped the single-CTA kernel (DESIGN.md).
// `m_tiles` counts tiles of 128 (256 for PAIR) rows.
template <bool PAIR>
__global__ void __launch_bounds__(TCP_THREADS, 1) tc_gemm_persistent_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                           const __grid_constant__ CUtensorMap map_b,
                                                                           const TcParams p, int m_tiles, int n_tiles) {
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
    const int cta = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int ncta = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t a_bytes = TC_BM * TC_BK * 4;
    const uint32_t b_bytes = (uint32_t)(PAIR ? p.nt / 2 : p.nt) * TC_BK * 4;
    const uint32_t stage_bytes = a_bytes + ((b_bytes + 1023) & ~1023u);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + p.stages;
    uint64_t* tmem_full = bars + 2 * p.stages;            // [2]
    uint64_t* tmem_empty = bars + 2 * p.stages + 2;       // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 4);
    // bias row staged once per CTA (zero padded; all zeros without a bias): the epilogue reads it with
    // broadcast 128-bit shared loads instead of 32 dependent global loads per chunk (ncu: the epilogue
    // warps sat on the long scoreboard of those loads and the tensor pipe idled at 15 %)
    float* s_bias = reinterpret_cast<float*>(bars + 2 * p.stages + 6);
    float* s_stage = s_bias + n_tiles * p.nt;               // 8 epilogue warps x 2 KB transpose staging

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int total_tiles = m_tiles * n_tiles;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < 2 * p.nt) tmem_cols <<= 1;
    for (int i = threadIdx.x; i < n_tiles * p.nt; i += TCP_THREADS)
        s_bias[i] = (p.bias && i < p.N) ? __ldg(p.bias + i) : 0.f;

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(smem_u32(&full[s]), 1);
            mbar_init(smem_u32(&empty[s]), 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(smem_u32(&tmem_full[b]), 1);
            mbar_init(smem_u32(&tmem_empty[b]), PAIR ? 16 : 8);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                         ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                         ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if (PAIR) cluster_sync_all();           // the peer's barriers are initialised before anything signals them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            int it = 0;                                    // running K-block counter across tiles
            for (int tile = cta; tile < total_tiles; tile += ncta) {
                // N index fastest: the CTAs that run at the same time share a few row blocks of A, which then
                // comes from DRAM once (B, the weights, is L2-resident anyway).  With the M index fastest a 268 MB
                // A was streamed from DRAM once per N tile (ncu: 1.09 GB read, L2 hit rate 44 %, DRAM 73 % busy).
                const int mt = (tile / n_tiles) * (PAIR ? 2 : 1) + (int)rank;        // this CTA's 128-row tile
                const int m0 = mt * TC_BM, n0 = (tile % n_tiles) * p.nt + (PAIR ? (int)rank * (p.nt / 2) : 0);
                // Every CTA walks the K blocks from a different starting block (the sum does not care about
                // the order): the ~148 CTAs that share one B tile then read different lines of it at any
                // moment instead of hammering the same L2 slices.
                const int rot = cta % p.num_kb;
                for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
                    const int s = it % p.stages;
                    const uint32_t phase = (it / p.stages) & 1;
                    mbar_wait(smem_u32(&empty[s]), phase ^ 1);
                    const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
                    // PAIR: both CTAs' copies complete on the LEADER's barrier, which expects the bytes of both
                    const uint32_t bar = PAIR ? mapa_rank(smem_u32(&full[s]), 0) : smem_u32(&full[s]);
                    if (!PAIR) mbar_arrive_expect_tx(bar, a_bytes + b_bytes);
                    else if (rank == 0) mbar_arrive_expect_tx(smem_u32(&full[s]), 2 * (a_bytes + b_bytes));
                    const int kbr = kb + rot >= p.num_kb ? kb + rot - p.num_kb : kb + rot;
                    const int kk = kbr * TC_BK;
                    if (p.win_w) {                         // 128 consecutive window positions of one image: a 3-D box
                        const int k = kbr / p.win_cblocks, cb = kbr - k * p.win_cblocks;
                        const int wx = (mt % p.win_tiles_per_img) * TC_BM + k - p.win_half, wn = mt / p.win_tiles_per_img;
                        if (PAIR) tma_load_3d_pair(sa, &map_a, bar, cb * TC_BK, wx, wn);
                        else tma_load_3d(sa, &map_a, bar, cb * TC_BK, wx, wn);
                    } else if (PAIR) {
                        tma_load_2d_pair(sa, &map_a, bar, kk, m0);
                    } else {
                        tma_load_2d(sa, &map_a, bar, kk, m0);
                    }
                    if (PAIR) tma_load_2d_pair(sa + a_bytes, &map_b, bar, kk, n0);
                    else tma_load_2d(sa + a_bytes, &map_b, bar, kk, n0);
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0 && rank == 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.nt >> 3) << 17) |
                                   ((uint32_t)((PAIR ? 2 * TC_BM : TC_BM) >> 4) << 24);
            int it = 0, local = 0;
            for (int tile = cta; tile < total_tiles; tile += ncta, ++local) {
                const int buf = local & 1;
                mbar_wait(smem_u32(&tmem_empty[buf]), ((local >> 1) & 1) ^ 1);   // epilogue drained this buffer
                tc_fence_after();
                const uint32_t tacc = tmem_base + (uint32_t)(buf * p.nt);
                for (int kb = 0; kb < p.num_kb; ++kb, ++it) {
                    const int s = it % p.stages;
                    const uint32_t phase = (it / p.stages) & 1;
                    mbar_wait(smem_u32(&full[s]), phase);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
                    const uint64_t da = make_kmajor_sw128_desc(sa);
                    const uint64_t db = make_kmajor_sw128_desc(sa + a_bytes);
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k) {
                        if (PAIR) tc_mma_tf32_pair(tacc, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc,
                                                   (kb > 0 || k > 0) ? 1u : 0u);
                        else tc_mma_tf32(tacc, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc,
                                         (kb > 0 || k > 0) ? 1u : 0u);
                    }
                    if (PAIR) tc_commit_pair(smem_u32(&empty[s]));      // frees the stage in both CTAs
                    else tc_commit(smem_u32(&empty[s]));
                }
                if (PAIR) tc_commit_pair(smem_u32(&tmem_full[buf]));
                else tc_commit(smem_u32(&tmem_full[buf]));
            }
        }
    } else {
        // ===================== epilogue (warps 2..9) =====================
        // Two warps per TMEM lane quarter (q = warp % 4), alternating 16-column half-chunks.  The tile is
        // drained at MMA pace only if (a) the next tcgen05.ld is in flight while the current half-chunk is
        // processed and (b) global stores are row-contiguous: thread = accumulator row after tcgen05.ld, so
        // a direct 128-bit store touches 32 cache lines; the 32 x 16 block is transposed through a per-warp
        // 2 KB staging block (16-byte granules XOR-swizzled with the row, conflict-free both ways) and
        // leaves as 8 rows x 64 contiguous bytes per store instruction.
        const int e = warp - 2, q = warp & 3, half = e >> 2;
        float4* stg = reinterpret_cast<float4*>(s_stage) + e * 128;
        const int nhc = p.nt >> 4;                           // half-chunks per tile
        const int sub_r = lane >> 2, sub_g = lane & 3;       // store phase: row within a group of 8, granule
        const bool vec_ok = ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0);
        int local = 0;
        // the accumulator buffer is released to the MMA issuer, which lives in the leader CTA
        auto release = [&](int buf) {
            if (PAIR) mbar_arrive_cluster(mapa_rank(smem_u32(&tmem_empty[buf]), 0));
            else mbar_arrive(smem_u32(&tmem_empty[buf]));
        };
        for (int tile = cta; tile < total_tiles; tile += ncta, ++local) {
            const int buf = local & 1;
            const int64_t row0 = ((int64_t)(tile / n_tiles) * (PAIR ? 2 : 1) + rank) * TC_BM + q * 32;   // first row of this warp
            const int n0 = (tile % n_tiles) * p.nt;
            mbar_wait(smem_u32(&tmem_full[buf]), (local >> 1) & 1);
            tc_fence_after();
            const uint32_t tq = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.nt);
            uint32_t va[16], vb[16];
            auto handle = [&](uint32_t* cur, uint32_t* nxt, int hc) {
                tc_wait_ld();                                // cur[] is in registers
                if (hc + 2 < nhc) {
                    tc_ld16_nowait(tq + (uint32_t)((hc + 2) * 16), nxt);
                } else {                                     // this warp has read all its columns of the buffer
                    tc_fence_before();
                    if (lane == 0) release(buf);
                }
                const int c = n0 + hc * 16;
                const int ncols = (int)min((int64_t)16, p.N - c);
                if (ncols <= 0) return;                      // warp-uniform
                const float4* bs = reinterpret_cast<const float4*>(s_bias + c);
                __syncwarp();                                // earlier reads of the staging block are done
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    const float4 b4 = bs[g];
                    stg[lane * 4 + (g ^ ((lane >> 1) & 3))] =
                        make_float4(apply_act_fast(__uint_as_float(cur[4 * g]) + b4.x, p.act, p.alpha),
                                    apply_act_fast(__uint_as_float(cur[4 * g + 1]) + b4.y, p.act, p.alpha),
                                    apply_act_fast(__uint_as_float(cur[4 * g + 2]) + b4.z, p.act, p.alpha),
                                    apply_act_fast(__uint_as_float(cur[4 * g + 3]) + b4.w, p.act, p.alpha));
                }
                __syncwarp();
                if (vec_ok && ncols == 16) {
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int rr = 8 * i + sub_r;
                        const float4 o = stg[rr * 4 + (sub_g ^ ((rr >> 1) & 3))];
                        if (row0 + rr >= p.M) continue;
                        float* dst = p.C + (row0 + rr) * p.ldc + c + 4 * sub_g;
                        if (p.accumulate) {
                            const float4 c4 = *reinterpret_cast<const float4*>(dst);
                            *reinterpret_cast<float4*>(dst) = make_float4(c4.x + o.x, c4.y + o.y, c4.z + o.z, c4.w + o.w);
                        } else {
                            *reinterpret_cast<float4*>(dst) = o;
                        }
                    }
                } else {
                    // rows that are not 16-byte multiples (dense_3: n_out = 162) or a ragged last chunk: scalar stores,
                    // a half-warp per row -- 16 consecutive floats = 64 contiguous bytes, 2 rows per instruction (the
                    // float4-shaped form wrote words 16 bytes apart: 16 sectors per instruction instead of 4-6)
                    const float* sf = reinterpret_cast<const float*>(stg);
                    const int col = lane & 15;
#pragma unroll 4
                    for (int i = 0; i < 16; ++i) {
                        const int rr = 2 * i + (lane >> 4);
                        const float o = sf[(rr * 4 + ((col >> 2) ^ ((rr >> 1) & 3))) * 4 + (col & 3)];
                        if (row0 + rr >= p.M || col >= ncols) continue;
                        float* dst = p.C + (row0 + rr) * p.ldc + c + col;
                        *dst = p.accumulate ? *dst + o : o;
                    }
                }
            };
            if (half < nhc) tc_ld16_nowait(tq + (uint32_t)(half * 16), va);
            else { tc_fence_before(); if (lane == 0) release(buf); }
            for (int hc = half; hc < nhc; hc += 4) {
                handle(va, vb, hc);
                if (hc + 2 < nhc) handle(vb, va, hc + 2);
            }
        }
    }

    tc_fence_before();
    if (PAIR) cluster_sync_all();           // the leader's MMAs read the peer's shared memory until the last commit
    else __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

struct WindowGeom { int64_t n, w, c; int width; };      // A = sliding windows over x (n, w, c): see TcParams::win_*

static int tc_gemm_tn_persistent_impl(const float* A, int64_t lda, const WindowGeom* win, const float* Bt, int64_t ldb,
                                      float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias, int act,
                                      float alpha, int accumulate, cudaStream_t st);

static int tc_gemm_tn_persistent(const float* A, int64_t lda, const float* Bt, int64_t ldb, float* C, int64_t ldc,
                                 int64_t M, int64_t N, int64_t K, const float* bias, int act, float alpha,
                                 int accumulate, cudaStream_t st) {
    return tc_gemm_tn_persistent_impl(A, lda, nullptr, Bt, ldb, C, ldc, M, N, K, bias, act, alpha, accumulate, st);
}

static int tc_gemm_tn_persistent_impl(const float* A, int64_t lda, const WindowGeom* win, const float* Bt, int64_t ldb,
                                      float* C, int64_t ldc, int64_t M, int64_t N, int64_t K, const float* bias, int act,
                                      float alpha, int accumulate, cudaStream_t st) {
    TcParams p{};
    p.C = C; p.ldc = ldc; p.M = M; p.N = N; p.num_kb = (int)ceil_div(K, TC_BK);
    if (win) {
        p.win_w = (int)win->w; p.win_cblocks = (int)(win->c / TC_BK); p.win_half = win->width / 2;
        p.win_tiles_per_img = (int)(win->w / TC_BM);
    }
    p.nt = N >= 256 ? 256 : (int)(((N + 15) / 16) * 16);
    p.bias = bias; p.act = act; p.alpha = alpha; p.accumulate = accumulate;
    // CTA pairs (cta_group::2) need full 256-column tiles.  Measured (tools/gemmbench.py): no gain where the fixed
    // costs dominate (dense_1 forward, 16 K blocks x 3.5 tiles per CTA: 47 us either way), +5 % with K = 1024
    // (its dgrad), +10 % at 14 tiles per CTA (504 -> 556 TFLOP/s).  UOCR_TC_PAIR = 0 / 1 forces never / always.
    const char* pe = getenv("UOCR_TC_PAIR");
    const int pair_mode = pe ? atoi(pe) : -1;
    const bool pair_fits = p.nt == 256 && M >= 4096;            // nt = 128 pairs work but gain nothing (dense_2: 21.5 vs 20.4 us)
    const bool pair = pair_fits && (pair_mode > 0 || (pair_mode < 0 && (K >= 1024 || M * N >= ((int64_t)1 << 25))));
    const size_t a_bytes = TC_BM * TC_BK * 4;
    const size_t b_bytes = (((size_t)(pair ? p.nt / 2 : p.nt) * TC_BK * 4) + 1023) & ~(size_t)1023;
    p.stages = (int)((196 * 1024) / (a_bytes + b_bytes));
    if (p.stages > 8) p.stages = 8;
    if (p.stages < 2) return UOCR_ERR_UNSUPPORTED;
    const size_t bias_floats = (size_t)ceil_div(N, p.nt) * p.nt;
    if (bias_floats > 2048) return UOCR_ERR_UNSUPPORTED;
    const size_t smem = (size_t)p.stages * (a_bytes + b_bytes) + 1024 + (2 * p.stages + 6) * 8 + bias_floats * 4 + 8 * 2048 + 64;
    CUtensorMap ma, mb;
    int rc;
    if (win) {                                            // x (n, w, c): out-of-range window columns read as zeros
        const uint64_t da[3] = {(uint64_t)win->c, (uint64_t)win->w, (uint64_t)win->n};
        const uint64_t sa[2] = {(uint64_t)win->c * 4, (uint64_t)win->w * win->c * 4};
        const uint32_t ba[3] = {TC_BK, TC_BM, 1};
        rc = make_tmap(&ma, A, 3, da, sa, ba);
    } else {
        const uint64_t da[2] = {(uint64_t)K, (uint64_t)M}, sa[1] = {(uint64_t)lda * 4};
        const uint32_t ba[2] = {TC_BK, TC_BM};
        rc = make_tmap(&ma, A, 2, da, sa, ba);
    }
    if (rc) return rc;
    const uint64_t db[2] = {(uint64_t)K, (uint64_t)N}, sb[1] = {(uint64_t)ldb * 4};
    const uint32_t bb[2] = {TC_BK, (uint32_t)(pair ? p.nt / 2 : p.nt)};
    rc = make_tmap(&mb, Bt, 2, db, sb, bb);
    if (rc) return rc;
    static int num_sms = 0, num_pairs = 0;
    if (!num_sms) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev);
        cudaError_t e = cudaFuncSetAttribute(tc_gemm_persistent_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             227 * 1024);
        if (e == cudaSuccess)
            e = cudaFuncSetAttribute(tc_gemm_persistent_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     227 * 1024);
        if (e != cudaSuccess) { num_sms = 0; set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
    }
    const int n_tiles = (int)ceil_div(N, p.nt);
    if (pair) {
        const int m_tiles = (int)ceil_div(M, 2 * TC_BM);
        const int64_t tiles = (int64_t)m_tiles * n_tiles;
        cudaLaunchConfig_t cfg{};
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.blockDim = dim3(TCP_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = st; cfg.attrs = attr; cfg.numAttrs = 1;
        if (!num_pairs) {
            cfg.gridDim = dim3((unsigned)num_sms & ~1u);
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, tc_gemm_persistent_kernel<true>, &cfg) != cudaSuccess || n <= 0) {
                cudaGetLastError();
                n = num_sms / 2;
            }
            num_pairs = n < num_sms / 2 ? n : num_sms / 2;
        }
        cfg.gridDim = dim3(2u * (unsigned)(tiles < num_pairs ? tiles : num_pairs));
        cudaError_t e = cudaLaunchKernelEx(&cfg, tc_gemm_persistent_kernel<true>, ma, mb, p, m_tiles, n_tiles);
        if (e != cudaSuccess) { set_error("cluster launch: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
        UOCR_LAUNCHED("tc_gemm_persistent_pair_tf32");
        return UOCR_OK;
    }
    const int m_tiles = (int)ceil_div(M, TC_BM);
    const int64_t tiles = (int64_t)m_tiles * n_tiles;
    const unsigned grid = (unsigned)(tiles < num_sms ? tiles : num_sms);
    tc_gemm_persistent_kernel<false><<<grid, TCP_THREADS, smem, st>>>(ma, mb, p, m_tiles, n_tiles);
    UOCR_LAUNCHED("tc_gemm_persistent_tf32");
    return UOCR_OK;
}

// C[M,N] += At[K,M]^T . B[K,N]   (both operands stored with the contraction index K as the ROW index:
// "MN-major"), split over K, partial tiles added with atomicAdd.  C must hold the value to add to.
int tc_gemm_mn_atomic(const float* At, int64_t lda, const float* B, int64_t ldb, float* C, int64_t ldc,
                      int64_t M, int64_t N, int64_t K, cudaStream_t st) {
    if ((lda % 4) || (ldb % 4) || ((reinterpret_cast<uintptr_t>(At) | reinterpret_cast<uintptr_t>(B)) & 15))
        return UOCR_ERR_UNSUPPORTED;
    if (M <= 0 || N <= 0 || K <= 0 || M > 0x7fffffff || K > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    TcParams p{};
    p.C = C; p.ldc = ldc; p.M = M; p.N = N; p.num_kb = (int)ceil_div(K, TC_BK);
    p.nt = N >= 256 ? 256 : (int)(((N + 31) / 32) * 32);
    p.act = UOCR_ACT_NONE; p.atomic = 1;
    const int64_t tiles = ceil_div(M, TC_BM) * ceil_div(N, p.nt);
    // split K so that tiles x splits is about ONE wave of CTAs and every CTA owns >= 8 K blocks: the partial tiles meet in
    // atomicAdds, and two waves of shorter CTAs (the first version) doubled that traffic for nothing -- measured on the
    // Char head's weight gradients (tools/trainprof.py): dense_1 0.185 -> 0.149 ms, dense_2 0.105 -> 0.097, dense_3
    // (one tile, 128-way contention) 0.085 -> 0.071
    int64_t splits = (148 + tiles - 1) / tiles;
    if (splits > p.num_kb / 8) splits = p.num_kb / 8;
    if (splits < 1) splits = 1;
    if (splits > 65535) splits = 65535;
    p.kb_per_split = (int)ceil_div(p.num_kb, splits);
    splits = ceil_div(p.num_kb, p.kb_per_split);
    CUtensorMap ma, mb;
    const uint64_t da[2] = {(uint64_t)M, (uint64_t)K}, sa[1] = {(uint64_t)lda * 4};
    const uint32_t box[2] = {32, TC_BK};
    int rc = make_tmap(&ma, At, 2, da, sa, box, true);
    if (rc) return rc;
    const uint64_t db[2] = {(uint64_t)N, (uint64_t)K}, sb[1] = {(uint64_t)ldb * 4};
    rc = make_tmap(&mb, B, 2, db, sb, box, true);
    if (rc) return rc;
    dim3 grid((unsigned)ceil_div(M, TC_BM), (unsigned)ceil_div(N, p.nt), (unsigned)splits);
    return launch_tc<TC_GEMM_MN>(ma, mb, p, grid, st);
}

// ------------------------------------------------------------------ small transposes into scratch
// dst[c][r] = src[r][c]   (rows x cols -> cols x rows), 32x32 smem tiles
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                        int rows, int cols, int64_t src_pitch, int64_t dst_pitch) {
    __shared__ float t[32][33];
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int i = ty; i < 32; i += 8) {
        const int r = r0 + i, c = c0 + tx;
        t[i][tx] = (r < rows && c < cols) ? src[(int64_t)r * src_pitch + c] : 0.f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, r = r0 + tx;
        if (c < cols && r < rows) dst[(int64_t)c * dst_pitch + r] = t[tx][i];
    }
}

static int transpose_async(const float* src, float* dst, int rows, int cols, int64_t src_pitch, int64_t dst_pitch,
                           cudaStream_t st) {
    dim3 grid((cols + 31) / 32, (rows + 31) / 32);
    transpose_kernel<<<grid, 256, 0, st>>>(src, dst, rows, cols, src_pitch, dst_pitch);
    UOCR_LAUNCHED("transpose");
    return UOCR_OK;
}

// ------------------------------------------------------------------ FullyConnected
int fc_fwd_fast(int math_mode, const float* x, const float* w, const float* w_kmajor, float* y, int64_t batch,
                int64_t n_in, int64_t n_out, int act, float alpha, cudaStream_t st) {
    if (math_mode != UOCR_MATH_TF32) return UOCR_ERR_UNSUPPORTED;
    if (n_in % 4 || batch < 128 || n_in < 32 || n_out < 16) return UOCR_ERR_UNSUPPORTED;
    if (!encode_tiled()) return UOCR_ERR_UNSUPPORTED;
    // W (n_in + 1, n_out) is N-major: the tensor cores want the weight rows K-major, Wt (n_out, n_in) -- either the
    // caller's cached copy (uocr_weights_to_kmajor) or a transpose into stream-ordered scratch; the bias row stays
    Scratch wt(st);
    if (!w_kmajor) {
        int rc = wt.alloc(sizeof(float) * n_out * n_in);
        if (rc) return rc;
        rc = transpose_async(w, (float*)wt.ptr, (int)n_in, (int)n_out, n_out, n_in, st);
        if (rc) return rc;
        w_kmajor = (const float*)wt.ptr;
    }
    return tc_gemm_tn(x, n_in, w_kmajor, n_in, y, n_out, batch, n_out, n_in, w + n_in * n_out, act, alpha, 0, st);
}

// y (n*w, n_out) = act([windows(x), 1] . W): Conv2DToBatchedFixedWidthed(width) + Flatten + FullyConnected in one GEMM whose
// A tiles are gathered from x (n, 1, w, c) by TMA (an implicit 1-D convolution over the width): the (n*w, width*c)
// window matrix (33 MB for Char at batch 64) is never written or read.
int fc_window_fwd_fast(int math_mode, const float* x, const float* w, const float* w_kmajor, float* y, int64_t n,
                       int64_t wd, int64_t c, int width, int64_t n_out, int act, float alpha, cudaStream_t st) {
    const int64_t n_in = (int64_t)width * c, batch = n * wd;
    if (math_mode != UOCR_MATH_TF32 || !encode_tiled()) return UOCR_ERR_UNSUPPORTED;
    if (wd % TC_BM || c % TC_BK || n_out < 128 || n_out % 4 || (reinterpret_cast<uintptr_t>(x) & 15)) return UOCR_ERR_UNSUPPORTED;
    const int64_t nt = n_out >= 256 ? 256 : ((n_out + 15) / 16) * 16;
    if (ceil_div(batch, TC_BM) * ceil_div(n_out, nt) < 96) return UOCR_ERR_UNSUPPORTED;
    Scratch wt(st);
    if (!w_kmajor) {
        int rc = wt.alloc(sizeof(float) * n_out * n_in);
        if (rc) return rc;
        rc = transpose_async(w, (float*)wt.ptr, (int)n_in, (int)n_out, n_out, n_in, st);
        if (rc) return rc;
        w_kmajor = (const float*)wt.ptr;
    }
    const WindowGeom win{n, wd, c, width};
    return tc_gemm_tn_persistent_impl(x, 0, &win, w_kmajor, n_in, y, n_out, batch, n_out, n_in, w + n_in * n_out, act,
                                      alpha, 0, st);
}

int weights_to_kmajor(const float* w, float* wt, int64_t k_rows, int64_t n_cols, cudaStream_t st) {
    if (k_rows > 0x7fffffff || n_cols > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    return transpose_async(w, wt, (int)k_rows, (int)n_cols, n_cols, k_rows, st);
}

// out[c] += sum_r src[r][c] : bias gradients (the "ones" column of [x, 1]^T . dy).  Rows are split over
// gridDim.y blocks (enough CTAs to pull the matrix at HBM speed -- one block per 32 columns took 1.2 ms
// for Char conv_2's 21 MB); each block adds its partial column sums with atomicAdd, like the split-K
// weight gradients they accompany.
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ src, int64_t rows, int cols,
                                                     int64_t rows_per_block, float* __restrict__ out) {
    __shared__ float red[8][33];
    const int c = blockIdx.x * 32 + (threadIdx.x & 31);
    const int ty = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.y * rows_per_block;
    const int64_t r1 = min(rows, r0 + rows_per_block);
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
    if (c < cols) {
        int64_t r = r0 + ty;
        for (; r + 24 < r1; r += 32) {                       // 4 independent loads in flight per thread
            s0 += __ldg(src + r * cols + c);
            s1 += __ldg(src + (r + 8) * cols + c);
            s2 += __ldg(src + (r + 16) * cols + c);
            s3 += __ldg(src + (r + 24) * cols + c);
        }
        for (; r < r1; r += 8) s0 += __ldg(src + r * cols + c);
    }
    red[ty][threadIdx.x & 31] = (s0 + s1) + (s2 + s3);
    __syncthreads();
    if (ty == 0 && c < cols) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += red[k][threadIdx.x];
        atomicAdd(out + c, t);
    }
}

static int colsum_async(const float* src, int64_t rows, int cols, float* out, int accumulate, cudaStream_t st) {
    if (!accumulate) {
        cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float) * cols, st);
        if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
    }
    const int gx = (cols + 31) / 32;
    int64_t gy = ceil_div(148 * 8, gx);                      // ~8 CTAs per SM in total
    const int64_t max_gy = ceil_div(rows, 64);               // at least 64 rows per block
    if (gy > max_gy) gy = max_gy;
    if (gy < 1) gy = 1;
    if (gy > 65535) gy = 65535;
    const int64_t rpb = ceil_div(rows, gy);
    colsum_kernel<<<dim3((unsigned)gx, (unsigned)ceil_div(rows, rpb)), 256, 0, st>>>(src, rows, cols, rpb, out);
    UOCR_LAUNCHED("colsum");
    return UOCR_OK;
}

// dst (rows, cols_pad) = src (rows, cols) with zeros in the pad columns: operands whose row pitch is not a multiple of
// 16 bytes (Char dense_3: n_out = 162) cannot be fetched by TMA as they are
__global__ void __launch_bounds__(256) pad_cols_kernel(const float* __restrict__ src, float* __restrict__ dst, int64_t rows,
                                                       int cols, int cols_pad) {
    const int64_t total = rows * cols_pad;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
        const int64_t r = i / cols_pad;
        const int c = (int)(i - r * cols_pad);
        dst[i] = c < cols ? src[r * cols + c] : 0.f;
    }
}

static int pad_cols_async(const float* src, float* dst, int64_t rows, int cols, int cols_pad, cudaStream_t st) {
    const int64_t blocks = ceil_div(rows * cols_pad, 256 * 4);
    pad_cols_kernel<<<(unsigned)(blocks < 148 * 8 ? (blocks > 0 ? blocks : 1) : 148 * 8), 256, 0, st>>>(src, dst, rows, cols, cols_pad);
    UOCR_LAUNCHED("pad_cols");
    return UOCR_OK;
}

int fc_bwd_fast(int math_mode, const float* x, const float* w, const float* dy, float* dx, float* dw,
                int64_t batch, int64_t n_in, int64_t n_out, int accumulate, cudaStream_t st) {
    if (math_mode != UOCR_MATH_TF32) return UOCR_ERR_UNSUPPORTED;
    if (n_in % 4 || batch < 128 || n_out < 32 || n_in < 32 || !encode_tiled())
        return UOCR_ERR_UNSUPPORTED;
    if (n_out % 4) {
        // Char dense_3 (n_out = 162): dy and W padded to a 16-byte row pitch in scratch (zero columns contribute
        // nothing), then the same two tensor-core GEMMs; was 0.099 ms on the FP32 SGEMM path
        if (n_out > 0x7fffffff - 4) return UOCR_ERR_UNSUPPORTED;
        const int n_pad = (int)((n_out + 3) & ~(int64_t)3);
        Scratch dyp(st), wp(st);
        int rc = dyp.alloc(sizeof(float) * (size_t)batch * n_pad);
        if (rc) return rc;
        rc = pad_cols_async(dy, (float*)dyp.ptr, batch, (int)n_out, n_pad, st);
        if (rc) return rc;
        if (dx) {
            rc = wp.alloc(sizeof(float) * (size_t)n_in * n_pad);
            if (rc) return rc;
            rc = pad_cols_async(w, (float*)wp.ptr, n_in, (int)n_out, n_pad, st);
            if (rc) return rc;
            rc = tc_gemm_tn((const float*)dyp.ptr, n_pad, (const float*)wp.ptr, n_pad, dx, n_in, batch, n_in, n_pad, nullptr,
                            UOCR_ACT_NONE, 0.f, 0, st);
            if (rc) return rc;
        }
        if (!accumulate) {
            cudaError_t e = cudaMemsetAsync(dw, 0, sizeof(float) * (n_in + 1) * n_out, st);
            if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
        }
        rc = tc_gemm_mn_atomic(x, n_in, (const float*)dyp.ptr, n_pad, dw, n_out, n_in, n_out, batch, st);
        if (rc) return rc;
        return colsum_async(dy, batch, (int)n_out, dw + n_in * n_out, 1, st);
    }
    // dx = dy . W[:-1]^T : A = dy (batch, n_out) K-major; B^T = W[:-1] (n_in, n_out) is already K-major
    if (dx) {
        int rc = tc_gemm_tn(dy, n_out, w, n_out, dx, n_in, batch, n_in, n_out, nullptr, UOCR_ACT_NONE, 0.f, 0, st);
        if (rc) return rc;
    }
    // dW[:-1] += x^T . dy : both operands are batch-major -> MN-major tensor-core GEMM, split over the batch
    if (!accumulate) {
        cudaError_t e = cudaMemsetAsync(dw, 0, sizeof(float) * (n_in + 1) * n_out, st);
        if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
    }
    int rc = tc_gemm_mn_atomic(x, n_in, dy, n_out, dw, n_out, n_in, n_out, batch, st);
    if (rc) return rc;
    // dW[-1] += column sums of dy (the bias row)
    return colsum_async(dy, batch, (int)n_out, dw + n_in * n_out, 1, st);
}

// ------------------------------------------------------------------ Convolutional2D forward
// implicit GEMM: M = N*Ho*Wo pixels (tiles of 128 consecutive ox), N = Cout, K = kh*kw*Cin
static int conv_fwd_tc_slab(const ConvGeom& g, const float* x, const float* wt, const float* b, float* y, int act,
                            float alpha, cudaStream_t st);

int conv_fwd_tc(const ConvGeom& g, const float* x, const float* w, const float* w_kmajor, const float* b, float* y,
                int act, float alpha, cudaStream_t st) {
    if (g.cin % TC_BK || g.sw != 1 || g.padding_value != 0.f || g.ups != 1) return UOCR_ERR_UNSUPPORTED;
    if (g.cout % 16 || g.cout > 256 || g.cout < 16) return UOCR_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) & 15) || !encode_tiled()) return UOCR_ERR_UNSUPPORTED;
    const int K = g.kh * g.kw * g.cin;
    Scratch wt(st);
    int rc;
    if (!w_kmajor) {
        rc = wt.alloc(sizeof(float) * (size_t)K * g.cout);
        if (rc) return rc;
        rc = transpose_async(w, (float*)wt.ptr, K, g.cout, g.cout, K, st);       // (K, Cout) -> (Cout, K)
        if (rc) return rc;
        w_kmajor = (const float*)wt.ptr;
    }
    rc = conv_fwd_tc_slab(g, x, w_kmajor, b, y, act, alpha, st);
    if (rc != UOCR_ERR_UNSUPPORTED) return rc;
    TcParams p{};
    p.C = y; p.ldc = g.cout; p.M = (int64_t)g.n * g.ho * g.wo; p.N = g.cout;
    p.cblocks = g.cin / TC_BK;
    p.num_kb = g.kh * g.kw * p.cblocks;
    p.nt = g.cout;
    p.bias = g.bias ? b : nullptr; p.act = act; p.alpha = alpha; p.accumulate = 0;
    p.ho = g.ho; p.wo = g.wo; p.sh = g.sh; p.ph = g.ph; p.pw = g.pw; p.kw = g.kw;
    p.xtiles = (g.wo + TC_BM - 1) / TC_BM;
    CUtensorMap ma, mb;
    const uint64_t da[4] = {(uint64_t)g.cin, (uint64_t)g.w, (uint64_t)g.h, (uint64_t)g.n};
    const uint64_t sa[3] = {(uint64_t)g.cin * 4, (uint64_t)g.w * g.cin * 4, (uint64_t)g.h * g.w * g.cin * 4};
    const uint32_t ba[4] = {TC_BK, TC_BM, 1, 1};
    rc = make_tmap(&ma, x, 4, da, sa, ba);
    if (rc) return rc;
    const uint64_t db[2] = {(uint64_t)K, (uint64_t)g.cout}, sb[1] = {(uint64_t)K * 4};
    const uint32_t bb[2] = {TC_BK, (uint32_t)g.cout};
    rc = make_tmap(&mb, w_kmajor, 2, db, sb, bb);
    if (rc) return rc;
    const int64_t tiles = (int64_t)g.n * g.ho * p.xtiles;
    if (tiles > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    dim3 grid((unsigned)tiles, 1);
    return launch_tc<TC_CONV_FWD>(ma, mb, p, grid, st);
}

// ------------------------------------------------------------------------------------------
// Convolutional2D forward, slab variant (Char conv_2 / conv_3: 5x3, 64 -> 64, stride (2, 1)).
// ncu on the one-tile-per-CTA kernel above: every (ky, kx, channel block) step re-fetches a 16 KB A tile and an
// 8 KB B tile from L2 -- 720 KB per 128-pixel tile, 460 MB through L2 for a 59 MB input, i.e. L2 -> SM bandwidth
// bound at 20 % of the tensor peak.  Here a CTA owns one 128-pixel x-block of one output row, and a pipeline stage
// holds, for one (ky, channel block),
//   * an input-row SLAB of 128 + kw - 1 pixels x 32 channels: the kw horizontal taps are the SAME slab read from a
//     start address shifted by kx pixel rows (128 B each; the 128-byte swizzle is a function of the absolute
//     shared-memory address, so a start address that is not 1024-byte aligned needs nothing else -- setting the
//     descriptor's base-offset field to the row phase gives wrong results, tested), so A is fetched once per kernel
//     ROW instead of once per tap, and
//   * the kw weight chunks of that kernel row.
// Per 128-pixel tile that is 286 KB instead of 720 KB through L2.
// ------------------------------------------------------------------------------------------
struct SlabParams {
    float* y; const float* bias;
    int n_img, ho, wo, cout, nt;
    int kh, kw, sh, ph, pw, cblocks;
    int stages;
    uint32_t slab_bytes, slab_box_bytes, b_bytes;
    int act; float alpha;
};

__global__ void __launch_bounds__(TC_THREADS, 1) tc_conv_slab_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                     const __grid_constant__ CUtensorMap map_b,
                                                                     const SlabParams p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const uint32_t stage_bytes = p.slab_bytes + (uint32_t)p.kw * p.b_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + p.stages;
    uint64_t* tmem_full = bars + 2 * p.stages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * p.stages + 1);
    float* s_bias = reinterpret_cast<float*>(bars + 2 * p.stages + 2);      // nt floats (zeros without a bias)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < p.nt; i += TC_THREADS) s_bias[i] = (p.bias && i < p.cout) ? __ldg(p.bias + i) : 0.f;
    const int cx = blockIdx.x * TC_BM, oy = blockIdx.y, cn = blockIdx.z;
    const int num_it = p.kh * p.cblocks;
    uint32_t tmem_cols = 32;
    while ((int)tmem_cols < p.nt) tmem_cols <<= 1;

    if (threadIdx.x == 0) {
        for (int s = 0; s < p.stages; ++s) {
            mbar_init(smem_u32(&full[s]), 1);
            mbar_init(smem_u32(&empty[s]), 1);
        }
        mbar_init(smem_u32(tmem_full), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            for (int it = 0; it < num_it; ++it) {
                const int s = it % p.stages;
                mbar_wait(smem_u32(&empty[s]), ((it / p.stages) & 1) ^ 1);
                const int ky = it / p.cblocks, cb = it - ky * p.cblocks;
                const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
                const uint32_t sb = sa + p.slab_bytes;
                const uint32_t bar = smem_u32(&full[s]);
                mbar_arrive_expect_tx(bar, p.slab_box_bytes + (uint32_t)p.kw * p.b_bytes);
                tma_load_4d(sa, &map_a, bar, cb * TC_BK, cx - p.pw, oy * p.sh + ky - p.ph, cn);
                for (int kx = 0; kx < p.kw; ++kx) {
                    const int k0 = ((ky * p.kw + kx) * p.cblocks + cb) * TC_BK;
                    tma_load_2d(sb + (uint32_t)kx * p.b_bytes, &map_b, bar, k0, 0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.nt >> 3) << 17) |
                                   ((uint32_t)(TC_BM >> 4) << 24);
            for (int it = 0; it < num_it; ++it) {
                const int s = it % p.stages;
                mbar_wait(smem_u32(&full[s]), (it / p.stages) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + (size_t)s * stage_bytes);
                const uint32_t sb = sa + p.slab_bytes;
                for (int kx = 0; kx < p.kw; ++kx) {
                    // the tap's A operand = the slab from pixel row kx on
                    const uint64_t da = make_kmajor_sw128_desc(sa + (uint32_t)kx * 128u);
                    const uint64_t db = make_kmajor_sw128_desc(sb + (uint32_t)kx * p.b_bytes);
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k)
                        tc_mma_tf32(tmem_base, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc,
                                    (it > 0 || kx > 0 || k > 0) ? 1u : 0u);
                }
                tc_commit(smem_u32(&empty[s]));
            }
            tc_commit(smem_u32(tmem_full));
        }
    } else {
        const int q = warp & 3;
        mbar_wait(smem_u32(tmem_full), 0);
        tc_fence_after();
        const int ox = cx + q * 32 + lane;
        float* dst = p.y + (((int64_t)cn * p.ho + oy) * p.wo + ox) * p.cout;
        for (int c0 = 0; c0 < p.nt; c0 += 32) {
            float v[32];
            tc_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
            if (ox >= p.wo) continue;
            const float4* bs = reinterpret_cast<const float4*>(s_bias + c0);
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                if (c0 + j < p.cout) {                                   // cout % 16 == 0
                    const float4 b4 = bs[j >> 2];
                    float4 o;
                    o.x = apply_act_fast(v[j] + b4.x, p.act, p.alpha);
                    o.y = apply_act_fast(v[j + 1] + b4.y, p.act, p.alpha);
                    o.z = apply_act_fast(v[j + 2] + b4.z, p.act, p.alpha);
                    o.w = apply_act_fast(v[j + 3] + b4.w, p.act, p.alpha);
                    *reinterpret_cast<float4*>(dst + c0 + j) = o;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
    }
}

static int conv_fwd_tc_slab(const ConvGeom& g, const float* x, const float* wt /* (Cout, K) */, const float* b, float* y,
                            int act, float alpha, cudaStream_t st) {
    if (g.kw > 8 || g.cout > 128 || (reinterpret_cast<uintptr_t>(y) & 15)) return UOCR_ERR_UNSUPPORTED;
    if (g.n > 65535 || g.ho > 65535) return UOCR_ERR_UNSUPPORTED;
    SlabParams p{};
    p.y = y; p.bias = g.bias ? b : nullptr;
    p.n_img = g.n; p.ho = g.ho; p.wo = g.wo; p.cout = g.cout; p.nt = g.cout;
    p.kh = g.kh; p.kw = g.kw; p.sh = g.sh; p.ph = g.ph; p.pw = g.pw; p.cblocks = g.cin / TC_BK;
    p.act = act; p.alpha = alpha;
    const int xtiles = (g.wo + TC_BM - 1) / TC_BM;
    // Measured on Char conv_2 (64 tiles of 5 x 256 pixels): 2 stages (84 KB: two CTAs per SM, so one CTA's prologue /
    // epilogue overlaps the other's main loop) 0.050 ms; 2 x-blocks per CTA sharing B with 3 stages (one CTA per SM)
    // 0.067 ms; the one-tile-per-CTA kernel 0.065 ms.
    const uint32_t box_rows = TC_BM + g.kw - 1;
    p.slab_box_bytes = box_rows * 128u;
    p.slab_bytes = (p.slab_box_bytes + 1023u) & ~1023u;
    p.b_bytes = (uint32_t)g.cout * 128u;                            // cout % 16 == 0 -> multiple of 2048: 1024-aligned
    const uint32_t stage_bytes = p.slab_bytes + (uint32_t)g.kw * p.b_bytes;
    p.stages = (int)((200u * 1024u) / stage_bytes);
    if (p.stages > 2) p.stages = 2;
    if (p.stages < 2 || (p.b_bytes & 1023u)) return UOCR_ERR_UNSUPPORTED;
    const size_t smem = (size_t)p.stages * stage_bytes + 1024 + (2 * p.stages + 2) * 8 + 4 * 128 + 64;
    const int K = g.kh * g.kw * g.cin;
    CUtensorMap ma, mb;
    const uint64_t da[4] = {(uint64_t)g.cin, (uint64_t)g.w, (uint64_t)g.h, (uint64_t)g.n};
    const uint64_t sa[3] = {(uint64_t)g.cin * 4, (uint64_t)g.w * g.cin * 4, (uint64_t)g.h * g.w * g.cin * 4};
    const uint32_t ba[4] = {TC_BK, box_rows, 1, 1};
    int rc = make_tmap(&ma, x, 4, da, sa, ba);
    if (rc) return rc;
    const uint64_t db[2] = {(uint64_t)K, (uint64_t)g.cout}, sb[1] = {(uint64_t)K * 4};
    const uint32_t bb[2] = {TC_BK, (uint32_t)g.cout};
    rc = make_tmap(&mb, wt, 2, db, sb, bb);
    if (rc) return rc;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(tc_conv_slab_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
        configured = true;
    }
    dim3 grid((unsigned)xtiles, (unsigned)g.ho, (unsigned)g.n);
    tc_conv_slab_kernel<<<grid, TC_THREADS, smem, st>>>(ma, mb, p);
    UOCR_LAUNCHED("tc_conv_slab_tf32");
    return UOCR_OK;
}

// ------------------------------------------------------------------ Convolutional2D dgrad
// implicit GEMM over the INPUT pixels: M = 128 consecutive ix of one input row, N = Cin,
// K = (kernel rows that hit this row's parity) x kw x Cout.  A tiles are boxes of dy, B tiles are
// the (Cin x 32) slabs of w[ky, kx] -- the weight tensor is already K-major for this product.
int conv_dgrad_tc(const ConvGeom& g, const float* dy, const float* w, float* dx, cudaStream_t st) {
    if (g.cout % TC_BK || g.sw != 1 || g.ups != 1 || g.kh > 31) return UOCR_ERR_UNSUPPORTED;
    if (g.cin % 16 || g.cin > 256 || g.cin < 16) return UOCR_ERR_UNSUPPORTED;
    if (((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(w)) & 15) || !encode_tiled())
        return UOCR_ERR_UNSUPPORTED;
    TcParams p{};
    p.C = dx; p.ldc = g.cin; p.M = (int64_t)g.n * g.h * g.w; p.N = g.cin;
    p.nt = g.cin; p.act = UOCR_ACT_NONE;
    p.ho = g.ho; p.wo = g.wo; p.sh = g.sh; p.ph = g.ph; p.pw = g.pw; p.kh = g.kh; p.kw = g.kw;
    p.cblocks = g.cout / TC_BK; p.cin = g.cin; p.h_in = g.h; p.w_in = g.w;
    p.xtiles = (g.w + TC_BM - 1) / TC_BM;
    CUtensorMap ma, mb;
    const uint64_t da[4] = {(uint64_t)g.cout, (uint64_t)g.wo, (uint64_t)g.ho, (uint64_t)g.n};
    const uint64_t sa[3] = {(uint64_t)g.cout * 4, (uint64_t)g.wo * g.cout * 4, (uint64_t)g.ho * g.wo * g.cout * 4};
    const uint32_t ba[4] = {TC_BK, TC_BM, 1, 1};
    int rc = make_tmap(&ma, dy, 4, da, sa, ba);
    if (rc) return rc;
    const uint64_t db[2] = {(uint64_t)g.cout, (uint64_t)g.kh * g.kw * g.cin}, sb[1] = {(uint64_t)g.cout * 4};
    const uint32_t bb[2] = {TC_BK, (uint32_t)g.cin};
    rc = make_tmap(&mb, w, 2, db, sb, bb);
    if (rc) return rc;
    const int64_t tiles = (int64_t)g.n * g.h * p.xtiles;
    if (tiles > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    return launch_tc<TC_CONV_DGRAD>(ma, mb, p, dim3((unsigned)tiles, 1), st);
}

// ------------------------------------------------------------------ Convolutional2D wgrad
// dW[(tap, ci), co] += sum over pixels x[n, oy*sh+ky-ph, ox+kx-pw, ci] * dy[n, oy, ox, co]:
// the contraction runs over pixels, which are the ROWS of both NHWC tensors -> MN-major operands.
// One CTA owns 128 / Cin kernel taps (M = 128 rows of dW) and a slice of the (n, oy) rows; per
// 32-pixel K block it fetches the shifted x boxes of its taps and the dy box, partial tiles are
// added with atomicAdd.  db is a column sum of dy.  Requires zero padding (TMA zero fill).
int conv_wgrad_tc(const ConvGeom& g, const float* x, const float* dy, float* dw, float* db, int accumulate,
                  cudaStream_t st) {
    if (g.sw != 1 || g.ups != 1 || g.padding_value != 0.f) return UOCR_ERR_UNSUPPORTED;
    if (!(g.cin == 32 || g.cin == 64 || g.cin == 128) || g.cout % 32 || g.cout > 256) return UOCR_ERR_UNSUPPORTED;
    if (((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy)) & 15) || !encode_tiled())
        return UOCR_ERR_UNSUPPORTED;
    const int64_t kc = (int64_t)g.kh * g.kw * g.cin * g.cout;
    if (!accumulate) {
        cudaError_t e = cudaMemsetAsync(dw, 0, sizeof(float) * kc, st);
        if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
    }
    TcParams p{};
    p.C = dw; p.ldc = g.cout; p.N = g.cout; p.M = (int64_t)g.kh * g.kw * g.cin;
    p.nt = g.cout; p.act = UOCR_ACT_NONE; p.atomic = 1;
    p.ho = g.ho; p.wo = g.wo; p.sh = g.sh; p.ph = g.ph; p.pw = g.pw; p.kh = g.kh; p.kw = g.kw; p.cin = g.cin;
    p.ntaps = g.kh * g.kw; p.taps_per_cta = TC_BM / g.cin;
    p.kbx = (g.wo + TC_BK - 1) / TC_BK;
    p.rows_total = g.n * g.ho;
    const int tap_groups = (p.ntaps + p.taps_per_cta - 1) / p.taps_per_cta;
    int64_t splits = (148 * 2 + tap_groups - 1) / tap_groups;
    if (splits > p.rows_total) splits = p.rows_total;
    if (splits < 1) splits = 1;
    p.rows_per_split = (int)ceil_div(p.rows_total, splits);
    splits = ceil_div(p.rows_total, p.rows_per_split);
    if (splits > 65535) return UOCR_ERR_UNSUPPORTED;
    CUtensorMap ma, mb;
    const uint32_t box[4] = {32, TC_BK, 1, 1};
    const uint64_t da[4] = {(uint64_t)g.cin, (uint64_t)g.w, (uint64_t)g.h, (uint64_t)g.n};
    const uint64_t sa[3] = {(uint64_t)g.cin * 4, (uint64_t)g.w * g.cin * 4, (uint64_t)g.h * g.w * g.cin * 4};
    int rc = make_tmap(&ma, x, 4, da, sa, box, true);
    if (rc) return rc;
    const uint64_t db_[4] = {(uint64_t)g.cout, (uint64_t)g.wo, (uint64_t)g.ho, (uint64_t)g.n};
    const uint64_t sb[3] = {(uint64_t)g.cout * 4, (uint64_t)g.wo * g.cout * 4, (uint64_t)g.ho * g.wo * g.cout * 4};
    rc = make_tmap(&mb, dy, 4, db_, sb, box, true);
    if (rc) return rc;
    rc = launch_tc<TC_CONV_WGRAD>(ma, mb, p, dim3((unsigned)tap_groups, 1, (unsigned)splits), st);
    if (rc) return rc;
    if (g.bias) return colsum_async(dy, (int64_t)g.n * g.ho * g.wo, g.cout, db, accumulate, st);
    if (!accumulate) {
        cudaError_t e = cudaMemsetAsync(db, 0, sizeof(float) * g.cout, st);
        if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
    }
    return UOCR_OK;
}

// ------------------------------------------------------------------------------------------
// Two FullyConnected layers in one kernel (inference): y = (act1(x . W1 + b1)) . W2 + b2 for a hidden width of 128
// (Char dense_2 + LeakyRelu + dense_3, my_model/model.py:251-304; nn/layers/layers.py:335-347).  Per 128-row tile:
//   GEMM 1  the usual TMA -> 128B-swizzled ring -> tcgen05.mma pipeline over K1, accumulator 1 in TMEM columns 0..127
//   middle  the four epilogue warps read accumulator 1 (lane = row), add b1, apply act1, round to TF32 and write the
//           128 x 128 hidden tile INTO SHARED MEMORY IN THE OPERAND LAYOUT the next MMA reads (K-major rows of 128
//           bytes, 16-byte chunks XOR-swizzled with the row like a SWIZZLE_128B TMA box): it never goes to HBM
//   GEMM 2  the producer warp simply keeps going: W2's four K blocks travel through the same ring (one per stage);
//           A = the hidden tile, accumulator 2 in TMEM columns 128..
//   last    accumulator 2 + b2 is staged in the (now idle) ring as packed rows of n2 floats and leaves as one linear,
//           16-byte-coalesced copy -- a tile's rows are contiguous in y even when n2 = 162 is not a multiple of 4
// Saves the hidden matrix's round trip (2 x 8.4 MB at batch 16384), one launch, and dense_3's operand loads.
// ------------------------------------------------------------------------------------------
constexpr int FC2_HID = 128;              // hidden width = N of GEMM 1 = K of GEMM 2
constexpr int FC2_STAGES = 4;
constexpr int FC2_STAGE_BYTES = 2 * TC_BM * TC_BK * 4;                    // A 16 KB + B 16 KB; a W2 block uses <= 32 KB of it

struct Fc2Params {
    float* y; int64_t M; int n2, nt2, num_kb1;
    const float* b1; const float* b2;
    int act1; float alpha1;
};

__global__ void __launch_bounds__(TC_THREADS, 1) fc_chain2_kernel(const __grid_constant__ CUtensorMap map_x,
                                                                  const __grid_constant__ CUtensorMap map_w1,
                                                                  const __grid_constant__ CUtensorMap map_w2,
                                                                  const Fc2Params p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* s_hid = smem + FC2_STAGES * FC2_STAGE_BYTES;                  // 4 K blocks x 16 KB, 1024-aligned
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_hid + 4 * TC_BM * TC_BK * 4);
    uint64_t* full = bars;
    uint64_t* empty = bars + FC2_STAGES;
    uint64_t* acc1_full = bars + 2 * FC2_STAGES;
    uint64_t* hid_full = acc1_full + 1;
    uint64_t* acc2_full = acc1_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc1_full + 3);
    float* s_bias = reinterpret_cast<float*>(tmem_slot + 2);               // b1[128], b2[nt2]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t m0 = (int64_t)blockIdx.x * TC_BM;
    const int m_rows = (int)min((int64_t)TC_BM, p.M - m0);
    const int total_kb = p.num_kb1 + FC2_HID / TC_BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < FC2_STAGES; ++s) { mbar_init(smem_u32(&full[s]), 1); mbar_init(smem_u32(&empty[s]), 1); }
        mbar_init(smem_u32(acc1_full), 1);
        mbar_init(smem_u32(hid_full), 128);
        mbar_init(smem_u32(acc2_full), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = threadIdx.x; i < FC2_HID + p.nt2; i += TC_THREADS)
        s_bias[i] = i < FC2_HID ? __ldg(p.b1 + i) : (i - FC2_HID < p.n2 ? __ldg(p.b2 + i - FC2_HID) : 0.f);
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===================== TMA producer: K1 / 32 blocks of (x, W1), then the 4 blocks of W2 =====================
        if (lane == 0) {
            for (int kb = 0; kb < total_kb; ++kb) {
                const int s = kb % FC2_STAGES;
                mbar_wait(smem_u32(&empty[s]), ((kb / FC2_STAGES) & 1) ^ 1);
                const uint32_t sa = smem_u32(smem + (size_t)s * FC2_STAGE_BYTES), bar = smem_u32(&full[s]);
                if (kb < p.num_kb1) {
                    mbar_arrive_expect_tx(bar, (uint32_t)FC2_STAGE_BYTES);
                    tma_load_2d(sa, &map_x, bar, kb * TC_BK, (int)m0);
                    tma_load_2d(sa + TC_BM * TC_BK * 4, &map_w1, bar, kb * TC_BK, 0);
                } else {
                    mbar_arrive_expect_tx(bar, (uint32_t)p.nt2 * TC_BK * 4);
                    tma_load_2d(sa, &map_w2, bar, (kb - p.num_kb1) * TC_BK, 0);
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            const uint32_t idesc1 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(FC2_HID >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            const uint32_t idesc2 = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.nt2 >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            for (int kb = 0; kb < total_kb; ++kb) {
                const int s = kb % FC2_STAGES;
                if (kb == p.num_kb1) {                         // GEMM 1 is complete; GEMM 2 needs the hidden tile
                    tc_commit(smem_u32(acc1_full));
                    mbar_wait(smem_u32(hid_full), 0);
                }
                mbar_wait(smem_u32(&full[s]), (kb / FC2_STAGES) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + (size_t)s * FC2_STAGE_BYTES);
                if (kb < p.num_kb1) {
                    const uint64_t da = make_kmajor_sw128_desc(sa), db = make_kmajor_sw128_desc(sa + TC_BM * TC_BK * 4);
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k)
                        tc_mma_tf32(tmem_base, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc1, (kb > 0 || k > 0) ? 1u : 0u);
                } else {
                    const int j = kb - p.num_kb1;
                    const uint64_t da = make_kmajor_sw128_desc(smem_u32(s_hid + (size_t)j * TC_BM * TC_BK * 4));
                    const uint64_t db = make_kmajor_sw128_desc(sa);
#pragma unroll
                    for (int k = 0; k < TC_BK / 8; ++k)
                        tc_mma_tf32(tmem_base + FC2_HID, da + (uint64_t)(k * 2), db + (uint64_t)(k * 2), idesc2, (j > 0 || k > 0) ? 1u : 0u);
                }
                tc_commit(smem_u32(&empty[s]));
            }
            tc_commit(smem_u32(acc2_full));
        }
    } else {
        // ===================== epilogue warps (lane quarter q, row r of the tile) =====================
        const int q = warp & 3, r = q * 32 + lane;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        mbar_wait(smem_u32(acc1_full), 0);
        tc_fence_after();
        for (int j = 0; j < FC2_HID / TC_BK; ++j) {
            float v[32];
            tc_ld_32x32(lane_base + (uint32_t)(j * TC_BK), v);
            uint8_t* row = s_hid + (size_t)j * TC_BM * TC_BK * 4 + (size_t)r * 128;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint32_t o[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float t = apply_act_fast(v[4 * c + e] + s_bias[j * TC_BK + 4 * c + e], p.act1, p.alpha1);
                    o[e] = (__float_as_uint(t) + 0x1000u) & 0xffffe000u;      // TF32, round to nearest
                }
                *reinterpret_cast<uint4*>(row + ((c ^ (r & 7)) << 4)) = make_uint4(o[0], o[1], o[2], o[3]);
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");        // generic writes -> the MMA's async-proxy reads
        mbar_arrive(smem_u32(hid_full));
        // ---- accumulator 2 -> packed rows in the idle ring -> one linear copy
        mbar_wait(smem_u32(acc2_full), 0);
        tc_fence_after();
        float* stage = reinterpret_cast<float*>(smem);
        for (int c0 = 0; c0 < p.nt2; c0 += 32) {
            float v[32];
            tc_ld_32x32(lane_base + (uint32_t)(FC2_HID + c0), v);
#pragma unroll
            for (int e = 0; e < 32; ++e)
                if (c0 + e < p.n2) stage[r * p.n2 + c0 + e] = v[e] + s_bias[FC2_HID + c0 + e];
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        const int t = threadIdx.x - 64;                                      // 0..127
        const int64_t count = (int64_t)m_rows * p.n2;
        float* dst = p.y + m0 * p.n2;
        if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
            const int64_t quads = count >> 2;
            for (int64_t i = t; i < quads; i += 128)
                reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(stage)[i];
            for (int64_t i = (quads << 2) + t; i < count; i += 128) dst[i] = stage[i];
        } else {
            for (int64_t i = t; i < count; i += 128) dst[i] = stage[i];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// y (batch, n2) = act1([x, 1] . W1) . W2[:-1] + W2[-1];  W1: (k1 + 1, 128), W2: (129, n2); w1t / w2t: K-major copies
int fc_chain2_fwd_fast(int math_mode, const float* x, const float* w1, const float* w1t, const float* w2, const float* w2t,
                       float* y, int64_t batch, int64_t k1, int64_t n1, int64_t n2, int act1, float alpha1, cudaStream_t st) {
    if (math_mode != UOCR_MATH_TF32 || !encode_tiled()) return UOCR_ERR_UNSUPPORTED;
    if (n1 != FC2_HID || k1 % TC_BK || k1 < TC_BK || n2 < 16 || n2 > 256 || batch < 128 || batch > 0x7fffffff) return UOCR_ERR_UNSUPPORTED;
    if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) return UOCR_ERR_UNSUPPORTED;
    Scratch t1(st), t2(st);
    if (!w1t) {
        int rc = t1.alloc(sizeof(float) * n1 * k1);
        if (rc) return rc;
        rc = transpose_async(w1, (float*)t1.ptr, (int)k1, (int)n1, n1, k1, st);
        if (rc) return rc;
        w1t = (const float*)t1.ptr;
    }
    if (!w2t) {
        int rc = t2.alloc(sizeof(float) * n2 * n1);
        if (rc) return rc;
        rc = transpose_async(w2, (float*)t2.ptr, (int)n1, (int)n2, n2, n1, st);
        if (rc) return rc;
        w2t = (const float*)t2.ptr;
    }
    Fc2Params p{};
    p.y = y; p.M = batch; p.n2 = (int)n2; p.nt2 = (int)(((n2 + 15) / 16) * 16); p.num_kb1 = (int)(k1 / TC_BK);
    p.b1 = w1 + k1 * n1; p.b2 = w2 + n1 * n2; p.act1 = act1; p.alpha1 = alpha1;
    CUtensorMap mx, m1, m2;
    const uint64_t dx[2] = {(uint64_t)k1, (uint64_t)batch}, sx[1] = {(uint64_t)k1 * 4};
    const uint32_t bx[2] = {TC_BK, TC_BM};
    int rc = make_tmap(&mx, x, 2, dx, sx, bx);
    if (rc) return rc;
    const uint64_t d1[2] = {(uint64_t)k1, (uint64_t)n1}, s1[1] = {(uint64_t)k1 * 4};
    const uint32_t b1[2] = {TC_BK, (uint32_t)FC2_HID};
    rc = make_tmap(&m1, w1t, 2, d1, s1, b1);
    if (rc) return rc;
    const uint64_t d2[2] = {(uint64_t)n1, (uint64_t)n2}, s2[1] = {(uint64_t)n1 * 4};
    const uint32_t b2[2] = {TC_BK, (uint32_t)p.nt2};
    rc = make_tmap(&m2, w2t, 2, d2, s2, b2);
    if (rc) return rc;
    const size_t smem = 1024 + (size_t)FC2_STAGES * FC2_STAGE_BYTES + 4 * TC_BM * TC_BK * 4 + (2 * FC2_STAGES + 3) * 8 + 16 +
                        (FC2_HID + p.nt2) * sizeof(float) + 64;
    static bool configured = false;
    if (!configured) {
        cudaError_t e = cudaFuncSetAttribute(fc_chain2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return UOCR_ERR_CUDA; }
        configured = true;
    }
    fc_chain2_kernel<<<(unsigned)ceil_div(batch, TC_BM), TC_THREADS, smem, st>>>(mx, m1, m2, p);
    UOCR_LAUNCHED("fc_chain2");
    return UOCR_OK;
}
}  // namespace uocr

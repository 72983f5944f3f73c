// Losses (nn/losses.py), regularisers (nn/regularizations.py) and optimiser updates
// (nn/optimizers.py) as fused streaming / reduction kernels.
//
// The reference evaluates each of these as a chain of whole-array CuPy expressions with
// temporaries (Adam: ~9 kernels per parameter, optimizers.py:56-61; Dice: 3 reductions + 4
// elementwise passes, losses.py:12-25) and forces a device sync per loss through float().
// Here: Dice/Jaccard = one reduction pass + one gradient pass; Adam (+ optional folded L2 and
// gradient scaling) = one pass over (w, g, v, a); the loss value stays on the device.
#include "common.cuh"

namespace uocr {

constexpr double kEpsLoss = 1e-8;     // losses.py:19,36

// ---------------------------------------------------------------- Dice / Jaccard
// pass 1: per (n, c) sums of p*g, p, g over H*W.  grid = (chunks, N); sums[3][N*C] (double).
__global__ void __launch_bounds__(kThreads) seg_sums_kernel(const float* __restrict__ pred,
                                                            const float* __restrict__ gt,
                                                            double* __restrict__ sums, int64_t hw,
                                                            int c, int64_t nc) {
    __shared__ double red[8];
    const int n = blockIdx.y;
    const float* p = pred + (int64_t)n * hw * c;
    const float* g = gt + (int64_t)n * hw * c;
    const int64_t per = (hw + gridDim.x - 1) / gridDim.x;
    const int64_t lo = (int64_t)blockIdx.x * per, hi = min(hw, lo + per);
    for (int ch = 0; ch < c; ++ch) {
        float spg = 0.f, sp = 0.f, sg = 0.f;
        if (c == 1) {
            // contiguous: 128-bit loads over the 16-byte aligned body
            const int64_t a0 = min(hi, (lo + 3) & ~(int64_t)3);
            const bool al = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g)) & 15) == 0;
            if (al) {
                for (int64_t i = lo + threadIdx.x; i < a0; i += kThreads) {
                    const float a = p[i], b = g[i];
                    spg = fmaf(a, b, spg); sp += a; sg += b;
                }
                const int64_t v0 = a0 / 4, v1 = hi / 4;
                const float4* p4 = reinterpret_cast<const float4*>(p);
                const float4* g4 = reinterpret_cast<const float4*>(g);
                for (int64_t i = v0 + threadIdx.x; i < v1; i += kThreads) {
                    const float4 a = p4[i], b = g4[i];
                    spg = fmaf(a.x, b.x, spg); spg = fmaf(a.y, b.y, spg);
                    spg = fmaf(a.z, b.z, spg); spg = fmaf(a.w, b.w, spg);
                    sp += (a.x + a.y) + (a.z + a.w);
                    sg += (b.x + b.y) + (b.z + b.w);
                }
                for (int64_t i = max(a0, v1 * 4) + threadIdx.x; i < hi; i += kThreads) {
                    const float a = p[i], b = g[i];
                    spg = fmaf(a, b, spg); sp += a; sg += b;
                }
            } else {
                for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) {
                    const float a = p[i], b = g[i];
                    spg = fmaf(a, b, spg); sp += a; sg += b;
                }
            }
        } else {
            for (int64_t i = lo + threadIdx.x; i < hi; i += kThreads) {
                const float a = p[i * c + ch], b = g[i * c + ch];
                spg = fmaf(a, b, spg); sp += a; sg += b;
            }
        }
        const double r0 = block_sum((double)spg, red);
        const double r1 = block_sum((double)sp, red);
        const double r2 = block_sum((double)sg, red);
        if (threadIdx.x == 0) {
            atomicAdd(&sums[0 * nc + n * c + ch], r0);
            atomicAdd(&sums[1 * nc + n * c + ch], r1);
            atomicAdd(&sums[2 * nc + n * c + ch], r2);
        }
    }
}

// pass 1.5: one CTA: loss and the two per-(n,c) gradient coefficients  grad = a * gt + b
__global__ void __launch_bounds__(kThreads) seg_finalize_kernel(int kind, const double* __restrict__ sums,
                                                                float* __restrict__ coef, int64_t nc,
                                                                float* __restrict__ loss) {
    __shared__ double red[8];
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < nc; i += kThreads) {
        const double num = sums[i] + kEpsLoss;
        double den, a, b, l;
        if (kind == UOCR_SEG_DICE) {                      // losses.py:20-24
            den = sums[nc + i] + sums[2 * nc + i] + 2 * kEpsLoss;
            l = 1.0 - 2.0 * num / den;
            a = -2.0 / den;
            b = 2.0 * num / (den * den);
        } else {                                          // losses.py:37-41
            den = sums[nc + i] + sums[2 * nc + i] - num + 2 * kEpsLoss;
            l = 1.0 - num / den;
            a = -(den + num) / (den * den);
            b = num / (den * den);
        }
        coef[2 * i] = (float)a;
        coef[2 * i + 1] = (float)b;
        acc += l;
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) loss[0] = (float)acc;
}

// pass 1 of a ragged batch: the same sums over image n's h_n x w_n region of the (N, H, W, C) canvas only.
// grid = (chunks, N): the chunks split the region's rows, one warp per row; a row is w_n * c contiguous floats, read
// with 16-byte loads where the alignment allows (c == 1).
__global__ void __launch_bounds__(kThreads) seg_sums_ragged_kernel(const float* __restrict__ pred,
                                                                   const float* __restrict__ gt,
                                                                   const int32_t* __restrict__ ext,
                                                                   double* __restrict__ sums, int64_t h, int64_t w,
                                                                   int c, int64_t nc) {
    __shared__ double red[8];
    const int n = blockIdx.y;
    const int lane = threadIdx.x & 31;
    int64_t hn, wn;
    ragged_extent(ext, n, h, w, hn, wn);
    const int64_t per = (hn + gridDim.x - 1) / gridDim.x;
    const int64_t y0 = (int64_t)blockIdx.x * per, y1 = min(hn, y0 + per);
    const int64_t len = wn * c, stride = w * c;
    const bool al = ((reinterpret_cast<uintptr_t>(pred) ^ reinterpret_cast<uintptr_t>(gt)) & 15) == 0;
    for (int ch = 0; ch < c; ++ch) {
        float spg = 0.f, sp = 0.f, sg = 0.f;
        auto add = [&](float a, float b) { spg = fmaf(a, b, spg); sp += a; sg += b; };
        for (int64_t y = y0 + (threadIdx.x >> 5); y < y1; y += kThreads / 32) {
            const float* p = pred + ((int64_t)n * h + y) * stride;
            const float* g = gt + ((int64_t)n * h + y) * stride;
            if (c == 1) {
                // scalar head up to a 16-byte boundary of p (and g: same offset), float4 body, scalar tail
                const int64_t head = al ? min(len, (int64_t)((4 - ((reinterpret_cast<uintptr_t>(p) >> 2) & 3)) & 3))
                                        : len;
                for (int64_t j = lane; j < head; j += 32) add(p[j], g[j]);
                const int64_t quads = (len - head) >> 2;
                const float4* p4 = reinterpret_cast<const float4*>(p + head);
                const float4* g4 = reinterpret_cast<const float4*>(g + head);
                for (int64_t q = lane; q < quads; q += 32) {
                    const float4 a = p4[q], b = g4[q];
                    spg = fmaf(a.x, b.x, spg); spg = fmaf(a.y, b.y, spg);
                    spg = fmaf(a.z, b.z, spg); spg = fmaf(a.w, b.w, spg);
                    sp += (a.x + a.y) + (a.z + a.w);
                    sg += (b.x + b.y) + (b.z + b.w);
                }
                for (int64_t j = head + 4 * quads + lane; j < len; j += 32) add(p[j], g[j]);
            } else {
                for (int64_t x = lane; x < wn; x += 32) add(p[x * c + ch], g[x * c + ch]);
            }
        }
        const double r0 = block_sum((double)spg, red);
        const double r1 = block_sum((double)sp, red);
        const double r2 = block_sum((double)sg, red);
        if (threadIdx.x == 0) {
            atomicAdd(&sums[0 * nc + n * c + ch], r0);
            atomicAdd(&sums[1 * nc + n * c + ch], r1);
            atomicAdd(&sums[2 * nc + n * c + ch], r2);
        }
    }
}

// one gradient element: a * gt + b, with SIG times the Sigmoid derivative e / (e + 1)^2, e = exp(-x)
template <bool SIG>
__device__ __forceinline__ float seg_grad_value(float a, float b, float gv, float xv) {
    const float gr = fmaf(a, gv, b);
    if (!SIG) return gr;
    const float e = expf(-xv);                               // same expression as SigmoidBwd (elementwise.cu)
    const float d = e + 1.f;
    return gr * e / (d * d);
}

// pass 2: grad = a[n,c] * gt + b[n,c]  (SIG: times the Sigmoid derivative e / (e + 1)^2, e = exp(-x), of the
// pre-activation x the prediction came from -- loss gradient and Sigmoid backward in one pass).  grid = (chunks, N)
template <bool SIG>
__global__ void __launch_bounds__(kThreads) seg_grad_kernel(const float* __restrict__ gt,
                                                            const float* __restrict__ coef,
                                                            const float* __restrict__ xpre,
                                                            float* __restrict__ grad, int64_t hw, int c) {
    const int n = blockIdx.y;
    const int64_t len = hw * c;
    const float* g = gt + (int64_t)n * len;
    const float* xp = SIG ? xpre + (int64_t)n * len : nullptr;
    float* o = grad + (int64_t)n * len;
    const float* cf = coef + (int64_t)n * c * 2;
    auto one = [&](float a, float b, float gv, float xv) { return seg_grad_value<SIG>(a, b, gv, xv); };
    const bool al = ((reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(o) |
                      (SIG ? reinterpret_cast<uintptr_t>(xp) : 0)) & 15) == 0;
    if (c == 1 && al) {
        const float a = cf[0], b = cf[1];
        const int64_t n4 = len / 4;
        const float4* g4 = reinterpret_cast<const float4*>(g);
        const float4* x4 = reinterpret_cast<const float4*>(xp);
        float4* o4 = reinterpret_cast<float4*>(o);
        for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n4;
             i += (int64_t)gridDim.x * kThreads) {
            const float4 v = g4[i];
            const float4 xv = SIG ? x4[i] : make_float4(0.f, 0.f, 0.f, 0.f);
            o4[i] = make_float4(one(a, b, v.x, xv.x), one(a, b, v.y, xv.y), one(a, b, v.z, xv.z), one(a, b, v.w, xv.w));
        }
        for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * kThreads + threadIdx.x; i < len;
             i += (int64_t)gridDim.x * kThreads)
            o[i] = one(a, b, g[i], SIG ? xp[i] : 0.f);
    } else {
        for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < len;
             i += (int64_t)gridDim.x * kThreads) {
            const int ch = (int)(i % c);
            o[i] = one(cf[2 * ch], cf[2 * ch + 1], g[i], SIG ? xp[i] : 0.f);
        }
    }
}

// pass 2 of a ragged batch: one warp per canvas row writes the whole row -- the gradient over image i's w_i * c floats
// when the row is inside its extent, 0 everywhere else -- and reads gt / x_pre inside the extent only.  16-byte stores
// (and loads) where the alignment allows.
template <bool SIG>
__global__ void __launch_bounds__(kThreads) seg_grad_ragged_kernel(const float* __restrict__ gt,
                                                                   const float* __restrict__ coef,
                                                                   const float* __restrict__ xpre,
                                                                   float* __restrict__ grad,
                                                                   const int32_t* __restrict__ ext, int64_t n,
                                                                   int64_t h, int64_t w, int c) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
    const bool al = ((reinterpret_cast<uintptr_t>(grad) ^ reinterpret_cast<uintptr_t>(gt)) & 15) == 0 &&
                    (!SIG || ((reinterpret_cast<uintptr_t>(grad) ^ reinterpret_cast<uintptr_t>(xpre)) & 15) == 0);
    const int64_t end = w * c;
    for (int64_t row = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); row < n * h; row += warps) {
        const int64_t i = row / h, y = row - i * h;
        int64_t hi, wi;
        ragged_extent(ext, i, h, w, hi, wi);
        const int64_t len = (y < hi ? wi : 0) * c;
        const float* g = gt + row * end;
        const float* xp = SIG ? xpre + row * end : nullptr;
        float* o = grad + row * end;
        const float* cf = coef + i * c * 2;
        auto val = [&](int64_t j, float gv, float xv) {
            const int ch = c == 1 ? 0 : (int)(j % c);
            return seg_grad_value<SIG>(cf[2 * ch], cf[2 * ch + 1], gv, xv);
        };
        auto scalar = [&](int64_t j) { return j < len ? val(j, g[j], SIG ? xp[j] : 0.f) : 0.f; };
        const int64_t head = al ? min(end, (int64_t)((4 - ((reinterpret_cast<uintptr_t>(o) >> 2) & 3)) & 3)) : end;
        for (int64_t j = lane; j < head; j += 32) o[j] = scalar(j);
        const int64_t quads = (end - head) >> 2;
        for (int64_t q = lane; q < quads; q += 32) {
            const int64_t j = head + 4 * q;
            float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j + 4 <= len) {
                const float4 gv = *reinterpret_cast<const float4*>(g + j);
                const float4 xv = SIG ? *reinterpret_cast<const float4*>(xp + j) : make_float4(0.f, 0.f, 0.f, 0.f);
                r = make_float4(val(j, gv.x, xv.x), val(j + 1, gv.y, xv.y), val(j + 2, gv.z, xv.z),
                                val(j + 3, gv.w, xv.w));
            } else if (j < len) {
                r = make_float4(scalar(j), scalar(j + 1), scalar(j + 2), scalar(j + 3));
            }
            *reinterpret_cast<float4*>(o + j) = r;
        }
        for (int64_t j = head + 4 * quads + lane; j < end; j += 32) o[j] = scalar(j);
    }
}

// ---------------------------------------------------------------- softmax cross-entropy
// one warp per row.  log p is evaluated as (x - max) - log(sum) (more accurate in FP32 than
// log(e / s)); p underflows to exactly 0 in the reference's float64 when x - max < -745.13, and
// there log p = -inf, so 0 * log 0 = NaN and 1 * log 0 = -inf are reproduced (losses.py:71).
// one row, one warp: row_loss[r] = sum(gt * log p), grad = (p - gt) * inv
__device__ __forceinline__ void softmax_ce_row(const float* __restrict__ logits, const float* __restrict__ gt,
                                               float* __restrict__ grad, float* __restrict__ row_loss, int64_t r,
                                               int classes, float inv, int lane) {
    const float* x = logits + r * classes;
    const float* g = gt + r * classes;
    float m = -INFINITY;
    for (int j = lane; j < classes; j += 32) m = fmaxf(m, x[j]);
    m = warp_max(m);
    float s = 0.f;
    for (int j = lane; j < classes; j += 32) s += expf(x[j] - m);
    s = warp_sum(s);
    const float ls = logf(s);
    float l = 0.f;
    for (int j = lane; j < classes; j += 32) {
        const float d = x[j] - m;
        const float gj = g[j];
        const float lp = (d < -745.13f) ? -INFINITY : d - ls;
        l += gj * lp;
        if (grad) grad[r * classes + j] = (expf(d) / s - gj) * inv;
    }
    l = warp_sum(l);
    if (lane == 0) row_loss[r] = l;
}

__global__ void __launch_bounds__(kThreads) softmax_ce_kernel(const float* __restrict__ logits,
                                                              const float* __restrict__ gt,
                                                              float* __restrict__ grad,
                                                              float* __restrict__ row_loss,
                                                              int64_t batch, int classes) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
    const float inv_b = 1.f / (float)batch;
    for (int64_t r = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); r < batch; r += warps)
        softmax_ce_row(logits, gt, grad, row_loss, r, classes, inv_b, lane);
}

// Is row r inside one of the [first, end) ranges?  Binary search for the last range with first <= r: the ranges are
// sorted by `first` (ragged_analysis gives them so); any other table makes the answer wrong, never an access out of
// bounds, since r itself is always a row of the batch.
__device__ __forceinline__ bool row_in_ranges(const int32_t* __restrict__ ranges, int64_t n_ranges, int64_t r) {
    int64_t lo = 0, hi = n_ranges;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((int64_t)__ldg(ranges + 2 * mid) <= r) lo = mid + 1;
        else hi = mid;
    }
    return lo > 0 && r < (int64_t)__ldg(ranges + 2 * (lo - 1) + 1);
}

// softmax_ce_kernel over the rows of the ranges; every other row gets row_loss 0 and a zero gradient row
__global__ void __launch_bounds__(kThreads) softmax_ce_rows_kernel(const float* __restrict__ logits,
                                                                   const float* __restrict__ gt,
                                                                   float* __restrict__ grad,
                                                                   float* __restrict__ row_loss,
                                                                   const int32_t* __restrict__ ranges,
                                                                   int64_t n_ranges, int64_t batch, int classes,
                                                                   float denom) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (kThreads / 32);
    const float inv = 1.f / denom;
    for (int64_t r = (int64_t)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); r < batch; r += warps) {
        if (row_in_ranges(ranges, n_ranges, r)) {
            softmax_ce_row(logits, gt, grad, row_loss, r, classes, inv, lane);
            continue;
        }
        if (grad)
            for (int j = lane; j < classes; j += 32) grad[r * classes + j] = 0.f;
        if (lane == 0) row_loss[r] = 0.f;
    }
}

// out = -sum(v[0:n]) / denom, in double
__device__ __forceinline__ void neg_sum_over(const float* __restrict__ v, int64_t n, double denom,
                                             float* __restrict__ out) {
    __shared__ double part[32];
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) acc += (double)v[i];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double r = warp_sum(part[threadIdx.x]);
        if (threadIdx.x == 0) out[0] = (float)(-r / denom);
    }
}

__global__ void __launch_bounds__(1024) neg_mean_kernel(const float* __restrict__ v, int64_t n,
                                                        float* __restrict__ out) {
    neg_sum_over(v, n, (double)n, out);
}

__global__ void __launch_bounds__(1024) neg_sum_over_kernel(const float* __restrict__ v, int64_t n, float denom,
                                                            float* __restrict__ out) {
    neg_sum_over(v, n, (double)denom, out);
}

// ---------------------------------------------------------------- sigmoid cross-entropy
__global__ void __launch_bounds__(kThreads) sigmoid_ce_kernel(const float* __restrict__ logits,
                                                              const float* __restrict__ gt,
                                                              float* __restrict__ grad,
                                                              float* __restrict__ loss, int64_t n,
                                                              float inv_b) {
    __shared__ float red[8];
    float acc = 0.f;
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * kThreads) {
        const float x = logits[i];
        const float p = 1.f / (1.f + expf(-x));
        const float g = gt[i];
        // log p = -softplus(-x), log(1 - p) = -softplus(x): logf(1 - p) on the FP32 p is -inf from x ~ 16.6 on, where
        // the float64 reference is still finite.  The reference's own 0 * -inf = NaN / -inf are kept where FLOAT64
        // produces them: p == 1.0 for x > 36.74 (1 + e^-x rounds to 1), p == 0.0 for x < -745.13 (e^-x overflows).
        const float t = log1pf(expf(-fabsf(x)));
        float logp = -(fmaxf(-x, 0.f) + t), logq = -(fmaxf(x, 0.f) + t);
        if (x > 36.7368f) { logp = 0.f; logq = -INFINITY; }
        if (x < -745.13f) { logp = -INFINITY; logq = 0.f; }
        acc += g * logp + (1.f - g) * logq;                      // losses.py:54
        // losses.py:56: g (p - 1) + (1 - g) p, with p - 1 formed as -sigmoid(-x): on the FP32 p it cancels to 0 from
        // x ~ 17 on, where the float64 reference still has -e^-x
        if (grad) grad[i] = ((1.f - g) * p - g / (1.f + expf(x))) * inv_b;
    }
    acc = block_sum(acc, red);
    if (threadIdx.x == 0) atomicAdd(loss, -acc * inv_b);
}

// ---------------------------------------------------------------- regularisers
// single CTA (parameter-sized tensors): grad += d reg / dw ; loss += strength * sum(...)
__global__ void __launch_bounds__(1024) regularize_kernel(int kind, const float* __restrict__ w,
                                                          float* grad, float* loss, int64_t n,
                                                          float strength) {
    __shared__ double part[32];
    double acc = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += 1024) {
        const float v = w[i];
        if (kind == UOCR_REG_L2) {
            acc += (double)v * (double)v;
            if (grad) grad[i] += strength * 2.f * v;                       // regularizations.py:25
        } else {
            acc += fabs((double)v);
            const float sgn = (v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f);
            if (grad) grad[i] += strength * sgn;                           // regularizations.py:18
        }
    }
    if (!loss) return;
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double r = warp_sum(part[threadIdx.x]);
        if (threadIdx.x == 0) loss[0] += (float)((double)strength * r);
    }
}

// ---------------------------------------------------------------- optimisers
struct AdamP {
    float lr, b1, b2, eps, gscale, l2;
};

__device__ __forceinline__ void adam_one(float& w, float g, float& v, float& a, const AdamP& p) {
    g = g * p.gscale + p.l2 * 2.f * w;
    v = p.b1 * v + (1.f - p.b1) * g;                       // optimizers.py:58
    a = p.b2 * a + (1.f - p.b2) * g * g;                   // optimizers.py:59
    w -= p.lr / (sqrtf(a) + p.eps) * v;                    // optimizers.py:60-61
}

__global__ void __launch_bounds__(kThreads) adam_kernel(float* w, const float* __restrict__ g, float* v,
                                                        float* a, int64_t n, AdamP p, int vec) {
    if (vec) {
        const int64_t n4 = n / 4;
        float4* w4 = reinterpret_cast<float4*>(w);
        const float4* g4 = reinterpret_cast<const float4*>(g);
        float4* v4 = reinterpret_cast<float4*>(v);
        float4* a4 = reinterpret_cast<float4*>(a);
        for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n4;
             i += (int64_t)gridDim.x * kThreads) {
            float4 ww = w4[i], gg = g4[i], vv = v4[i], aa = a4[i];
            adam_one(ww.x, gg.x, vv.x, aa.x, p);
            adam_one(ww.y, gg.y, vv.y, aa.y, p);
            adam_one(ww.z, gg.z, vv.z, aa.z, p);
            adam_one(ww.w, gg.w, vv.w, aa.w, p);
            w4[i] = ww; v4[i] = vv; a4[i] = aa;
        }
        for (int64_t i = n4 * 4 + (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n;
             i += (int64_t)gridDim.x * kThreads)
            adam_one(w[i], g[i], v[i], a[i], p);
    } else {
        for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n;
             i += (int64_t)gridDim.x * kThreads)
            adam_one(w[i], g[i], v[i], a[i], p);
    }
}

__global__ void __launch_bounds__(kThreads) momentum_kernel(float* w, const float* __restrict__ g,
                                                            float* v, int64_t n, float lr, float mom) {
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * kThreads) {
        const float nv = mom * v[i] - lr * g[i];           // optimizers.py:78
        v[i] = nv;
        w[i] += nv;
    }
}

__global__ void __launch_bounds__(kThreads) rmsprop_kernel(float* w, const float* __restrict__ g,
                                                           float* a, int64_t n, float lr, float rho,
                                                           float eps) {
    for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * kThreads) {
        const float gi = g[i];
        const float na = rho * a[i] + (1.f - rho) * gi * gi;   // optimizers.py:94
        a[i] = na;
        w[i] -= lr / (sqrtf(na) + eps) * gi;
    }
}

}  // namespace uocr

using namespace uocr;

extern "C" {

int uocr_seg_loss_workspace(int64_t n, int64_t c, size_t* bytes) {
    UOCR_REQUIRE(bytes && n > 0 && c > 0, "bad argument");
    *bytes = (size_t)(n * c) * (3 * sizeof(double) + 2 * sizeof(float));
    return UOCR_OK;
}

int uocr_seg_loss(int kind, const float* pred, const float* gt, float* grad, float* loss, int64_t n,
                  int64_t hw, int64_t c, void* workspace, void* stream) {
    UOCR_REQUIRE(kind == UOCR_SEG_DICE || kind == UOCR_SEG_JACCARD, "unknown segmentation loss %d", kind);
    UOCR_REQUIRE(pred && gt && loss && workspace, "NULL pointer");
    UOCR_REQUIRE(n > 0 && hw > 0 && c > 0 && n < 65536 && c < 65536, "bad dimension");
    cudaStream_t st = as_stream(stream);
    const int64_t nc = n * c;
    double* sums = reinterpret_cast<double*>(workspace);
    float* coef = reinterpret_cast<float*>(sums + 3 * nc);
    UOCR_CUDA(cudaMemsetAsync(sums, 0, 3 * nc * sizeof(double), st));
    int64_t chunks = ceil_div(hw, (int64_t)kThreads * 16);
    const int64_t cap = ceil_div(148 * 8, n);
    if (chunks > cap) chunks = cap;
    if (chunks < 1) chunks = 1;
    seg_sums_kernel<<<dim3((unsigned)chunks, (unsigned)n), kThreads, 0, st>>>(pred, gt, sums, hw, (int)c, nc);
    UOCR_LAUNCHED("seg_sums");
    seg_finalize_kernel<<<1, kThreads, 0, st>>>(kind, sums, coef, nc, loss);
    UOCR_LAUNCHED("seg_finalize");
    if (grad) return uocr_seg_grad(gt, nullptr, grad, n, hw, c, workspace, stream);
    return UOCR_OK;
}

int uocr_seg_grad(const float* gt, const float* x_pre, float* out, int64_t n, int64_t hw, int64_t c,
                  const void* workspace, void* stream) {
    UOCR_REQUIRE(gt && out && workspace, "NULL pointer");
    UOCR_REQUIRE(n > 0 && hw > 0 && c > 0 && n < 65536 && c < 65536, "bad dimension");
    cudaStream_t st = as_stream(stream);
    const float* coef = reinterpret_cast<const float*>(reinterpret_cast<const double*>(workspace) + 3 * n * c);
    const int64_t cap = ceil_div(148 * 8, n);
    int64_t gchunks = ceil_div(hw * c, (int64_t)kThreads * 16);
    if (gchunks > cap) gchunks = cap;
    if (gchunks < 1) gchunks = 1;
    const dim3 grid((unsigned)gchunks, (unsigned)n);
    if (x_pre) seg_grad_kernel<true><<<grid, kThreads, 0, st>>>(gt, coef, x_pre, out, hw, (int)c);
    else seg_grad_kernel<false><<<grid, kThreads, 0, st>>>(gt, coef, nullptr, out, hw, (int)c);
    UOCR_LAUNCHED("seg_grad");
    return UOCR_OK;
}

int uocr_seg_loss_ragged(int kind, const float* pred, const float* gt, float* grad, float* loss,
                         const int32_t* extents, int64_t n, int64_t h, int64_t w, int64_t c, void* workspace,
                         void* stream) {
    UOCR_REQUIRE(kind == UOCR_SEG_DICE || kind == UOCR_SEG_JACCARD, "unknown segmentation loss %d", kind);
    UOCR_REQUIRE(pred && gt && loss && extents && workspace, "NULL pointer");
    UOCR_REQUIRE(n > 0 && h > 0 && w > 0 && c > 0 && n < 65536 && c < 65536, "bad dimension");
    cudaStream_t st = as_stream(stream);
    const int64_t nc = n * c;
    double* sums = reinterpret_cast<double*>(workspace);
    float* coef = reinterpret_cast<float*>(sums + 3 * nc);
    UOCR_CUDA(cudaMemsetAsync(sums, 0, 3 * nc * sizeof(double), st));
    int64_t chunks = ceil_div(h * w * c, (int64_t)kThreads * 16);
    const int64_t cap = ceil_div(148 * 8, n);
    if (chunks > cap) chunks = cap;
    if (chunks > h) chunks = h;
    if (chunks < 1) chunks = 1;
    seg_sums_ragged_kernel<<<dim3((unsigned)chunks, (unsigned)n), kThreads, 0, st>>>(pred, gt, extents, sums, h, w,
                                                                                     (int)c, nc);
    UOCR_LAUNCHED("seg_sums_ragged");
    seg_finalize_kernel<<<1, kThreads, 0, st>>>(kind, sums, coef, nc, loss);
    UOCR_LAUNCHED("seg_finalize");
    if (grad) return uocr_seg_grad_ragged(gt, nullptr, grad, extents, n, h, w, c, workspace, stream);
    return UOCR_OK;
}

int uocr_seg_grad_ragged(const float* gt, const float* x_pre, float* out, const int32_t* extents, int64_t n,
                         int64_t h, int64_t w, int64_t c, const void* workspace, void* stream) {
    UOCR_REQUIRE(gt && out && extents && workspace, "NULL pointer");
    UOCR_REQUIRE(n > 0 && h > 0 && w > 0 && c > 0 && n < 65536 && c < 65536, "bad dimension");
    cudaStream_t st = as_stream(stream);
    const float* coef = reinterpret_cast<const float*>(reinterpret_cast<const double*>(workspace) + 3 * n * c);
    int64_t blocks = ceil_div(n * h, kThreads / 32);
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (x_pre) seg_grad_ragged_kernel<true><<<(int)blocks, kThreads, 0, st>>>(gt, coef, x_pre, out, extents, n, h, w, (int)c);
    else seg_grad_ragged_kernel<false><<<(int)blocks, kThreads, 0, st>>>(gt, coef, nullptr, out, extents, n, h, w, (int)c);
    UOCR_LAUNCHED("seg_grad_ragged");
    return UOCR_OK;
}

int uocr_softmax_ce_rows(const float* logits, const float* gt, float* grad, float* loss, const int32_t* ranges,
                         int64_t n_images, int64_t batch, int64_t classes, float denom, float* workspace,
                         void* stream) {
    UOCR_REQUIRE(logits && gt && loss && ranges && workspace, "NULL pointer");
    UOCR_REQUIRE(n_images > 0 && batch > 0 && classes > 0 && classes < (1 << 30), "bad dimension");
    UOCR_REQUIRE(denom > 0.f, "denominator %g must be positive", (double)denom);
    cudaStream_t st = as_stream(stream);
    int64_t blocks = ceil_div(batch, kThreads / 32);
    if (blocks > 148 * 8) blocks = 148 * 8;
    softmax_ce_rows_kernel<<<(int)blocks, kThreads, 0, st>>>(logits, gt, grad, workspace, ranges, n_images, batch,
                                                             (int)classes, denom);
    UOCR_LAUNCHED("softmax_ce_rows");
    neg_sum_over_kernel<<<1, 1024, 0, st>>>(workspace, batch, denom, loss);
    UOCR_LAUNCHED("softmax_ce_rows_loss");
    return UOCR_OK;
}

int uocr_softmax_ce(const float* logits, const float* gt, float* grad, float* loss, int64_t batch,
                    int64_t classes, float* workspace, void* stream) {
    UOCR_REQUIRE(logits && gt && loss && workspace, "NULL pointer");
    UOCR_REQUIRE(batch > 0 && classes > 0 && classes < (1 << 30), "bad dimension");
    cudaStream_t st = as_stream(stream);
    int64_t blocks = ceil_div(batch, kThreads / 32);
    if (blocks > 148 * 8) blocks = 148 * 8;
    softmax_ce_kernel<<<(int)blocks, kThreads, 0, st>>>(logits, gt, grad, workspace, batch, (int)classes);
    UOCR_LAUNCHED("softmax_ce");
    neg_mean_kernel<<<1, 1024, 0, st>>>(workspace, batch, loss);
    UOCR_LAUNCHED("softmax_ce_loss");
    return UOCR_OK;
}

int uocr_sigmoid_ce(const float* logits, const float* gt, float* grad, float* loss, int64_t batch,
                    int64_t classes, void* stream) {
    UOCR_REQUIRE(logits && gt && loss, "NULL pointer");
    UOCR_REQUIRE(batch > 0 && classes > 0, "bad dimension");
    cudaStream_t st = as_stream(stream);
    UOCR_CUDA(cudaMemsetAsync(loss, 0, sizeof(float), st));
    const int64_t n = batch * classes;
    sigmoid_ce_kernel<<<ew_grid(n, 4), kThreads, 0, st>>>(logits, gt, grad, loss, n, 1.f / (float)batch);
    UOCR_LAUNCHED("sigmoid_ce");
    return UOCR_OK;
}

int uocr_regularize(int kind, const float* w, float* grad, float* loss, int64_t n, float strength,
                    void* stream) {
    UOCR_REQUIRE(kind == UOCR_REG_L1 || kind == UOCR_REG_L2, "unknown regulariser %d", kind);
    UOCR_REQUIRE(w && n > 0, "bad argument");
    regularize_kernel<<<1, 1024, 0, as_stream(stream)>>>(kind, w, grad, loss, n, strength);
    UOCR_LAUNCHED("regularize");
    return UOCR_OK;
}

int uocr_adam_update(float* w, const float* g, float* v, float* a, int64_t n, float lr, float beta1,
                     float beta2, float eps, float grad_scale, float l2, float* reg_loss,
                     void* stream) {
    UOCR_REQUIRE(w && g && v && a && n > 0, "bad argument");
    cudaStream_t st = as_stream(stream);
    if (reg_loss && l2 != 0.f) {
        regularize_kernel<<<1, 1024, 0, st>>>(UOCR_REG_L2, w, nullptr, reg_loss, n, l2);
        UOCR_LAUNCHED("adam_reg_loss");
    }
    const int vec = ((reinterpret_cast<uintptr_t>(w) | reinterpret_cast<uintptr_t>(g) |
                      reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(a)) & 15) == 0;
    AdamP p{lr, beta1, beta2, eps, grad_scale, l2};
    adam_kernel<<<ew_grid(n, 4), kThreads, 0, st>>>(w, g, v, a, n, p, vec);
    UOCR_LAUNCHED("adam_update");
    return UOCR_OK;
}

int uocr_momentum_update(float* w, const float* g, float* v, int64_t n, float lr, float momentum,
                         void* stream) {
    UOCR_REQUIRE(w && g && v && n > 0, "bad argument");
    momentum_kernel<<<ew_grid(n, 4), kThreads, 0, as_stream(stream)>>>(w, g, v, n, lr, momentum);
    UOCR_LAUNCHED("momentum_update");
    return UOCR_OK;
}

int uocr_rmsprop_update(float* w, const float* g, float* a, int64_t n, float lr, float rho, float eps,
                        void* stream) {
    UOCR_REQUIRE(w && g && a && n > 0, "bad argument");
    rmsprop_kernel<<<ew_grid(n, 4), kThreads, 0, as_stream(stream)>>>(w, g, a, n, lr, rho, eps);
    UOCR_LAUNCHED("rmsprop_update");
    return UOCR_OK;
}

}  // extern "C"

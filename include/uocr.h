/*
 * uocr.h -- C ABI of libuocr.so: the B200 (sm_100a) implementation of the layer stack of
 * KerkDovan/univer-ocr's self-written deep-learning framework (web_app/components/nn).
 *
 * The reference has NO native boundary: its seam is the Python layer protocol
 * (`BaseLayerGPU._make_forward_gpu/_make_backward_gpu`, nn/layers/layers.py:169-237), whose
 * Numba kernels receive CuPy arrays through __cuda_array_interface__
 * (nn/layers/convolutional.py:185-193).  Every entry point below replaces one of those Python
 * call sites; the `replaces:` note of each function cites it (paths relative to
 * web_app/components/nn/ of the reference).  INTEGRATION.md shows the ctypes stub a
 * maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success, a negative UOCR_ERR_* otherwise;
 *     uocr_last_error() returns a thread-local message for the last failure.
 *   - all array arguments are RAW DEVICE POINTERS (float32 unless noted), NHWC, densely
 *     packed; conv weights are (kh, kw, Cin, Cout), FC weights (n_in + 1, n_out) with the
 *     bias as last row -- the reference's layouts (convolutional.py:41-44, layers.py:324-329).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - asynchronous: nothing synchronises the device except the functions that say so.
 *   - no ownership transfer: the library never frees or retains a caller pointer.
 *   - there is no CPU fallback: without a CUDA device every compute entry point fails with
 *     UOCR_ERR_CUDA.
 */
#ifndef UOCR_H_
#define UOCR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define UOCR_VERSION 100

#define UOCR_OK               0
#define UOCR_ERR_INVALID     -1   /* bad argument (null pointer, non-positive dim, ...)   */
#define UOCR_ERR_CUDA        -2   /* CUDA runtime error, see uocr_last_error()             */
#define UOCR_ERR_UNSUPPORTED -3   /* valid request this build has no kernel for           */
#define UOCR_ERR_WORKSPACE   -4   /* workspace too small                                   */

/* activation fused into a producing kernel / undone in a consuming one */
#define UOCR_ACT_NONE     0
#define UOCR_ACT_LEAKY    1       /* y = x >= 0 ? x : alpha * x   (layers.py:390-401)      */
#define UOCR_ACT_SIGMOID  2       /* y = 1 / (1 + exp(-x))        (layers.py:407-415)      */

/* arithmetic of the contraction kernels */
#define UOCR_MATH_FP32   0        /* FP32 FFMA everywhere ("check mode")                   */
#define UOCR_MATH_TF32   1        /* tcgen05 kind::tf32, FP32 accumulate in TMEM, where a   */
                                  /* tensor-core kernel exists for the shape; else FP32    */

/* ------------------------------------------------------------------ runtime / plumbing */

int         uocr_version(void);
const char* uocr_last_error(void);

int uocr_device_count(int* count);
int uocr_set_device(int device);
int uocr_get_device(int* device);
/* name: caller buffer of name_len bytes; any out pointer may be NULL */
int uocr_device_info(int device, char* name, size_t name_len, int* sm_count,
                     int* cc_major, int* cc_minor, size_t* total_mem, size_t* free_mem);

/* caching device allocator: uocr_free parks the block in a per-(device, stream) free list and
 * uocr_malloc reuses a parked block of the same size class for work queued later on the SAME
 * stream (stream order = reuse order), so steady-state steps never call the driver.  Replaces
 * CuPy's memory pool behind cupy.asarray / cp.zeros (gpu.py:18-22, layers.py:12-13). */
int uocr_malloc(void** ptr, size_t bytes, void* stream);
int uocr_free(void* ptr, void* stream);
int uocr_mempool_trim(void);                        /* cudaFree every parked block (synchronises) */
int uocr_mempool_reserved(size_t* bytes);           /* bytes obtained from cudaMalloc so far */
int uocr_host_alloc(void** ptr, size_t bytes);      /* pinned host memory */
int uocr_host_free(void* ptr);
int uocr_memcpy_h2d(void* dst, const void* src, size_t bytes, void* stream);   /* CP.copy     gpu.py:18-22 */
int uocr_memcpy_d2h(void* dst, const void* src, size_t bytes, void* stream);   /* CP.asnumpy  gpu.py:24-28 */
int uocr_memcpy_d2d(void* dst, const void* src, size_t bytes, void* stream);
int uocr_memset(void* dst, int byte_value, size_t bytes, void* stream);        /* cp.zeros_like, layers.py:13,21 */

int uocr_stream_create(void** stream);
int uocr_stream_destroy(void* stream);
int uocr_stream_sync(void* stream);                 /* blocks the host   */
int uocr_device_sync(void);                         /* blocks the host; replaces cuda.synchronize(), convolutional.py:192 */
int uocr_event_create(void** event);
int uocr_event_destroy(void* event);
int uocr_event_record(void* event, void* stream);
int uocr_event_sync(void* event);                   /* blocks the host   */
int uocr_event_elapsed_ms(void* start, void* stop, float* ms);
int uocr_stream_wait_event(void* stream, void* event);

/* CUDA-graph capture of a launch sequence (one inference step): everything issued on `stream` (and on streams
 * forked from it through events) between _begin and _end becomes one replayable graph.  Blocks freed with
 * uocr_free while capturing stay reserved for the graph (its kernels carry their addresses) until
 * uocr_graph_destroy; uocr_launch_count advances by the captured kernel count on every uocr_graph_launch.
 * The sequence must not synchronise, read back, or depend on host data that changes between replays. */
int uocr_graph_begin(void* stream);
int uocr_graph_end(void* stream, void** graph_exec);
int uocr_graph_launch(void* graph_exec, void* stream);
int uocr_graph_destroy(void* graph_exec);

/* number of kernels this library has launched in this process (all threads) */
int uocr_launch_count(uint64_t* count);

/* ------------------------------------------------------------------ collectives (data-parallel training)
 * The reference has no distributed backend at all (SURVEY.md 2: "Distributed communication backend: none");
 * these entry points are what north_star's "NCCL gradient allreduce over NVLink overlapped with backward" binds
 * (SURVEY.md 8b names them).  One communicator per process (= per GPU).  NCCL is resolved at run time with
 * dlopen -- a libnccl.so.2 already mapped into the process is reused, else `uocr_nccl_load(path)`'s library,
 * else the system one -- so libuocr.so carries no link-time dependency on a particular NCCL build.
 *   uocr_nccl_unique_id : rank 0 creates the 128-byte id; the caller ships it to the other ranks (file, env, ...)
 *   uocr_nccl_init      : collective over all `world` ranks; binds the communicator to the CURRENT device
 *   uocr_allreduce_sum_f32 / uocr_broadcast_f32 : in place, asynchronous on `stream` (capturable into a CUDA graph)
 *   uocr_allreduce_f64  : op 0 = sum, 1 = max, 2 = min (epoch-loss sums, max-over-ranks timings, barriers)
 * Every rank must issue the same collectives in the same order.  UOCR_ERR_COMM on NCCL errors. */
#define UOCR_ERR_COMM        -5   /* NCCL error / not initialised, see uocr_last_error()   */
#define UOCR_NCCL_UNIQUE_ID_BYTES 128
int uocr_nccl_load(const char* path);
int uocr_nccl_version(int* version);
int uocr_nccl_unique_id(void* id_out);
int uocr_nccl_init(int rank, int world, const void* unique_id);
int uocr_nccl_rank(int* rank, int* world);
int uocr_nccl_finalize(void);
int uocr_allreduce_sum_f32(float* data, int64_t count, void* stream);
int uocr_allreduce_f64(double* data, int64_t count, int op, void* stream);
int uocr_broadcast_f32(float* data, int64_t count, int root, void* stream);

/* ------------------------------------------------------------------ array helpers
 * the whole-array NumPy/CuPy expressions the reference's graph executor and Param use */
int uocr_fill_f32(float* dst, float value, int64_t n, void* stream);
int uocr_f64_to_f32(float* dst, const double* src, int64_t n, void* stream);
int uocr_f32_to_f64(double* dst, const float* src, int64_t n, void* stream);
int uocr_u8_to_f32(float* dst, const uint8_t* src, float scale, int64_t n, void* stream); /* encode_layers: /255, train_data_generator.py:24-37 */
/* dst = float32(src / divisor), correctly rounded (== np.float32(u / 255.0) for all 256 pixel values; a multiply by
 * 1/255 is not): uint8 image planes are uploaded as bytes and widened on the device -- 4x less host-link traffic than
 * the reference's float arrays (encode_layers, train_data_generator.py:24-37).  16-byte aligned pointers. */
int uocr_u8_div_f32(float* dst, const uint8_t* src, float divisor, int64_t n, void* stream);
/* y = a * x + b * y   (fan-out gradient sum models.py:218; `param.grad += grad` layers.py:153) */
int uocr_axpby_f32(float* y, const float* x, float a, float b, int64_t n, void* stream);
int uocr_mul_f32(float* out, const float* a, const float* b, int64_t n, void* stream);
/* *flag (int32 on device) |= any(isnan(x))   (BaseLayer.nan_weights, layers.py:139-140) */
int uocr_nan_flag_f32(const float* x, int64_t n, int32_t* flag, void* stream);
/* out[0] (+)= sum(x)  (float64 accumulation inside, float32 result) */
int uocr_sum_f32(const float* x, int64_t n, float* out, int accumulate, void* stream);
/* rows x cols strided 2-D copy, pitches in elements (Concat fwd/bwd, layers.py:240-269) */
int uocr_copy2d_f32(float* dst, int64_t dst_pitch, const float* src, int64_t src_pitch,
                    int64_t rows, int64_t cols, void* stream);
/* zero-pad H and W (make_divisible_by, my_model/model.py:26-34; conv padding)            */
int uocr_pad_hw_f32(float* dst, const float* src, int64_t n, int64_t h, int64_t w, int64_t c,
                    int64_t top, int64_t bottom, int64_t left, int64_t right, float value,
                    void* stream);

/* ------------------------------------------------------------------ Convolutional2D
 * geometry shared by the three conv entry points */
typedef struct uocr_conv2d_desc {
    int64_t n, h, w, cin;        /* input  (N, H, W, Cin)                          */
    int64_t cout;                /* output (N, Ho, Wo, Cout)                       */
    int32_t kh, kw;              /* kernel_size                                     */
    int32_t ph, pw;              /* padding                                         */
    int32_t sh, sw;              /* stride                                          */
    float   padding_value;       /* constant the border is filled with              */
    int32_t bias;                /* reference's `bias` flag (b is multiplied by it) */
    int32_t math_mode;           /* UOCR_MATH_*                                     */
    int32_t in_upsample;         /* 0/1: none.  2: x is (N, H/2, W/2, Cin) and is   */
                                 /* nearest-upsampled x2 on the fly (Upsample2D(2) + */
                                 /* Convolutional2D in one pass): forward, and the   */
                                 /* weight gradient of 5x5 / 1 -> 1 / stride 1 convs */
} uocr_conv2d_desc;

/* Ho = floor((H + 2ph - kh) / sh) + 1 ...   replaces: Convolutional2D.get_output_shapes,
 * convolutional.py:290-301 */
int uocr_conv2d_out_hw(const uocr_conv2d_desc* d, int64_t* ho, int64_t* wo);

/* y = act(conv(x, w) + bias * b).   replaces: Convolutional2D._forward_cpu / _forward_gpu,
 * convolutional.py:62-99 / :147-195 (+ the following LeakyRelu/Sigmoid layer when act != NONE,
 * layers.py:390-415).  x is the UNPADDED input; the border is synthesised from padding_value. */
int uocr_conv2d_fwd(const uocr_conv2d_desc* d, const float* x, const float* w, const float* b,
                    float* y, int act, float alpha, void* stream);
/* Same, with a caller-cached K-major copy of the weights: w_kmajor (Cout, kh*kw*Cin) = uocr_weights_to_kmajor(w,
 * kh*kw*Cin, Cout).  The tensor-core kernels read their B operand K-major; without the copy they transpose w into
 * scratch on every call (a few microseconds per layer -- 4 % of a my_model inference step).  The copy is only read by
 * the tcgen05 paths; every other geometry / math mode uses w as usual.  The caller keeps it in sync with w. */
int uocr_conv2d_fwd_kmajor(const uocr_conv2d_desc* d, const float* x, const float* w, const float* w_kmajor,
                           const float* b, float* y, int act, float alpha, void* stream);
/* wt (n_cols, k_rows) = transpose of w (k_rows, n_cols): conv weights (kh*kw*Cin, Cout), FC weights WITHOUT the bias
 * row (n_in, n_out). */
int uocr_weights_to_kmajor(const float* w, float* wt, int64_t k_rows, int64_t n_cols, void* stream);

/* y = act2(conv3x3(act1(conv3x3(x, w1) + b1), w2) + b2): two chained 3x3 / padding 1 / stride 1
 * convolutions 1 -> c_mid -> 1 channels with the c_mid-channel intermediate kept in registers
 * (inference only: nothing is saved for a backward pass).   replaces: the conv_1 -> leaky_relu_1
 * -> conv_2 -> sigmoid chain of make_monochrome (my_model/model.py:119-122), i.e. four
 * layer calls of convolutional.py:62-99 / layers.py:390-415.   x, y: (N, H, W, 1).
 * math_mode TF32 with c_mid == 16 runs BOTH convolutions on the tensor cores (tcgen05.mma): a persistent kernel
 * whose first convolution reads the image rows in shared memory directly (csrc/conv_pair_rows_tc.cu; W % 4 == 0,
 * W >= 8, 16-byte aligned x), otherwise the kernel that keeps its A operands in tensor memory (csrc/conv_pair_tc.cu).
 * math_mode FP32 and c_mid != 16 run the CUDA-core kernel. */
int uocr_conv3x3_pair_fwd(const float* x, const float* w1, const float* b1, const float* w2,
                          const float* b2, float* y, int64_t n, int64_t h, int64_t w, int32_t c_mid,
                          int act1, float alpha1, int act2, float alpha2, int math_mode, void* stream);

/* y = the whole single-channel "hourglass" network in ONE kernel (inference only):
 *   conv5x5 s2 + LeakyRelu -> conv5x5 s2 + LeakyRelu -> Upsample2D(2), conv5x5 + LeakyRelu ->
 *   Upsample2D(2), conv5x5 + LeakyRelu -> conv5x5 + act_end           (all 1 -> 1 channels, padding 2, zero padding)
 * replaces: make_paragraph's down_1, down_2, up_2, up_1, end blocks (my_model/model.py:137-190), i.e. five
 * Convolutional2D._forward (convolutional.py:62-99), two Upsample2D._forward (upsample.py:21-39) and five
 * activation layers (layers.py:390-415); every intermediate map stays in shared memory.
 * weights / biases: HOST arrays of 5 device pointers in the order down_1, down_2, up_2, up_1, end ((5,5,1,1) and (1)).
 * x, y: (N, H, W, 1) with H % 4 == 0 and W % 4 == 0 (the geometry for which the network's own output shape equals
 * its input shape); UOCR_ERR_UNSUPPORTED otherwise.  FP32 FFMA in every math mode. */
int uocr_hourglass1_fwd(const float* x, const float* const* weights, const float* const* biases, float* y,
                        int64_t n, int64_t h, int64_t w, float alpha, int act_end, float alpha_end, void* stream);
/* the same with a math mode, for callers that carry one: both modes run the same FP32 FFMA kernel, so the result is
 * bit-identical to uocr_hourglass1_fwd. */
int uocr_hourglass1_fwd_mode(const float* x, const float* const* weights, const float* const* biases, float* y,
                             int64_t n, int64_t h, int64_t w, float alpha, int act_end, float alpha_end,
                             int math_mode, void* stream);
/* The four-channel hourglass (make_line, my_model/model.py:194-248: 1 -> 4 -> 4 -> 4 -> 4 -> 2 channels, otherwise the
 * topology above) in ONE tensor-core kernel: every level is tcgen05.mma (TF32 operands, FP32 accumulators in tensor
 * memory) reading the previous level's block in shared memory in place.  weights: (5,5,1,4), (5,5,4,4) x 3, (5,5,4,2);
 * biases (4) x 4, (2); x: (N, H, W, 1), y: (N, H, W, 2), H % 4 == 0 and W % 4 == 0.  A TF32 kernel (tolerance 1e-3 of
 * the output range); callers in UOCR_MATH_FP32 mode run the layers one by one instead. */
int uocr_hourglass4_fwd(const float* x, const float* const* weights, const float* const* biases, float* y,
                        int64_t n, int64_t h, int64_t w, float alpha, int act_end, float alpha_end, void* stream);
/* The kernel reads the five weight tensors in a packed tensor-core operand layout (*floats of uocr_hourglass4_packed_floats
 * floats, 16-byte aligned, TF32-rounded, the two up levels pre-summed per output parity): uocr_hourglass4_fwd packs them
 * on every call; callers that keep the packed image until the weights change call these two instead. */
int uocr_hourglass4_packed_floats(int64_t* floats);
int uocr_hourglass4_pack(const float* const* weights, float* packed, void* stream);
int uocr_hourglass4_fwd_packed(const float* x, const float* packed, const float* const* biases, float* y,
                               int64_t n, int64_t h, int64_t w, float alpha, int act_end, float alpha_end, void* stream);

/* Ragged batches: N images of different sizes on one (N, H, W, C) canvas.  `extents` is a DEVICE table of int32
 * (N, 2): row i = (h_i, w_i), 0 < h_i <= H, 0 < w_i <= W; image i occupies canvas[i, :h_i, :w_i, :] and everything
 * outside that region is 0.  Every layer the networks run pads with zeros (convolutions with padding_value 0,
 * Upsample2D, the window layer), so a valid output pixel computed on the canvas equals the pixel of the image run alone
 * as long as every intermediate map is zero outside its own extent.  Each kernel clamps the extents to the canvas, so
 * a bad table cannot make it write outside the canvas (it can only make the result wrong).
 *
 * uocr_zero_outside_hw_f32: writes 0 to every element of x outside its image's extent.  One warp per canvas row touches
 * only the padding (16-byte stores where the alignment allows), so the cost is the padding, not the tensor.
 * uocr_pack_hw_f32: gathers N contiguous (1, h_i, w_i, c) images into the canvas and writes its zeros, one launch.
 * uocr_unpack_hw_f32: the inverse, scatters canvas[i, :h_i, :w_i, :] to N contiguous images.
 * srcs / dsts: HOST arrays of N device pointers (like the weight-pointer arrays of uocr_hourglass1_fwd); the library
 * copies them into its stream-ordered scratch, so the host array may be released when the call returns. */
int uocr_zero_outside_hw_f32(float* x, const int32_t* extents, int64_t n, int64_t h, int64_t w, int64_t c,
                             void* stream);
int uocr_pack_hw_f32(const float* const* srcs, const int32_t* extents, float* canvas, int64_t n, int64_t h, int64_t w,
                     int64_t c, void* stream);
int uocr_unpack_hw_f32(const float* canvas, const int32_t* extents, float* const* dsts, int64_t n, int64_t h, int64_t w,
                       int64_t c, void* stream);
/* uocr_hourglass4_fwd_packed on a ragged batch: x (N, H, W, 1) canvas, y (N, H, W, 2) canvas, extents as above.  Each
 * level's "inside the image" test uses the image's own extent scaled to that level, so image i's output region is
 * bit-identical to uocr_hourglass4_fwd_packed on that image alone, and y is 0 outside it.  A CTA whose block lies
 * wholly outside its image writes its zeros and exits.  Requires H, W, h_i and w_i to be multiples of 4 (the extents are
 * checked on the device: a CTA of an image that breaks this writes zeros only); UOCR_ERR_UNSUPPORTED for H, W. */
int uocr_hourglass4_fwd_packed_ragged(const float* x, const float* packed, const float* const* biases, float* y,
                                      const int32_t* extents, int64_t n, int64_t h, int64_t w, float alpha, int act_end,
                                      float alpha_end, void* stream);

/* Backward of the same pair in TRAINING (y = conv3x3(act1(conv3x3(x, w1) + b1), w2) + b2, the final
 * activation handled by its own layer): dw1/db1/dw2/db2 (+)= parameter gradients, dx = input gradient
 * (skipped when dx == NULL), from x and dy = dL/dy only -- the c_mid-channel hidden map is recomputed
 * inside the kernels instead of being stored.   replaces: Convolutional2D._backward of conv_2 and
 * conv_1 plus LeakyRelu._backward (convolutional.py:101-145, layers.py:399-401) and the saved
 * (N,H,W,c_mid) activations they need.  act1: UOCR_ACT_LEAKY (alpha > 0) or UOCR_ACT_NONE. */
int uocr_conv3x3_pair_bwd_workspace(int64_t n, int64_t h, int64_t w, int32_t c_mid, size_t* bytes);
/* uocr_conv3x3_pair_bwd_mode: same as uocr_conv3x3_pair_bwd with a math mode; UOCR_MATH_TF32 and c_mid == 16 recompute the
 * hidden map and its gradient with ONE tcgen05 GEMM per 128 pixels (operands resident in tensor memory) and keep only the
 * pixel sums on the CUDA cores (csrc/conv_pair_bwd_tc.cu). */
int uocr_conv3x3_pair_bwd(const float* x, const float* w1, const float* b1, const float* w2, const float* dy,
                          float* dx, float* dw1, float* db1, float* dw2, float* db2, int64_t n, int64_t h,
                          int64_t w, int32_t c_mid, int act1, float alpha1, int accumulate, void* workspace,
                          size_t workspace_bytes, void* stream);
int uocr_conv3x3_pair_bwd_mode(const float* x, const float* w1, const float* b1, const float* w2, const float* dy,
                               float* dx, float* dw1, float* db1, float* dw2, float* db2, int64_t n, int64_t h,
                               int64_t w, int32_t c_mid, int act1, float alpha1, int accumulate, void* workspace,
                               size_t workspace_bytes, int math_mode, void* stream);

/* dx = dgrad(dy, w) (overwrites dx).   replaces: _backward_gpu_kernel_dx + the crop of
 * convolutional.py:141-142 / :203-219,239-250. */
int uocr_conv2d_dgrad(const uocr_conv2d_desc* d, const float* dy, const float* w, float* dx,
                      void* stream);

/* dw (+)= wgrad(x_padded_with_padding_value, dy), db (+)= bias * sum(dy).
 * replaces: _backward_gpu_kernel_dw_db + cp.sum + `w.grad += dw_total`,
 * convolutional.py:221-237,252-265,274-283 (CPU :121-139).  `accumulate` != 0 adds into dw/db
 * (the reference's `+=`), 0 overwrites.  Deterministic two-stage reduction through
 * `workspace` (uocr_conv2d_wgrad_workspace bytes; may be NULL when that is 0). */
int uocr_conv2d_wgrad_workspace(const uocr_conv2d_desc* d, size_t* bytes);
int uocr_conv2d_wgrad(const uocr_conv2d_desc* d, const float* x, const float* dy, float* dw,
                      float* db, int accumulate, void* workspace, size_t workspace_bytes,
                      void* stream);

/* (N, H, W, C) -> (N*W, H, width, C): every width-`width` window of the W axis (zero padded
 * by width, width/2 on the left) becomes a batch row.   replaces:
 * Conv2DToBatchedFixedWidthed._forward/_backward, convolutional.py:335-360. */
int uocr_window_batch_fwd(const float* x, float* y, int64_t n, int64_t h, int64_t w, int64_t c,
                          int32_t width, void* stream);
int uocr_window_batch_bwd(const float* dy, float* dx, int64_t n, int64_t h, int64_t w, int64_t c,
                          int32_t width, void* stream);

/* ------------------------------------------------------------------ MaxPool2D / Upsample2D */

/* Ho/Wo with the reference's floor / ceil rule.  replaces: maxpool.py:204-216 */
int uocr_maxpool2d_out_hw(int64_t h, int64_t w, int32_t kh, int32_t kw, int32_t ph, int32_t pw,
                          int32_t sh, int32_t sw, int32_t ceil_mode, int64_t* ho, int64_t* wo);
/* y = window max over the zero-padded input (padding taps take part with value 0; taps
 * beyond the padded array are skipped); mask (uint8, (N, kh*Ho, kw*Wo, C)) = 1 where a tap
 * -- padding taps included -- equals the max: the reference's CPU semantics, maxpool.py:24-57.
 * Bit-exact outputs. */
int uocr_maxpool2d_fwd(const float* x, float* y, uint8_t* mask, int64_t n, int64_t h, int64_t w,
                       int64_t c, int32_t kh, int32_t kw, int32_t ph, int32_t pw, int32_t sh,
                       int32_t sw, int64_t ho, int64_t wo, void* stream);
/* dx[p] = sum over windows covering p of mask ? dy / tie_count : 0.  replaces: maxpool.py:61-88 */
int uocr_maxpool2d_bwd(const float* dy, const uint8_t* mask, float* dx, int64_t n, int64_t h,
                       int64_t w, int64_t c, int32_t kh, int32_t kw, int32_t ph, int32_t pw,
                       int32_t sh, int32_t sw, int64_t ho, int64_t wo, void* stream);

/* nearest-neighbour repeat by (sy, sx) and its adjoint (block sum); h, w are the SMALL
 * (un-upsampled) sizes.   replaces: upsample.py:21-39 / :41-110 */
int uocr_upsample2d_fwd(const float* x, float* y, int64_t n, int64_t h, int64_t w, int64_t c,
                        int32_t sy, int32_t sx, void* stream);
int uocr_upsample2d_bwd(const float* dy, float* dx, int64_t n, int64_t h, int64_t w, int64_t c,
                        int32_t sy, int32_t sx, void* stream);

/* ------------------------------------------------------------------ activations
 * Relu is Leaky with alpha = 0 (layers.py:377-384).  The backward recomputes the mask from the
 * saved INPUT x, as the reference's stored mask is a function of x only. */
int uocr_leaky_relu_fwd(const float* x, float* y, int64_t n, float alpha, void* stream);
int uocr_leaky_relu_bwd(const float* x, const float* dy, float* dx, int64_t n, float alpha,
                        void* stream);
int uocr_sigmoid_fwd(const float* x, float* y, int64_t n, void* stream);
int uocr_sigmoid_bwd(const float* x, const float* dy, float* dx, int64_t n, void* stream);
/* dx = dy * act'(.) expressed through the activation OUTPUT y (for fused conv+act chains:
 * leaky (alpha > 0): y >= 0 ? 1 : alpha;  sigmoid: y * (1 - y)) */
int uocr_act_bwd_from_output(const float* y, const float* dy, float* dx, int64_t n, int act,
                             float alpha, void* stream);

/* ------------------------------------------------------------------ FullyConnected
 * y = act([x, 1] . W), W (n_in + 1, n_out).   replaces: layers.py:335-339 */
int uocr_fc_fwd(const float* x, const float* w, float* y, int64_t batch, int64_t n_in,
                int64_t n_out, int act, float alpha, int math_mode, void* stream);
/* Same, with a caller-cached K-major copy w_kmajor (n_out, n_in) of the weight rows (see uocr_conv2d_fwd_kmajor);
 * the bias row is still read from w. */
/* y (n*w, n_out) = act([windows(x), 1] . W) for x (n, 1, w, c): Conv2DToBatchedFixedWidthed(width) + Flatten + FullyConnected
 * in one call.   replaces: convolutional.py:330-360 + layers.py:287-294 + layers.py:335-339 (the head of make_char,
 * my_model/model.py:250-304).  In TF32 mode with w % 128 == 0 and c % 32 == 0 the GEMM's A tiles are gathered from x by
 * TMA (implicit 1-D convolution; the (n*w, width*c) window matrix is never materialised); otherwise the windows go
 * through library scratch.  w_kmajor: optional cached K-major copy (n_out, width*c) of W's weight rows, may be NULL. */
int uocr_window_fc_fwd(const float* x, const float* w, const float* w_kmajor, float* y, int64_t n, int64_t wd,
                       int64_t c, int32_t width, int64_t n_out, int act, float alpha, int math_mode, void* stream);
/* y (batch, n_out) = act1([x, 1] . W1) extended by 1, times W2: two FullyConnected layers with an activation between
 * them in one call (make_dense_block, my_model/model.py:251-262: dense_2 + LeakyRelu + dense_3; layers.py:335-347 twice +
 * :390-401).  W1: (n_in + 1, n_hidden), W2: (n_hidden + 1, n_out), bias rows last; w1_kmajor / w2_kmajor: optional cached
 * K-major copies of the weight rows.  In TF32 mode with n_hidden == 128, n_in % 32 == 0, 16 <= n_out <= 256 and
 * batch >= 128 one tcgen05 kernel keeps the hidden tile in shared memory (written by the first epilogue in the operand
 * layout the second GEMM reads); otherwise the two layers run one after the other through library scratch. */
int uocr_fc_chain2_fwd(const float* x, const float* w1, const float* w1_kmajor, const float* w2, const float* w2_kmajor,
                       float* y, int64_t batch, int64_t n_in, int64_t n_hidden, int64_t n_out, int act1, float alpha1,
                       int math_mode, void* stream);
int uocr_fc_fwd_kmajor(const float* x, const float* w, const float* w_kmajor, float* y, int64_t batch, int64_t n_in,
                       int64_t n_out, int act, float alpha, int math_mode, void* stream);
/* dx = dy . W[:-1]^T (skipped when dx == NULL); dw (+)= [x, 1]^T . dy.  replaces: layers.py:341-347 */
int uocr_fc_bwd(const float* x, const float* w, const float* dy, float* dx, float* dw,
                int64_t batch, int64_t n_in, int64_t n_out, int accumulate, int math_mode,
                void* stream);

/* ------------------------------------------------------------------ losses
 * Each writes the gradient w.r.t. `pred` (may be NULL: loss only, Model.test) and ADDS nothing:
 * loss[0] (device float32) is overwritten.  One D2H read per step fetches it. */
#define UOCR_SEG_DICE     0      /* losses.py:9-25   */
#define UOCR_SEG_JACCARD  1      /* losses.py:28-42  */
/* pred, gt: (N, H*W, C).  workspace: uocr_seg_loss_workspace(n, c) bytes, 8-byte aligned. */
int uocr_seg_loss_workspace(int64_t n, int64_t c, size_t* bytes);
int uocr_seg_loss(int kind, const float* pred, const float* gt, float* grad, float* loss,
                  int64_t n, int64_t hw, int64_t c, void* workspace, void* stream);
/* The gradient pass on its own, from the per-(n, c) coefficients a uocr_seg_loss call (grad may have been NULL) left
 * in `workspace`: out = a[n,c] * gt + b[n,c]  (losses.py:24), and with x_pre != NULL multiplied by the Sigmoid
 * derivative exp(-x) / (1 + exp(-x))^2 of the pre-activation tensor the prediction was computed from
 * (layers.py:413-415): loss gradient + Sigmoid._backward of a network's last layer in one pass over memory. */
int uocr_seg_grad(const float* gt, const float* x_pre, float* out, int64_t n, int64_t hw, int64_t c,
                  const void* workspace, void* stream);
/* row softmax cross-entropy, (B, C); loss = -sum(gt * log p) / B, grad = (p - gt) / B;
 * 0 * log 0 -> NaN as in the reference.   replaces: losses.py:60-73 */
int uocr_softmax_ce(const float* logits, const float* gt, float* grad, float* loss, int64_t batch,
                    int64_t classes, float* workspace /* batch floats */, void* stream);
/* replaces: losses.py:45-57 */
int uocr_sigmoid_ce(const float* logits, const float* gt, float* grad, float* loss, int64_t batch,
                    int64_t classes, void* stream);

/* ------------------------------------------------------------------ regularisers + optimisers */
#define UOCR_REG_L1 1            /* regularizations.py:15-19 */
#define UOCR_REG_L2 2            /* regularizations.py:22-26 */
/* grad += d/dw strength * |w| or w^2 ; loss[0] += strength * sum(...)   (BaseLayer.regularize,
 * layers.py:147-155).  grad or loss may be NULL. */
int uocr_regularize(int kind, const float* w, float* grad, float* loss, int64_t n, float strength,
                    void* stream);

/* v = b1 v + (1-b1) g; a = b2 a + (1-b2) g^2; w -= lr / (sqrt(a) + eps) * v -- no bias
 * correction.   replaces: Adam.update, optimizers.py:56-61.
 * Fused extras (0 / 1 reproduce the reference exactly): g is first scaled by grad_scale
 * (1/world for averaged data-parallel gradients) and l2 * 2 * w is added (L2 regulariser folded
 * into the update; the regulariser's gradient is a function of w only).  When `reg_loss` is
 * non-NULL, l2 * sum(w^2) of the PRE-update weights is added to reg_loss[0]. */
int uocr_adam_update(float* w, const float* g, float* v, float* a, int64_t n, float lr, float beta1,
                     float beta2, float eps, float grad_scale, float l2, float* reg_loss,
                     void* stream);
/* v = m v - lr g; w += v.   replaces: optimizers.py:77-79 */
int uocr_momentum_update(float* w, const float* g, float* v, int64_t n, float lr, float momentum,
                         void* stream);
/* a = rho a + (1-rho) g^2; w -= lr / (sqrt(a) + eps) * g.   replaces: optimizers.py:93-96 */
int uocr_rmsprop_update(float* w, const float* g, float* a, int64_t n, float lr, float rho,
                        float eps, void* stream);

/* ------------------------------------------------------------------ exact-index output
 * hits[r, c] (uint8) = pred[r, c] == max(pred[r, :]) && max != 0   -- the index part of
 * PredToText._func1, interpreter/interpreter.py:596-602 (ties keep every column). */
int uocr_row_max_hits(const float* pred, uint8_t* hits, int64_t rows, int64_t cols, void* stream);
/* labels (int32, n x h x w) = connected components of every image of a uint8 mask, counts[n] = their number:
 * foreground = pixels strictly above the image's mean, 4-neighbourhood, labels 1..count in raster order of each
 * component's first pixel -- bit-identical to `ndimage.label(layer > np.mean(layer))` of label_layer
 * (interpreter/interpreter.py:16-22) on a (1, H, W, 1) layer, the first step of every crop stage (:437-470).
 * h * w < 2^31; workspace of uocr_label_components_workspace(n, h, w) bytes. */
int uocr_label_components_workspace(int64_t n, int64_t h, int64_t w, size_t* bytes);
int uocr_label_components(const uint8_t* mask, int32_t* labels, int32_t* counts, int64_t n, int64_t h, int64_t w,
                          void* workspace, void* stream);
/* stats[n][l - 1][0..6] (int64) = pixel count, sum of y, sum of x, y_min, y_max, x_min, x_max of component l of image n
 * (l = 1..max_labels; components beyond max_labels are ignored; absent components: count 0, min > max): the bounding
 * box ndimage.find_objects returns for an object mask and the exact integer sums ndimage.center_of_mass divides
 * (interpreter/interpreter.py:36-38, 125-148, 230, 303, 341, 496-497). */
int uocr_label_stats(const int32_t* labels, int64_t* stats, int64_t n, int64_t h, int64_t w, int64_t max_labels,
                     void* stream);
/* ---- the crop stages' selection and resampling (interpreter/interpreter.py:234-523; SciPy's arithmetic, bit for bit:
 * coordinates in double, every product and sum rounded separately, in ni_interpolation.c's order of operations).
 * out[n, y, x, k] = image[n, y0 + y, x0 + x, k] * (labels[n, y0 + y, x0 + x] == label): `(image * mask)[:, region_y,
 * region_x, :]` with mask = the label_layer object `label` (:303-309); labels == NULL: the plain crop (:511). */
int uocr_crop_masked_f32(const float* image, const int32_t* labels, int32_t label, float* out, int64_t n, int64_t h,
                         int64_t w, int64_t c, int64_t y0, int64_t x0, int64_t ch, int64_t cw, void* stream);
/* out[n, y, x] (uint8) = labels[n, y0 + y, x0 + x] == label: `mask[:, region_y, region_x, :]` (:304). */
int uocr_crop_label_mask(const int32_t* labels, int32_t label, uint8_t* out, int64_t n, int64_t h, int64_t w, int64_t y0,
                         int64_t x0, int64_t ch, int64_t cw, void* stream);
/* dst (n, out_h, out_wp, c) = ndimage.zoom(src (n, h, w, c), (1, out_h / h, out_w / w, 1), order=0) in its first out_w
 * columns, zeros in columns out_w .. out_wp - 1 (the `minimal_width` padding): CropRotateAndZoomLines._func2 (:513-521).
 * out_h, out_w: int(round(h * zf)), int(round(w * zf)) as ndimage.zoom computes them (host side). */
int uocr_zoom_nearest_f32(const float* src, float* dst, int64_t n, int64_t h, int64_t w, int64_t c, int64_t out_h,
                          int64_t out_w, int64_t out_wp, void* stream);
/* dst (n, out_h, out_w, c) = ndimage.rotate(src (n, h, w, c), angle, axes=(2, 1), order, reshape=True): rotate_array
 * (:188-192).  matrix (4 doubles, row-major) / offset (2 doubles): HOST pointers to ndimage.rotate's rot_matrix and
 * offset (input (y, x) = matrix . output (y, x) + offset); order 0 (nearest) or 1 (linear); mode constant, cval 0. */
int uocr_rotate_f32(const float* src, float* dst, int64_t n, int64_t h, int64_t w, int64_t c, int64_t out_h,
                    int64_t out_w, const double* matrix, const double* offset, int order, void* stream);
int uocr_rotate_nearest_u8(const uint8_t* src, uint8_t* dst, int64_t n, int64_t h, int64_t w, int64_t c, int64_t out_h,
                           int64_t out_w, const double* matrix, const double* offset, void* stream);
/* spans[2 k], spans[2 k + 1] (int32, device) = first and last output row of the nearest-rotated mask that holds a
 * non-zero element (INT_MAX, -1 if none), for count = 1 or 2 rotations of the same (n, h, w, c) uint8 mask at once and
 * without materialising them: FindObjectHeightInRotated._func (:229-232) for both probe angles of one step of the
 * ternary search (:318-333).  matrices (count x 4), offsets (count x 2), out_shapes (count x 2): HOST arrays as for
 * uocr_rotate_nearest_u8. */
int uocr_rotated_row_spans(const uint8_t* mask, int32_t* spans, int64_t n, int64_t h, int64_t w, int64_t c, int count,
                           const double* matrices, const double* offsets, const int64_t* out_shapes, int reset,
                           void* stream);
/* spans[0 .. 2 count) = (INT_MAX, -1) pairs: the state uocr_rotated_row_spans accumulates into.  reset != 0 in that
 * call does it for the call's own pairs; a caller that probes many (mask, step) slots resets the whole table once. */
int uocr_row_spans_reset(int32_t* spans, int64_t count, void* stream);
/* box[0..3] (int32, device) = y_min, y_max, x_min, x_max over the non-zero elements of a (n, h, w, c) uint8 array:
 * ndimage.find_objects(mask)[0] of a boolean array (:230, 303, 341); y_max = -1 when the array is all zero. */
int uocr_mask_bbox(const uint8_t* mask, int32_t* box, int64_t n, int64_t h, int64_t w, int64_t c, void* stream);
/* dst[p] = src[p, k] of a (positions, c) uint8 array: one channel of a multi-channel mask, `mask[:, :, :, k:k+1]` (:437-438). */
int uocr_channel_slice_u8(const uint8_t* src, uint8_t* dst, int64_t positions, int64_t c, int64_t k, void* stream);
/* dst[k, p] = src[p, k]: all channels of a (positions, c) uint8 array as c contiguous planes, so that the top / bottom
 * marks of a Line mask are labelled as two images of one uocr_label_components call (:437-447). */
int uocr_channel_planes_u8(const uint8_t* src, uint8_t* dst, int64_t positions, int64_t c, void* stream);
/* mask[n, p, c] (uint8) = x[n, p, c] > mean_p x[n, :, c]: the foreground of label_layer applied to a float map
 * (`layer > np.mean(layer)`, :16-17).  Workspace as for uocr_threshold_mask. */
int uocr_above_mean_mask(const float* x, uint8_t* mask, int64_t n, int64_t hw, int64_t c, void* workspace,
                         void* stream);
/* mask[n, p, c] (uint8) = x[n, p, c] > 0.5 * (mean_p x[n, :, c] + max_p x[n, :, c]) over the
 * hw positions of each (image, channel): the `thresholded()` of the crop stages,
 * interpreter/interpreter.py:437-438 (per mask channel) and :549.  Sums in float64, fixed order
 * (deterministic).  c <= 8; workspace of uocr_threshold_mask_workspace(n, c) bytes. */
int uocr_threshold_mask_workspace(int64_t n, int64_t c, size_t* bytes);
int uocr_threshold_mask(const float* x, uint8_t* mask, int64_t n, int64_t hw, int64_t c, void* workspace,
                        void* stream);

#ifdef __cplusplus
}
#endif
#endif /* UOCR_H_ */

/*
 * a3d.h -- C-ABI of liba3d.so, the B200 (sm_100a) compute library behind ann3depth_b200.
 *
 * The reference (shoeffner/ann3depth) has no native code: its hot path is the set of TensorFlow
 * 1.3 ops that `src/models.py` invokes through `session.run(model_op)` (src/ann3depth.py:126-127).
 * Each entry point below replaces one of those implicit TF kernels; the comment above each
 * function names the reference call sites (file:line under /root/reference) it stands in for.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes.  Every data pointer is a CALLER-OWNED DEVICE pointer
 *    (e.g. torch `tensor.data_ptr()`); the library never allocates device memory.
 *  - Every launch takes an explicit `cudaStream_t` passed as `void*` (0 = legacy default stream).
 *    All entry points are asynchronous and CUDA-graph capturable (no host sync, no allocation).
 *  - Return value: 0 on success; >0 a cudaError_t; <0 an A3D_E* code.  `a3d_last_error()` returns a
 *    thread-local message for the last failure.
 *  - Activations are NHWC.  "bf16" pointers are `uint16_t*` holding bfloat16 bit patterns.
 *  - Convolution kernels are stored OHWI ("packed"): W[Cout][R][S][Cin], i.e. the GEMM K index is
 *    (r*S+s)*Cin+ci.  Dense kernels are stored [out][in].  The TF layouts of the reference
 *    (HWIO and [in,out]) are converted at the Python boundary (ann3depth_b200/params.py).
 *  - No CPU fallback exists: without a CUDA device every launch returns an error.
 */
#ifndef A3D_H_
#define A3D_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define A3D_VERSION 201   /* 201: a3d_dense_wgrad_adam_rows removed.
                             200: a3d_conv_desc gained dil_w / pix_pitch; TF32, model-level and DCNF fully convolutional entry points */

/* negative error codes */
#define A3D_EINVAL   (-1)   /* bad argument / unsupported shape */
#define A3D_ENODEV   (-2)   /* no CUDA device / driver entry point missing */
#define A3D_ETMAP    (-3)   /* cuTensorMapEncode* failed */
#define A3D_ENCCL    (-4)   /* NCCL failure / libnccl not loadable */
#define A3D_ENOTSUP  (-5)   /* configuration not supported by the selected implementation */

/* element types */
#define A3D_F32  0
#define A3D_BF16 1
#define A3D_E4M3 3          /* E4M3 codes (e4m3fn: max 448, no infinities), one byte each: the FP8 inference mode */

/* conv / gemm implementation selector */
#define A3D_IMPL_AUTO 0     /* tcgen05 tensor-core kernels wherever the shape allows */
#define A3D_IMPL_SIMT 1     /* CUDA-core implicit GEMM (debug / shapes tcgen05 cannot take) */
#define A3D_IMPL_TC   2     /* tcgen05 only: error if the shape is not supported */

/* epilogue flags */
#define A3D_EPI_RELU     1u
#define A3D_EPI_SIGMOID  2u
#define A3D_EPI_POOL4    4u   /* a3d_conv2d_pool4_fwd only (set internally) */

typedef struct a3d_ctx a3d_ctx;

/* ---- context ------------------------------------------------------------------------------ */
int  a3d_version(void);
const char* a3d_last_error(void);
/* One context per device / rank.  Not thread-safe per context. */
int  a3d_create(int device, a3d_ctx** out);
int  a3d_destroy(a3d_ctx* ctx);
int  a3d_sm_count(a3d_ctx* ctx);
/* Number of kernels this context has launched since creation (bench.py's "gpu_launches"). */
uint64_t a3d_launch_count(a3d_ctx* ctx);

/* ---- tf.image.resize_images, BILINEAR, TF1 legacy mapping ---------------------------------- */
/* Replaces: src/models.py:282-283 (MSDN preprocessing), :180-181,189-191 (DCNF).
 * src f32 [B,H,W,C] -> dst [B,OH,OW,dstC] (channels >= C are written as zero), dst_dtype F32|BF16. */
int a3d_resize_bilinear_tf1(a3d_ctx*, const float* src, int B, int H, int W, int C,
                            void* dst, int OH, int OW, int dstC, int dst_dtype, void* stream);

/* Same resize, written directly in space-to-depth layout (bf16): an s x s block of resized pixels becomes one
 * pixel of s*s*C channels, dst[b][Y][X][(dy*s+dx)*C + c] = resized[b][s*Y+dy][s*X+dx][c]; channels
 * [s*s*C, dstC) are zero.  dst [B,OH/s,OW/s,dstC].  MSDN (src/models.py:282, then :211 and :241): the 228x304x3
 * image becomes 57x76x64, on which the stride-4 11x11 coarse/conv2d_0 and the pool-fused stride-2 9x9
 * fine/first are both 3x3 stride-1 convolutions with 128-byte pixels. */
int a3d_resize_bilinear_tf1_s2d(a3d_ctx*, const float* src, int B, int H, int W, int C,
                                uint16_t* dst, int OH, int OW, int s, int dstC, void* stream);
/* Same with 8-bit pixels (the images before tools/data_tf_converter.py:36-37 turned them into floats):
 * dst = space-to-depth(resize(src / 255)).  C == 3, s == 4, W*3 a multiple of 16.  A quarter of the bytes over
 * PCIe and HBM; beyond the reference's float32 tensor contract (src/data.py:82-86), offered next to it. */
int a3d_resize_bilinear_tf1_s2d_u8(a3d_ctx*, const uint8_t* src, int B, int H, int W, int C,
                                uint16_t* dst, int OH, int OW, int s, int dstC, void* stream);

/* ---- convolution --------------------------------------------------------------------------- */
typedef struct a3d_conv_desc {
  int N, H, W, C;          /* input  [N,H,W,C]  (C = channels as stored, incl. padding)        */
  int K, R, S;             /* filter [K,R,S,C]  (K = output channels)                           */
  int stride_h, stride_w;
  int pad_t, pad_l;        /* zero padding top/left (bottom/right implied by P,Q)               */
  int P, Q;                /* output [N,P,Q,K]                                                  */
  int ldy;                 /* channel stride of the output tensor (>= K; lets conv write into a
                              wider concat buffer, src/models.py:246)                           */
  int impl;                /* A3D_IMPL_*                                                        */
  /* Overlapped-pixel view (0 / 0 = plain tensor; used by the DCNF first layer, see a3d_extract_patches_s2d):
   * pix_pitch = elements between consecutive pixels when that is LESS than C, i.e. pixel w's C channels are
   * the pix_pitch-wide cells w .. w + C/pix_pitch - 1 of a row of cells; dil_w = horizontal tap spacing in pixels
   * (tap s reads pixel q*stride_w + s*dil_w).  Together: a filter S*C/pix_pitch cells wide over a cell image,
   * consumed in whole 128-byte rows, without materialising the fold.  Honoured by a3d_conv2d_pool4_fwd and
   * a3d_conv2d_wgrad on the tcgen05 path (and their CUDA-core cross-checks); every other call rejects it. */
  int dil_w, pix_pitch;
} a3d_conv_desc;

/* Scratch requirements.  op: 0 = fwd (split-K accumulator), 1 = dgrad (repacked filter + accumulator),
 * 2 = wgrad.  A launch given less scratch than this falls back to a configuration that needs none,
 * or fails with A3D_EINVAL where none exists. */
#define A3D_OP_FWD   0
#define A3D_OP_DGRAD 1
#define A3D_OP_WGRAD 2
size_t a3d_conv2d_ws_bytes(a3d_ctx*, const a3d_conv_desc*, int op);

/* Replaces tf.layers.conv2d forward = Conv2D + BiasAdd [+ Relu]:
 * src/models.py:211-223,241-251 (MSDN), :64-72 (DCNF).  x bf16, w bf16 OHWI, bias f32 (nullable),
 * y bf16 [N,P,Q,ldy] (or f32 when y_dtype == A3D_F32). */
int a3d_conv2d_fwd(a3d_ctx*, const a3d_conv_desc*, const uint16_t* x, const uint16_t* w,
                   const float* bias, void* y, int y_dtype, unsigned flags,
                   void* ws, size_t ws_bytes, void* stream);
/* Replaces Conv2DBackpropInput (autodiff of the above via compute_gradients, src/models.py:314,199).
 * dy bf16 [N,P,Q,ldy], w bf16 OHWI -> dx bf16 [N,H,W,C].
 * relu_src (nullable, bf16 [N,H,W,C]): the post-ReLU activation that was this layer's input; when given
 * the ReluGrad of the producing layer is fused: dx = relu_src > 0 ? dx : 0. */
int a3d_conv2d_dgrad(a3d_ctx*, const a3d_conv_desc*, const uint16_t* dy, const uint16_t* w,
                     uint16_t* dx, const uint16_t* relu_src, void* ws, size_t ws_bytes, void* stream);
/* Same op with the weight-only part hoisted out of the backward chain.  The dgrad of a stride-1 convolution is a
 * forward convolution of dy with the spatially flipped, channel-transposed filter; `prepare` writes that filter
 * (K*R*S*C bf16, caller-owned) from w on any stream once the step's weights are final, `prepared` consumes it.
 * prepare returns A3D_ENOTSUP for shapes whose dgrad does not use a flipped filter (strided convolutions). */
int a3d_conv2d_dgrad_prepare(a3d_ctx*, const a3d_conv_desc*, const uint16_t* w, uint16_t* wflip, void* stream);
int a3d_conv2d_dgrad_prepared(a3d_ctx*, const a3d_conv_desc*, const uint16_t* dy, const uint16_t* wflip,
                              uint16_t* dx, const uint16_t* relu_src, void* ws, size_t ws_bytes, void* stream);
/* Replaces Conv2DBackpropFilter + BiasAddGrad.  dw f32 OHWI, db f32 [K] (nullable).
 * Both are OVERWRITTEN (not accumulated). */
int a3d_conv2d_wgrad(a3d_ctx*, const a3d_conv_desc*, const uint16_t* x, const uint16_t* dy,
                     float* dw, float* db, void* ws, size_t ws_bytes, void* stream);

/* Replaces conv2d + ReLU + max_pooling2d(2, 2) as ONE GEMM (src/models.py:241-243, fine/first): the caller
 * supplies the "pool-embedded" filter in which the four conv outputs of a pool window are four groups of 64
 * filters (K = 256, filter g*64 + c, g = 2*a + b for window position (a, b)) over one common receptive field;
 * the pool is then a max over four accumulator columns of a GEMM row.  y bf16 [N,P,Q,ldy] (64 channels) =
 * act(max_g conv_g + bias[c]); idx u8 [N,P,Q,64] (nullable) = first arg-max g (the MaxPoolGrad routing).
 * Requires C % 64 == 0.  ws: only the A3D_IMPL_SIMT cross-check needs scratch (N*P*Q*256*4 bytes). */
int a3d_conv2d_pool4_fwd(a3d_ctx*, const a3d_conv_desc*, const uint16_t* x, const uint16_t* w,
                         const float* bias, uint16_t* y, uint8_t* idx, unsigned flags,
                         void* ws, size_t ws_bytes, void* stream);
/* MaxPoolGrad + ReluGrad of the above on the GEMM columns:
 * dybig[row][g*64 + c] = (idx[row][c] == g && y[row][c] > 0) ? dy[row][c] : 0   (bf16 [rows][256]);
 * a3d_conv2d_wgrad with the K = 256 descriptor then yields the embedded filter's gradient. */
int a3d_pool4_bwd(a3d_ctx*, const uint16_t* dy, int lddy, const uint16_t* y, int ldy, const uint8_t* idx,
                  uint16_t* dybig, size_t rows, void* stream);
/* Embedded-filter maps: idx int32 [G][n], idx[g][e] = position of canonical element e in copy g of a derived
 * tensor (-1: none).  gather_sum: dst[e] = sum_g src[idx[g][e]] (fold a derived filter's gradient into the
 * canonical variable);  scatter_cast: dst[idx[g][e]] = bf16(src[e]) (refresh the derived filter). */
int a3d_gather_sum_f32(a3d_ctx*, const float* src, const int* idx, int G, size_t n, float* dst, void* stream);
int a3d_scatter_cast_bf16(a3d_ctx*, const float* src, const int* idx, int G, size_t n, uint16_t* dst, void* stream);

/* ---- dense (tf.layers.dense) --------------------------------------------------------------- */
/* Replaces src/models.py:228-232 (MSDN dense_0/1), :80-82,93 (DCNF).
 * x bf16 [M,K] (row stride ldx), w bf16 [N,K] ("[out][in]"), bias f32 [N] (nullable),
 * keep_mask u8 [M,N] (nullable; dropout keep-mask, y *= mask/(1-rate), src/models.py:230),
 * y [M,N] bf16 or f32, acc_ws f32 [M,N] scratch (split-K accumulation). */
int a3d_dense_fwd(a3d_ctx*, const uint16_t* x, int ldx, const uint16_t* w, const float* bias,
                  const uint8_t* keep_mask, float drop_rate, void* y, int y_dtype, float* acc_ws,
                  int M, int N, int K, unsigned flags, int impl, void* stream);
/* dx[M,K] = dy[M,N] . w[N,K]   (MatMul grad wrt input).  dy bf16 with row stride lddy (a multiple of 8
 * elements for the tensor-core path), dx bf16 [M,K], acc_ws f32 [M,K]. */
int a3d_dense_dgrad(a3d_ctx*, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx, float* acc_ws,
                    int M, int N, int K, int impl, void* stream);
/* a3d_dense_dgrad followed by the activation gradient of the layer that produced x, in the dgrad's own finishing pass
 * (MatMul grad -> DropoutGrad -> ReluGrad / SigmoidGrad of src/models.py:228-232 backwards): y_act bf16 [M,K] is that
 * layer's stored post-activation (and post-dropout) output, keep_mask u8 [M,K] nullable, flags A3D_EPI_RELU/SIGMOID.
 * Equals a3d_dense_dgrad + a3d_dense_epilogue_bwd bit for bit. */
int a3d_dense_dgrad_act(a3d_ctx*, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx, float* acc_ws,
                        int M, int N, int K, int impl, const uint16_t* y_act, const uint8_t* keep_mask,
                        float drop_rate, unsigned flags, void* stream);
/* dw[N,K] = dy[M,N]^T . x[M,K] ; db[N] = sum_M dy.   dw/db f32, overwritten. */
int a3d_dense_wgrad(a3d_ctx*, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* dw, float* db,
                    int M, int N, int K, int impl, void* stream);
/* dense wgrad fused with the TF-Adam update of that kernel (single GPU): the gradient tiles are consumed
 * from tensor memory by the optimizer and never written to HBM.  w/m/v f32 [N,K] updated in place, w_bf16
 * (nullable) refreshed; db (nullable) f32 [N] receives the bias gradient.  Same formula and arguments as
 * a3d_adam_tf.  Requires K % 64 == 0 and 16-byte aligned row pitches.  The batch M is at most
 * A3D_DENSE_WGRAD_ADAM_MAX_M (the gradient is formed in two 16-deep mma.sync steps); a larger M, K % 256 != 0 or
 * w/m/v not 16-byte aligned return A3D_ENOTSUP: such callers run a3d_dense_wgrad + a3d_adam_tf instead. */
#define A3D_DENSE_WGRAD_ADAM_MAX_M 32
int a3d_dense_wgrad_adam(a3d_ctx*, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* db,
                         float* w, float* m, float* v, uint16_t* w_bf16, int M, int N, int K,
                         float lr_t, float beta1, float beta2, float eps, float grad_scale,
                         const float* lr_t_dev, void* stream);
/* BiasAddGrad alone: db[c] = sum over rows of dy[row][c] (dy bf16 [rows][ld]).  group_rows > 0: the rows are stored in
 * blocks -- row r is row r % group_rows of block r / group_rows, blocks group_stride elements apart. */
int a3d_bias_grad_bf16(a3d_ctx*, const uint16_t* dy, size_t rows, int C, int ld, float* db, int group_rows,
                       size_t group_stride, void* stream);
/* Elementwise backward of the dense epilogue: g_pre = g_post * mask/(1-rate) * act'(y).
 * y is the stored post-activation (pre-dropout) output; used between dense_1 dgrad and dense_0. */
int a3d_dense_epilogue_bwd(a3d_ctx*, const uint16_t* g_post, const uint16_t* y, const uint8_t* keep_mask,
                           float drop_rate, uint16_t* g_pre, size_t n, unsigned flags, void* stream);

/* ---- max-pool 2x2/2 VALID (tf.layers.max_pooling2d) ---------------------------------------- */
/* Replaces src/models.py:213,216,243 (MSDN), :65,68,73 (DCNF).  x bf16 [N,H,W,C] ->
 * y bf16 [N,H/2,W/2,ldy] (channel stride ldy >= C). */
int a3d_maxpool2x2_fwd(a3d_ctx*, const uint16_t* x, int N, int H, int W, int C,
                       uint16_t* y, int ldy, void* stream);
/* MaxPoolGrad fused with the ReluGrad of the conv that produced x (x is post-ReLU):
 * dx[n,h,w,c] = (x > 0 && (h,w) is the first arg-max of its window) ? dy[n,h/2,w/2,c] : 0.
 * dy has channel stride lddy. Rows/cols not covered by a window get 0. */
int a3d_maxpool2x2_relu_bwd(a3d_ctx*, const uint16_t* x, const uint16_t* dy, int lddy,
                            int N, int H, int W, int C, uint16_t* dx, void* stream);
/* Same pool, but on the f32 conv output and recording the routing decision: idx[n,oh,ow,c] in 0..3 is
 * the first arg-max of the window (row-major), 4 means "blocked" (max <= 0, i.e. the ReLU was inactive).
 * Deciding on f32 values avoids the arg-max ties that bf16-rounded activations produce (about 1 % of
 * windows), which would mis-route gradients relative to the reference's f32 MaxPoolGrad. */
int a3d_maxpool2x2_fwd_f32(a3d_ctx*, const float* x, int N, int H, int W, int C,
                           uint16_t* y, int ldy, uint8_t* idx, void* stream);
/* MaxPoolGrad + ReluGrad from the recorded routing: dx[n,2oh+i/2,2ow+i%2,c] = dy[n,oh,ow,c] where
 * i = idx < 4, zero everywhere else (including the odd trailing row / column). dx bf16 [N,H,W,C]. */
int a3d_maxpool2x2_idx_bwd(a3d_ctx*, const uint8_t* idx, const uint16_t* dy, int lddy,
                           int N, int H, int W, int C, uint16_t* dx, void* stream);
/* ReluGrad alone: dx = (y > 0) ? dy : 0 (dy channel stride lddy, y/dx dense [rows,C]). */
int a3d_relu_bwd(a3d_ctx*, const uint16_t* y, const uint16_t* dy, int lddy, uint16_t* dx,
                 size_t rows, int C, void* stream);

/* ---- scale-invariant log loss (src/models.py:255-275) + its gradient ------------------------ */
/* out,tar f32 [B,n]; loss_per_sample f32 [B]; loss f32 [1] (batch mean);
 * dout (nullable) = d loss / d out, written as f32 and/or bf16 (either pointer may be null) with row
 * stride dout_ld elements (0 = n; the padded stride keeps rows 16-byte aligned for TMA consumers).
 * lambda_over_n is the constant `lambd / (74*55)` of the reference. */
int a3d_silog_loss(a3d_ctx*, const float* out, const float* tar, int B, int n, float lambda_over_n,
                   float* loss_per_sample, float* loss, float* dout_f32, uint16_t* dout_bf16,
                   int dout_ld, void* stream);

/* ---- scale-and-shift-invariant loss (MiDaS, Ranftl et al. 2020) + its gradient -------------------
 * A training objective for relative depth (targets known up to a scale and a shift per image).  out, tar f32 [B, H*W],
 * each row an H x W row-major map; every pixel counts.  Per image, with n = H*W and sums in double over the floats:
 *   fit       D = Spp - Sp^2/n, N = Spg - Sp*Sg/n, sd = N/D, s = float(sd), t = float((Sg - sd*Sp)/n)
 *             (constant prediction, min p == max p or D <= 0: s = 0, t = float(Sg/n), gradient 0)
 *   residual  r_i = (float(s*p_i) + t) - g_i                (float32, no fused multiply-add)
 *   scales    k = 0..scales-1, h = 2^k: grid G_k = {y % h == 0, x % h == 0}, n_k = |G_k|; pairs = horizontally or
 *             vertically adjacent points of G_k (h pixels apart), a before b; D_ab = float(r_a - r_b)
 *   loss      L_b = sum r_i^2 / (2n) + alpha * sum_k (1/n_k) sum_pairs |D_ab|   (double, stored as float)
 *   gradient  dL_b/dp_i = s*r_i/n + alpha*(s*c_i + Q*(g_i - Sg/n - 2*sd*(p_i - Sp/n)) / D), with
 *             c_i = sum_k (1/n_k) sum_{pairs with i} (+sign(D_ab) if i == a, -sign(D_ab) if i == b), sign(0) = 0,
 *             Q = sum_k (1/n_k) sum_pairs sign(D_ab) * (p_a - p_b)
 * loss_per_sample f32 [B]; loss f32 [1] (batch mean); dout as in a3d_silog_loss: d loss / d out (the 1/B included),
 * f32 and/or bf16 (either may be null), row stride dout_ld (0 = H*W).  alpha >= 0, 1 <= scales <= 4,
 * 2*H*W floats must fit in 200 KB of shared memory.  No atomics: the same inputs give the same bits. */
int a3d_ssi_loss(a3d_ctx*, const float* out, const float* tar, int B, int H, int W, float alpha, int scales,
                 float* loss_per_sample, float* loss, float* dout_f32, uint16_t* dout_bf16, int dout_ld,
                 void* stream);

/* ---- optimizers (src/models.py:307-345 Adam x4, :198-200 SGD) ------------------------------- */
/* TF1 ApplyAdam on a flat segment: m = b1*m+(1-b1)*g ; v = b2*v+(1-b2)*g^2 ;
 * w -= lr_t*m/(sqrt(v)+eps), lr_t = lr*sqrt(1-b2^t)/(1-b1^t) computed by the caller in double.
 * g is multiplied by grad_scale first (1/world_size after a sum-allreduce).
 * w_bf16 (nullable) receives the bf16 copy of the updated weights. */
int a3d_adam_tf(a3d_ctx*, float* w, const float* g, float* m, float* v, uint16_t* w_bf16, size_t n,
                float lr_t, float beta1, float beta2, float eps, float grad_scale,
                const float* lr_t_dev /* nullable: device scalar that overrides lr_t, so a captured
                                         CUDA graph can follow the bias-correction schedule */,
                void* stream);
int a3d_sgd(a3d_ctx*, float* w, const float* g, uint16_t* w_bf16, size_t n, float lr,
            float grad_scale, void* stream);
/* a3d_adam_tf with the gradient given in bf16 (the dtype of the data-parallel gradient exchange). */
int a3d_adam_tf_bf16g(a3d_ctx*, float* w, const uint16_t* g_bf16, float* m, float* v, uint16_t* w_bf16, size_t n,
                      float lr_t, float beta1, float beta2, float eps, float grad_scale,
                      const float* lr_t_dev, void* stream);
/* Dropout keep-mask (tf.layers.dropout, src/models.py:230; unseeded in the reference): keep[i] = 1 with
 * probability keep_prob, from a counter-based hash of (seed, *counter_dev, i).  counter_dev is a device
 * int64 (e.g. the global step) so that a captured CUDA graph draws a fresh mask on every replay. */
int a3d_bernoulli_mask(a3d_ctx*, uint8_t* keep, size_t n, float keep_prob, uint64_t seed,
                       const int64_t* counter_dev, void* stream);
/* *p += 1 (device-resident global_step, src/models.py:279,329,343,356). */
int a3d_increment_i64(a3d_ctx*, int64_t* p, void* stream);
/* Timeline probe (src/tfhelper.py:192-249 TraceHook's role, for steps that run as ONE captured CUDA graph and therefore
 * cannot be timed call by call): enqueues a one-thread kernel that stores %globaltimer (ns) in *slot when the stream
 * reaches it.  Not counted as a launch (a3d_launch_count). */
int a3d_stamp(a3d_ctx*, uint64_t* slot, void* stream);
/* f32 -> bf16 cast of a flat segment (weight mirror refresh). */
int a3d_cast_f32_bf16(a3d_ctx*, const float* src, uint16_t* dst, size_t n, void* stream);

/* Space-to-depth by 2: dst[n,i,j,(di*2+dj)*C + c] = src[n,2i+di,2j+dj,c]  (bf16, C % 4 == 0, H and W even).
 * Turns a stride-2 convolution over C channels into a stride-1 convolution over 4C channels with half the
 * filter extent (MSDN fine/first, src/models.py:241: 9x9 stride 2 on 3(4) channels -> 5x5 stride 1 on 16). */
int a3d_space_to_depth2(a3d_ctx*, const uint16_t* src, int N, int H, int W, int C, uint16_t* dst, void* stream);

/* ---- small glue kernels -------------------------------------------------------------------- */
/* Write src f32 [rows] into channel `ch` of a bf16 NHWC buffer with channel stride ld
 * (tf.concat of the coarse map, src/models.py:246). */
int a3d_scatter_channel_bf16(a3d_ctx*, const float* src, uint16_t* dst, size_t rows, int ld, int ch,
                             void* stream);
int a3d_fill_zero(a3d_ctx*, void* p, size_t bytes, void* stream);
/* g[i] = keep[i] ? g[i] : 0 -- clears the gradient of layout-padding entries (zero taps / channels
 * added so that the 3-channel first layers fit the tensor-core path) before the optimizer runs. */
int a3d_apply_mask_f32(a3d_ctx*, float* g, const uint8_t* keep, size_t n, void* stream);

/* ---- DCNF CRF (src/models.py:129-177) ------------------------------------------------------ */
/* Batched closed-form CRF on the static pair graph.  For each of B graphs with n nodes and
 * n_pairs undirected edges (pl[k], pr[k]) with weights r[b,k]:
 *   A = I + diag(R 1) - R ;  y* = A^-1 z (MAP) ;  logdet = log det A ;  quad = z^T A^-1 z ;
 *   energy = y^T A y - 2 z^T y + z^T z ;
 *   nll = energy + n/2 log(pi) - logdet/2 + quad - z^T z          (stable closed form)
 *   dz  = grad_scale * d nll / d z = grad_scale * 2 (y* - y)   ... when dz != NULL (unary gradient)
 *   dr  = grad_scale * d nll / d r[b,k]   ... when dr != NULL (beyond-reference, SURVEY 8f N4)
 * status[b] = 0 ok, k+1 if pivot k of the Cholesky factorisation was not positive (outputs of
 * that graph are then zero, never NaN).  n <= 192.  f32 arrays; pl/pr/status int32.
 * naive != 0 reproduces the reference's literal evaluation (src/models.py:163-171):
 *   nll = -log(exp(-energy)/Z + eps), Z = pi^(n/2)/(sqrt(det A)+eps) * exp(z^T(A^-1+eps)z - z^T z) + eps,
 * eps = 1e-7, which saturates at -log(eps) = 16.118; dz is then scaled by u/(u+eps), u = exp(-energy)/Z. */
int a3d_crf_fwd_bwd(a3d_ctx*, const float* z, const float* y, const float* r, const int32_t* pl,
                    const int32_t* pr, int B, int n, int n_pairs, float grad_scale, int naive,
                    float* ystar, float* nll, float* logdet, float* dz, float* dr, int32_t* status,
                    void* stream);

/* Fused pairwise features (src/models.py:95-127): images f32 [B,H,W,3] (H,W multiples of 40) ->
 * sims f32 [B,n_pairs,2] = (exp(-g*||mean-colour tile l - tile r||), exp(-g*||hist_l - hist_r||)). */
int a3d_pairwise_features(a3d_ctx*, const float* images, int B, int H, int W, const int32_t* pl,
                          const int32_t* pr, int n_pairs, float gamma, float* tile_feat_ws,
                          float* sims, void* stream);
/* The 2 -> 1 `pairwise_dense` layer (src/models.py:91-93): r[i] = sims[i,0]*w[0] + sims[i,1]*w[1] + b[0]. */
int a3d_pairwise_dense(a3d_ctx*, const float* sims, const float* w2, const float* b1, float* r, size_t n,
                       void* stream);
/* Beyond the reference (SURVEY.md 8f N4): r = act(sims . w + b) with act = max(., 0) for A3D_EPI_RELU (keeps A = I + D - R
 * SPD; the reference's layer is unconstrained, src/models.py:92-93), and the gradient into the pairwise layer from the CRF
 * kernel's dr (TF 1.3 blocks it): dw2[j] = sum_i dr[i] act'(r[i]) sims[i][j], db1 = sum_i dr[i] act'(r[i]). */
int a3d_pairwise_dense_act(a3d_ctx*, const float* sims, const float* w2, const float* b1, float* r, size_t n,
                           unsigned flags, void* stream);
int a3d_pairwise_dense_bwd(a3d_ctx*, const float* sims, const float* r, const float* dr, float* dw2, float* db1, size_t n,
                           unsigned flags, void* stream);
/* out[0] = mean(v[0..n)) (tf.reduce_mean of per-sample losses, src/models.py:174,272). */
int a3d_mean_f32(a3d_ctx*, const float* v, int n, float* out, void* stream);
/* f32 -> bf16 with scaling: dst[i] = bf16(scale * src[i]). */
int a3d_scale_cast_bf16(a3d_ctx*, const float* src, uint16_t* dst, size_t n, float scale, void* stream);
size_t a3d_pairwise_ws_bytes(int B, int H, int W);
/* Tile means of a 1-channel map (src/models.py:131-132): depth f32 [B,H,W] -> y f32 [B,n]. */
int a3d_tile_means(a3d_ctx*, const float* depth, int B, int H, int W, float* y, void* stream);
/* Gather 100x100 stride-40 SAME patches (src/models.py:50-59) as bf16 NHWC with dstC channels:
 * images f32 [B,H,W,3] -> patches bf16 [B*rows*cols,100,100,dstC]. */
int a3d_extract_patches(a3d_ctx*, const float* images, int B, int H, int W, uint16_t* patches,
                        int dstC, void* stream);
/* The same patches after space-to-depth(2), for the pool-fused first layer (11x11 conv + ReLU + 2x2 max-pool as ONE
 * 6x6-cell convolution with 4 x 64 filters, a3d_conv2d_pool4_fwd): cells bf16 [B*n][50][50][16], channel (2a+b)*3+c =
 * patch pixel (2Y+a, 2X+b, c), channels 12..15 zero (fold = 1); fold = 4 writes [B*n][50][50][64] with position X
 * holding cells X..X+3.  The layer reads the fold = 1 tensor through a3d_conv_desc{C = 64, S = 2, dil_w = 4,
 * pix_pitch = 16}: whole 128-byte rows per TMA load, a quarter of the bytes.  The caller keeps >= 128 zero bytes after
 * the fold = 1 tensor (the last positions of the last row read past it, against zero weights). */
int a3d_extract_patches_s2d(a3d_ctx*, const float* images, int B, int H, int W, uint16_t* cells, int fold, void* stream);
/* Fully convolutional form of the DCNF unary network (src/models.py:50-83): the patches are plain windows (stride 40,
 * zero border 30) and every layer is a VALID convolution or an even-aligned 2x2 pool, so each layer of patch (prow, pcol)
 * is a window of the same layer of the zero-padded whole image.  a3d_image_cells_s2d: the padded image after
 * space-to-depth(2), cells bf16 [B][(H+2pad)/2][(W+2pad)/2][16] (channel (2a+b)*3+c, 12..15 zero; keep >= 128 zero bytes
 * after it for the overlapped view).  a3d_window_gather: out [B*rows*cols][win][win][C] = the windows of src [B,Hs,Ws,C]
 * at stride `stride` (the per-patch inputs of the first dense layer: 7x7x256 at stride 5).  a3d_window_scatter_sum: its
 * transpose for the backward pass (float32 sum over the overlapping windows, one bf16 rounding). */
int a3d_image_cells_s2d(a3d_ctx*, const float* images, int B, int H, int W, int pad, uint16_t* cells, void* stream);
int a3d_window_gather(a3d_ctx*, const uint16_t* src, int B, int Hs, int Ws, int C, int rows, int cols, int win, int stride,
                      uint16_t* out, void* stream);
int a3d_window_scatter_sum(a3d_ctx*, const uint16_t* g_out, int B, int Hs, int Ws, int C, int rows, int cols, int win,
                           int stride, uint16_t* g_src, void* stream);

/* ---- depth-estimation metrics (Eigen et al. 2014), beyond the reference (it has no evaluation) -----------------------
 * pred f32 [B,ph,pw] is sampled at every pixel of gt f32 [B,gh,gw] with the TF1 legacy bilinear mapping of
 * a3d_resize_bilinear_tf1, bit for bit (no upsampled map is materialised).  Valid pixels: min_depth < gt <= max_depth
 * (0 < min_depth < max_depth).  p~ = the sampled prediction clamped to [min_depth, max_depth]; a NaN maps to min_depth.
 * scale_mode A3D_DM_SCALE_NONE: p = p~.  A3D_DM_SCALE_MEDIAN: s = median(gt) / median(p~) over the valid pixels (float32
 * division of the two exact lower medians, the elements of rank floor((n-1)/2)), p = clamp(s * p~); s = 1 for an image
 * without a valid pixel.  A3D_DM_SCALE_AFFINE (for relative depth, known only up to a scale and shift per image):
 * (s, t) = argmin sum (s * p~ + t - g)^2 over the valid pixels, in float64 from the raw moments:
 *   n, mp = sum p~ / n, mg = sum g / n, Sxx = sum p~^2 - sum p~ * mp, Sxy = sum p~ g - sum p~ * mg,
 *   sd = Sxy / Sxx (may be negative), or sd = 1 when min p~ = max p~ or Sxx <= 0 (a constant prediction),
 *   s = float32(sd), t = float32(mg - sd * mp);  s = 1, t = 0 for an image without a valid pixel;
 *   p = fminf(fmaxf(float32(float32(s * p~) + t), min_depth), max_depth) (two float32 roundings, no fused
 *   multiply-add; a NaN maps to min_depth).
 * With d = ln p - ln g, writes sums[b][A3D_DM_*] (float64, overwritten per image) over the
 * valid pixels, and if `scale` is non-null: scale[b] = s (NONE, MEDIAN) or scale[b][0..1] = (s, t) (AFFINE, [B][2]).
 * The ratio tests are float32: max(p/g, g/p) < 1.25^k.
 * No workspace, no host sync, CUDA-graph capturable; the sums do not depend on scheduling (fixed reduction order). */
#define A3D_DM_SCALE_NONE    0
#define A3D_DM_SCALE_MEDIAN  1
#define A3D_DM_SCALE_AFFINE  2
#define A3D_DM_N          0   /* number of valid pixels */
#define A3D_DM_ABS_REL    1   /* sum |p - g| / g */
#define A3D_DM_SQ_REL     2   /* sum (p - g)^2 / g */
#define A3D_DM_SQ         3   /* sum (p - g)^2 */
#define A3D_DM_LOG        4   /* sum d */
#define A3D_DM_LOG_SQ     5   /* sum d^2 */
#define A3D_DM_LOG10      6   /* sum |d| / ln 10 = sum |log10 p - log10 g| */
#define A3D_DM_DELTA1     7   /* count max(p/g, g/p) < 1.25 */
#define A3D_DM_DELTA2     8   /* count ... < 1.25^2 */
#define A3D_DM_DELTA3     9   /* count ... < 1.25^3 */
#define A3D_DM_NONFINITE 10   /* count of valid pixels whose sampled prediction was NaN or +-inf */
#define A3D_DM_SLOTS     11
int a3d_depth_metrics(a3d_ctx*, const float* pred, int B, int ph, int pw, const float* gt, int gh, int gw,
                      float min_depth, float max_depth, int scale_mode, double* sums, float* scale, void* stream);

/* ---- training-time augmentation (Eigen et al. 2014, section 3.3), beyond the reference (it has none) ------------------
 * Every image of a batch gets one random transform, shared by the image and its depth target:
 *   output pixel (oy, ox) of an OH x OW output sits at the TF1 legacy position (u, v) = (ox*W/OW, oy*H/OH) (tf1_coord);
 *   p = (u/W, v/H); T(p) = c + R(theta) F (p - 1/2) f/s = M p + m (M, m: the normalised 2x3 matrix below), with
 *   R(theta) a rotation in the pixel space of a frame of height/width `aspect`, F = diag(+-1, 1) the horizontal flip,
 *   f the crop fraction, s the scale, c the crop centre;
 *   the source is sampled at T(p) * (W, H), clamped to [0, W-1] x [0, H-1] (border replicated), with TF1 bilinear.
 * Each tensor applies the transform in its own pixel units, so a 480x640 image and a 55x73 depth map see one geometry.
 * Values: images are multiplied per channel by c_rgb after interpolation (one rounding to the storage type); depths by
 * 1/s.  With identity parameters both resize entry points write exactly what the plain TF1 resizes write. */
typedef struct a3d_augment_desc {
  float scale_lo, scale_hi;     /* s ~ U[scale_lo, scale_hi], > 0 */
  float max_rotation_deg;       /* theta ~ U[-max, max] degrees */
  float crop_fraction;          /* f in (0, 1]: the window spans f/s of the frame */
  float flip_prob;              /* P(horizontal flip) */
  float color_lo, color_hi;     /* c_rgb ~ U[color_lo, color_hi]^3 */
  float aspect;                 /* height / width of the frame the rotation is a rotation of (0.75 for 480x640) */
} a3d_augment_desc;
/* params [B][A3D_AUG_PARAMS] float32, one row per image */
#define A3D_AUG_M00       0    /* T_x(p) = M00 p_x + M01 p_y + M02 */
#define A3D_AUG_M01       1
#define A3D_AUG_M02       2
#define A3D_AUG_M10       3    /* T_y(p) = M10 p_x + M11 p_y + M12 */
#define A3D_AUG_M11       4
#define A3D_AUG_M12       5
#define A3D_AUG_COLOR     6    /* c_r, c_g, c_b at 6, 7, 8 */
#define A3D_AUG_INV_SCALE 9    /* 1/s */
#define A3D_AUG_SCALE    10    /* raw draws, for inspection: s, theta (degrees), flip (0/1), c_x, c_y, f */
#define A3D_AUG_THETA    11
#define A3D_AUG_FLIP     12
#define A3D_AUG_CX       13
#define A3D_AUG_CY       14
#define A3D_AUG_CROP     15
#define A3D_AUG_PARAMS   16
#define A3D_AUG_VALUE_COLOR 0  /* a3d_resize_affine_tf1 value rule: v * c_rgb[c] (C <= 3) */
#define A3D_AUG_VALUE_DEPTH 1  /* v / s */
#define A3D_U8 2               /* source dtype of a3d_resize_affine_tf1_s2d: 8-bit pixels, read as pixel / 255 */
/* Draws params[b] from a splitmix64 hash of (seed, *counter_dev, b) in float64 (ranges of `desc`), on the device: a
 * replayed CUDA graph draws fresh parameters whenever *counter_dev (the global step) moves.  counter_dev may be NULL
 * (counter 0).  c_x, c_y ~ 1/2 + U[-1, 1] (1 - f/s)/2: the unrotated window lies inside the frame. */
int a3d_augment_draw(a3d_ctx*, const a3d_augment_desc* desc, int B, uint64_t seed, const int64_t* counter_dev,
                     float* params, void* stream);
/* The MSDN image path: augmented resize written in the space-to-depth(s) layout of a3d_resize_bilinear_tf1_s2d.
 * src_dtype A3D_F32 or A3D_U8 (pixel / 255); dst_dtype A3D_BF16 or A3D_F32.  C == 3, s == 4, dstC % 4 == 0, >= 48
 * (channels [48, dstC) zero), dst 16-byte aligned.  Colour value rule. */
int a3d_resize_affine_tf1_s2d(a3d_ctx*, const void* src, int src_dtype, int B, int H, int W, int C, void* dst,
                              int dst_dtype, int OH, int OW, int s, int dstC, const float* params, void* stream);
/* Generic NHWC: src f32 [B,H,W,C] -> dst f32 [B,OH,OW,C], C <= 4; value_mode A3D_AUG_VALUE_COLOR | _DEPTH. */
int a3d_resize_affine_tf1(a3d_ctx*, const float* src, int B, int H, int W, int C, float* dst, int OH, int OW,
                          const float* params, int value_mode, void* stream);

/* ---- data parallelism (replaces the PS/gRPC replication of src/ann3depth.py:78-92) ---------- */
/* NCCL is dlopen()ed at first use (path = NULL -> "libnccl.so.2"). */
int a3d_comm_unique_id(const char* nccl_path, void* id128);              /* 128-byte ncclUniqueId */
int a3d_comm_init(a3d_ctx*, const char* nccl_path, const void* id128, int rank, int nranks);
int a3d_comm_destroy(a3d_ctx*);
/* In-place sum-allreduce of a flat gradient bucket on `stream`. */
int a3d_allreduce_sum(a3d_ctx*, void* buf, size_t count, int dtype, void* stream);
/* Sharded-optimizer exchange (reduce-scatter gradients -> each rank updates its 1/n slice -> all-gather the
 * bf16 weight mirror).  Both are in place on a buffer of nranks*chunk elements: after the reduce-scatter,
 * rank r holds the sum in buf[r*chunk, (r+1)*chunk); the all-gather publishes every rank's slice. */
int a3d_reduce_scatter_sum(a3d_ctx*, void* buf, size_t chunk, int dtype, void* stream);
int a3d_allgather(a3d_ctx*, void* buf, size_t chunk, int dtype, void* stream);
/* n all-gathers as one NCCL group (one launch): bufs[i] = nranks * chunks[i] elements, gathered in place. */
int a3d_allgather_multi(a3d_ctx*, void* const* bufs, const size_t* chunks, int n, int dtype, void* stream);

/* ---- TF32 precision mode ------------------------------------------------------------------------------------------
 * models.msdn(images, depths, dtype="tf32"): every activation / activation gradient is a float32 tensor (the reference's
 * own storage type), the contractions run on tcgen05.mma kind::tf32 with float32 accumulation.  Same operations, layouts
 * (NHWC, OHWI filters, [out][in] dense kernels) and TF call sites as the bf16 entry points above; C must be a multiple of
 * 32 for the convolutions (128-byte pixels), K of 32 for the dense layers.  Weights are the float32 master copy itself. */
size_t a3d_conv2d_ws_bytes_tf32(a3d_ctx*, const a3d_conv_desc*, int op);
int a3d_conv2d_fwd_tf32(a3d_ctx*, const a3d_conv_desc*, const float* x, const float* w, const float* bias, float* y,
                        unsigned flags, void* ws, size_t ws_bytes, void* stream);
int a3d_conv2d_dgrad_tf32(a3d_ctx*, const a3d_conv_desc*, const float* dy, const float* w, float* dx,
                          const float* relu_src, void* ws, size_t ws_bytes, void* stream);
int a3d_conv2d_wgrad_tf32(a3d_ctx*, const a3d_conv_desc*, const float* x, const float* dy, float* dw, float* db,
                          void* stream);
int a3d_dense_fwd_tf32(a3d_ctx*, const float* x, int ldx, const float* w, const float* bias, const uint8_t* keep_mask,
                       float drop_rate, float* y, float* acc_ws, int M, int N, int K, unsigned flags, void* stream);
/* y_act / keep_mask nullable: the producer layer's activation gradient folded into the finishing pass */
int a3d_dense_dgrad_tf32(a3d_ctx*, const float* dy, int lddy, const float* w, float* dx, float* acc_ws, int M, int N,
                         int K, const float* y_act, const uint8_t* keep_mask, float drop_rate, unsigned flags,
                         void* stream);
int a3d_dense_wgrad_tf32(a3d_ctx*, const float* x, int ldx, const float* dy, int lddy, float* dw, float* db, int M, int N,
                         int K, void* stream);
/* float32 counterparts of the memory-bound kernels (f32_ops.cu) */
int a3d_resize_bilinear_tf1_s2d_f32(a3d_ctx*, const float* src, int B, int H, int W, int C, float* dst, int OH, int OW,
                                    int s, int dstC, void* stream);
int a3d_maxpool2x2_f32(a3d_ctx*, const float* x, int N, int H, int W, int C, float* y, int ldy, uint8_t* idx, void* stream);
int a3d_maxpool2x2_idx_bwd_f32(a3d_ctx*, const uint8_t* idx, const float* dy, int lddy, int N, int H, int W, int C,
                               float* dx, void* stream);
int a3d_act_bwd_f32(a3d_ctx*, const float* g_post, int ldg, const float* y, const uint8_t* keep_mask, float drop_rate,
                    float* g_pre, size_t rows, int C, unsigned flags, void* stream);
int a3d_scatter_channel_f32(a3d_ctx*, const float* src, float* dst, size_t rows, int ld, int ch, void* stream);
int a3d_pool4_reduce_f32(a3d_ctx*, const float* acc, const float* bias, float* y, int ldy, uint8_t* idx, size_t rows,
                         unsigned flags, void* stream);
int a3d_pool4_bwd_f32(a3d_ctx*, const float* dy, int lddy, const float* y, int ldy, const uint8_t* idx, float* dybig,
                      size_t rows, void* stream);
int a3d_bias_grad_f32(a3d_ctx*, const float* dy, size_t rows, int C, int ld, float* db, void* stream);
int a3d_scatter_f32(a3d_ctx*, const float* src, const int* idx, int G, size_t n, float* dst, void* stream);
/* 3xTF32 forward ("tf32x3" precision mode): both operands are split into hi = tf32(x) and lo = x - hi (a3d_split_tf32;
 * rows x cols floats at pitch ld, outputs dense) and  lo.hi + hi.lo + hi.hi  is summed in the float32 accumulator --
 * float32-grade Conv2D / MatMul (src/models.py:211-251) at three times the kind::tf32 tensor work.  Same arguments as
 * a3d_conv2d_fwd_tf32 / a3d_dense_fwd_tf32 except for the workspace, whose size the *_ws_bytes_tf32x3 calls return. */
int a3d_split_tf32(a3d_ctx*, const float* x, size_t rows, int cols, long long ld, float* hi, float* lo, void* stream);
size_t a3d_conv2d_ws_bytes_tf32x3(a3d_ctx*, const a3d_conv_desc*);
int a3d_conv2d_fwd_tf32x3(a3d_ctx*, const a3d_conv_desc*, const float* x, const float* w, const float* bias, float* y,
                          unsigned flags, void* ws, size_t ws_bytes, void* stream);
size_t a3d_dense_ws_bytes_tf32x3(int M, int N, int K);
int a3d_dense_fwd_tf32x3(a3d_ctx*, const float* x, int ldx, const float* w, const float* bias, const uint8_t* keep_mask,
                         float drop_rate, float* y, void* ws, size_t ws_bytes, int M, int N, int K, unsigned flags,
                         void* stream);
/* single-filter convolution (K == 1: MSDN fine/third, src/models.py:250) in exact float32: forward, dgrad (+ ReluGrad
 * of relu_src, nullable), wgrad (+ db, nullable).  dy / y row pitch = ldy floats. */
int a3d_conv_k1_fwd_f32(a3d_ctx*, const a3d_conv_desc*, const float* x, const float* w, const float* bias, float* y,
                        unsigned flags, void* stream);
int a3d_conv_k1_dgrad_f32(a3d_ctx*, const a3d_conv_desc*, const float* dy, const float* w, float* dx,
                          const float* relu_src, void* stream);
int a3d_conv_k1_wgrad_f32(a3d_ctx*, const a3d_conv_desc*, const float* x, const float* dy, float* dw, float* db,
                          void* stream);

/* ---- model-level entry points (SURVEY.md 8b): the whole MSDN step behind the C-ABI ---------------------------------
 * A host in any language drives `session.run(model_op)` (src/ann3depth.py:126-127) for `models.msdn`
 * (src/models.py:203-367) with these calls alone.  The caller owns ONE device buffer of a3d_msdn_workspace_bytes() that
 * the net carves into parameter arena (f32 master / gradients / Adam m, v / bf16 mirror; segment table =
 * a3d_msdn_segment, packed layouts of ann3depth_b200/params.py), activations and scratch.  Sequential single-stream
 * schedule, BF16 storage; forward of both stacks + both losses, backward + TF-Adam of the active tf.case branch
 * (phase 1 coarse / 2 fine / 3 idle by global_step, src/models.py:301-364), global_step += 1. */
typedef struct a3d_msdn a3d_msdn;
size_t a3d_msdn_workspace_bytes(a3d_ctx*, int batch, int in_h, int in_w, int depth_h, int depth_w, int train);
int a3d_msdn_create(a3d_ctx*, int batch, int in_h, int in_w, int depth_h, int depth_w, int train, void* workspace,
                    size_t workspace_bytes, void* stream, a3d_msdn** out);
int a3d_msdn_destroy(a3d_msdn*);
/* beta2 of the four AdamOptimizers (src/models.py:309 passes 1: the default) and the dropout seed */
int a3d_msdn_configure(a3d_msdn*, float adam_beta2, uint64_t dropout_seed);
/* segment `index` of the arena: TF variable name, element offset, element count, packed shape; returns the segment count */
int a3d_msdn_segment(const a3d_msdn*, int index, const char** name, size_t* offset, size_t* numel, int shape[4]);
/* device pointers of the arena buffers (each `total` elements); after writing `w` call a3d_msdn_sync_weights */
int a3d_msdn_arena(a3d_msdn*, float** w, float** m, float** v, float** g, uint16_t** w_bf16, size_t* total);
int a3d_msdn_sync_weights(a3d_msdn*, void* stream);
int a3d_msdn_set_step(a3d_msdn*, long long global_step, const int adam_t[4], void* stream);
long long a3d_msdn_global_step(const a3d_msdn*);
/* one step = host half (counters, Adam step sizes -> device scalars; returns the phase, < 0 on error) + device half
 * (kernel launches only: capturable in a CUDA graph, one graph per phase).  a3d_msdn_step does both and copies the two
 * losses (coarse, fine) to `losses` (device, nullable).  images f32 [B,in_h,in_w,3], depths f32 [B,depth_h,depth_w,1],
 * keep_mask u8 [B,4096] or NULL (device RNG, Bernoulli(0.5) per (seed, global_step)). */
int a3d_msdn_step_begin(a3d_msdn*, void* stream);
int a3d_msdn_step_enqueue(a3d_msdn*, int phase, const float* images, const float* depths, const uint8_t* keep_mask,
                          void* stream);
int a3d_msdn_step(a3d_msdn*, const float* images, const float* depths, const uint8_t* keep_mask, float* losses,
                  void* stream);
/* inference (dropout off): fine / coarse depth maps f32 [B,55,74] (device, nullable) */
int a3d_msdn_infer(a3d_msdn*, const float* images, float* fine, float* coarse, void* stream);
const float* a3d_msdn_losses(const a3d_msdn*);

/* ---- the whole DCNF step behind the C-ABI (models.dcnf, src/models.py:9-200): counterpart of a3d_msdn_* ---------------
 * Caller-owned workspace; arena = f32 master / gradients / bf16 mirror (plain SGD: no optimizer slots), segment table and
 * packed layouts of ann3depth_b200/params.py dcnf_specs().  a3d_dcnf_step = forward (resize, patches, unary CNN on B*48
 * patches, pairwise features, CRF NLL) + backward through the unary CNN + SGD lr 0.1; kernel launches only (capturable). */
typedef struct a3d_dcnf a3d_dcnf;
size_t a3d_dcnf_workspace_bytes(a3d_ctx*, int batch, int in_h, int in_w, int depth_h, int depth_w, int train);
int a3d_dcnf_create(a3d_ctx*, int batch, int in_h, int in_w, int depth_h, int depth_w, int train, void* workspace,
                    size_t workspace_bytes, void* stream, a3d_dcnf** out);
int a3d_dcnf_destroy(a3d_dcnf*);
int a3d_dcnf_configure(a3d_dcnf*, int naive_loss);   /* 1 (default): the reference's exp(-E)/Z form; 0: stable closed form */
int a3d_dcnf_segment(const a3d_dcnf*, int index, const char** name, size_t* offset, size_t* numel, int shape[4]);
int a3d_dcnf_arena(a3d_dcnf*, float** w, float** g, uint16_t** w_bf16, size_t* total);
int a3d_dcnf_sync_weights(a3d_dcnf*, void* stream);
long long a3d_dcnf_global_step(const a3d_dcnf*);
int a3d_dcnf_step(a3d_dcnf*, const float* images, const float* depths, float* loss, void* stream);
/* output f32 [B,240,320] (upsampled unary prediction), z f32 [B,48], r f32 [B,48]; device, nullable */
int a3d_dcnf_infer(a3d_dcnf*, const float* images, float* output, float* z, float* r, void* stream);
/* device pointers into the net: CRF MAP estimate y* = A^-1 z [B,48], per-graph Cholesky status, the loss scalar */
int a3d_dcnf_state(a3d_dcnf*, const float** ystar, const int32_t** status, const float** loss);

/* ---- FP8 inference (E4M3 operands, tcgen05.mma kind::f8f6f4, f32 accumulation) -------------------------------------
 * The MSDN forward (src/models.py:208-253) with every convolution and dense product on E4M3 codes.  Numerics:
 *   quantiser   amax = max |x|, s = amax / 448, code = e4m3_rn_satfinite(x * (448 / amax)); amax == 0: s = 0, codes 0
 *   weights     one scale per output row of the operand matrix the kernels read (a3d_quantize_rows_e4m3 of the bf16
 *               mirror: [K][R][S][C] filters, [N][K] dense kernels) -- the TF variable's per-output-channel scale
 *   activations one scale per image (a3d_quantize_e4m3 / a3d_maxpool2x2_quantize_e4m3); the image itself has the fixed
 *               scale 2^-8 (a3d_resize_bilinear_tf1_s2d_e4m3)
 *   products    y[m][n] = act(acc[m][n] * x_scale[image(m)] * w_scale[n] + bias[n]), image(m) = m / (P*Q) for a
 *               convolution and m for a dense layer: an image's result never depends on its batch-mates
 * Every call is asynchronous on `stream` and capturable in a CUDA graph. */
/* Weight rows: q[r][0..cols) = codes of x[r*ldx + 0..cols) (bf16), scale[r].  cols % 8 == 0. */
int a3d_quantize_rows_e4m3(a3d_ctx*, const uint16_t* x, int rows, int cols, long long ldx, uint8_t* q, float* scale,
                           void* stream);
/* Per image: y[b][0..n) = codes of x[b][0..n) (bf16, n % 8 == 0), y_scale[b].  ws: a3d_quantize_ws_bytes_e4m3(B, n) bytes
 * (per-image partial maxima).  Replaces the bf16 storage of conv2d_2 / conv2d_3 / conv2d_4 / dense_0 outputs and of the
 * fine stack's concat (src/models.py:217-229, 246) as operands of the next layer. */
size_t a3d_quantize_ws_bytes_e4m3(int B, size_t n);
int a3d_quantize_e4m3(a3d_ctx*, const uint16_t* x, int B, size_t n, uint8_t* y, float* y_scale, void* ws, size_t ws_bytes,
                      void* stream);
/* 2x2/2 max-pool of x bf16 [B,H,W,C] quantised per image: y [B,H/2,W/2,ldy] (channels C..ldy-1 zero), y_scale[b];
 * src/models.py:212,215.  ws: a3d_quantize_ws_bytes_e4m3(B, (H/2)*(W/2)*ldy) bytes. */
int a3d_maxpool2x2_quantize_e4m3(a3d_ctx*, const uint16_t* x, int B, int H, int W, int C, uint8_t* y, int ldy,
                                 float* y_scale, void* ws, size_t ws_bytes, void* stream);
/* Resize (src/models.py:282) + space-to-depth(4) into E4M3 codes of 256 * value: dst [B,OH/4,OW/4,64] (channels 48..63
 * zero).  src_dtype A3D_F32 or A3D_U8 (pixel / 255), C == 3. */
int a3d_resize_bilinear_tf1_s2d_e4m3(a3d_ctx*, const void* src, int src_dtype, int B, int H, int W, int C, uint8_t* dst,
                                     int OH, int OW, int s, int dstC, void* stream);
/* Convolution forward (src/models.py:211-223, 247): x E4M3 NHWC (C % 64 == 0), w E4M3 [K][R][S][C]; y bf16 or f32
 * (y_dtype) [N,P,Q,ldy].  ws: a3d_conv2d_ws_bytes(.., A3D_OP_FWD) bytes enable split-K (nullable). */
int a3d_conv2d_fwd_fp8(a3d_ctx*, const a3d_conv_desc*, const uint8_t* x, const float* x_scale, const uint8_t* w,
                       const float* w_scale, const float* bias, void* y, int y_dtype, unsigned flags, void* ws,
                       size_t ws_bytes, void* stream);
/* conv + bias + act + 2x2 max-pool over the pool-embedded filter (as a3d_conv2d_pool4_fwd; src/models.py:241-245):
 * K = 256 = 4 window positions x 64 filters, y bf16 [N,P,Q,ldy] (64 pooled channels). */
int a3d_conv2d_pool4_fwd_fp8(a3d_ctx*, const a3d_conv_desc*, const uint8_t* x, const float* x_scale, const uint8_t* w,
                             const float* w_scale, const float* bias, uint16_t* y, unsigned flags, void* stream);
/* Dense forward (src/models.py:228, 231): y[M][N] = act(x[M][K] . w[N][K]^T * x_scale[m] * w_scale[n] + bias[n]), y bf16 or
 * f32; K % 128 == 0; acc_ws f32 [M][N]. */
int a3d_dense_fwd_fp8(a3d_ctx*, const uint8_t* x, int ldx, const float* x_scale, const uint8_t* w, const float* w_scale,
                      const float* bias, void* y, int y_dtype, float* acc_ws, int M, int N, int K, unsigned flags,
                      void* stream);

#ifdef __cplusplus
}
#endif
#endif /* A3D_H_ */

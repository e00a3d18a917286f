// conv.cu -- public convolution / dense entry points: argument checks and implementation dispatch
// (tcgen05 engine in tc_gemm.cu where the shape allows, CUDA-core kernels otherwise), plus the small
// helper kernels around them (filter flip for dgrad, col2im, single-filter convolution).
#include "common.cuh"
#include <stdlib.h>

int a3d_tc_conv_fwd(a3d_ctx*, const a3d_conv_desc*, const uint16_t* x, const uint16_t* w, const float* bias, void* y,
                    int y_dtype, unsigned flags, void* ws, size_t ws_bytes, cudaStream_t st, uint8_t* pool_idx = nullptr);
int a3d_tc_conv_wgrad_supported(const a3d_conv_desc* d);
int a3d_tc_conv_wgrad(a3d_ctx*, const a3d_conv_desc*, const uint16_t* x, const uint16_t* dy, float* dw, cudaStream_t st);
int a3d_tc_dgrad_cols(a3d_ctx*, const a3d_conv_desc*, const uint16_t* dy, const uint16_t* w, float* col, cudaStream_t st);
int a3d_tc_dense_fwd(a3d_ctx*, const uint16_t* x, int ldx, const uint16_t* w, const float* bias, const uint8_t* mask,
                     float drop_rate, void* y, int y_dtype, float* acc_ws, int M, int N, int K, unsigned flags,
                     cudaStream_t st);
struct a3d_actbwd_args { const uint16_t* y; const uint8_t* keep_mask; float drop_rate; unsigned flags; };
int a3d_tc_dense_dgrad(a3d_ctx*, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx, float* acc_ws, int M,
                       int N, int K, cudaStream_t st, const a3d_actbwd_args* ab = nullptr);
int a3d_tc_dense_dgrad_rows(a3d_ctx*, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx, int M, int N, int K,
                            cudaStream_t st);
int a3d_tc_dense_wgrad(a3d_ctx*, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* dw, int M, int N, int K,
                       cudaStream_t st);

int a3d_mma_dense_wgrad_adam(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* w, float* m,
                             float* v, uint16_t* wb, int M, int N, int K, float lr_t, float beta1, float beta2, float eps,
                             float grad_scale, const float* lr_t_dev, cudaStream_t st);

static size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

// overlapped-pixel view (a3d_conv_desc dil_w / pix_pitch): only the pool-fused forward and the weight gradient take it
static bool is_view(const a3d_conv_desc* d) { return d->dil_w > 1 || (d->pix_pitch && d->pix_pitch != d->C); }

static int check_desc(const a3d_conv_desc* d, bool allow_view = false) {
  A3D_REQUIRE(d, "conv: null descriptor");
  A3D_REQUIRE(d->dil_w >= 0 && d->pix_pitch >= 0, "conv: negative dil_w / pix_pitch");
  if (is_view(d)) {
    A3D_REQUIRE(allow_view, "conv: dil_w / pix_pitch views are taken by a3d_conv2d_pool4_fwd and a3d_conv2d_wgrad only");
    const int pp = d->pix_pitch ? d->pix_pitch : d->C, dil = d->dil_w > 1 ? d->dil_w : 1;
    A3D_REQUIRE(pp % 8 == 0 && pp <= d->C && d->C % pp == 0, "conv: pix_pitch must divide C and be a multiple of 8");
    A3D_REQUIRE(d->pad_l == 0 && (d->Q - 1) * d->stride_w + (d->S - 1) * dil < d->W,
                "conv: a dilated / overlapped view needs pad_l == 0 and every tap inside the row");
  }
  A3D_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0 && d->C > 0 && d->K > 0 && d->R > 0 && d->S > 0, "conv: bad dims");
  A3D_REQUIRE(d->stride_h > 0 && d->stride_w > 0 && d->pad_t >= 0 && d->pad_l >= 0, "conv: bad stride/pad");
  A3D_REQUIRE(d->P > 0 && d->Q > 0 && d->ldy >= d->K, "conv: bad output dims");
  // every tap of every output pixel must start inside the padded input
  A3D_REQUIRE((d->P - 1) * d->stride_h - d->pad_t < d->H && (d->Q - 1) * d->stride_w - d->pad_l < d->W,
              "conv: output larger than the input supports");
  return 0;
}

// A layer with fewer than 16 channels cannot feed the im2col TMA (>= 32 B per pixel for UMMA K = 16).
// If the horizontal stride is a multiple of g = 16/C pixels, g adjacent pixels can be read as ONE
// pixel of g*C channels of a [N, H, W/g, g*C] tensor: the filter [K,R,S,C] is then the same memory
// as [K,R,S/g,g*C] and the stride becomes stride_w/g.  (MSDN conv2d_0: 11x12x4 s4 -> 11x3x16 s1.)
// With stride_w only a multiple of 8/C pixels the group is 8 channels wide (MSDN fine/first:
// 9x10x4 s2 -> 9x5x8 s1), which the engine takes in its chunked no-swizzle mode.
static bool virtualize(const a3d_conv_desc* d, a3d_conv_desc* v) {
  if (d->C >= 16 || 16 % d->C) return false;
  for (int g = 16 / d->C; g * d->C >= 8 && g >= 2; g /= 2) {
    if (d->stride_w % g || d->W % g || d->S % g || d->pad_l != 0) continue;
    *v = *d;
    v->C = d->C * g; v->W = d->W / g; v->S = d->S / g; v->stride_w = d->stride_w / g;
    return true;
  }
  return false;
}

// dgrad of a stride-1 conv == forward conv of dy with the spatially flipped, channel-transposed filter
static bool dgrad_as_fwd_ok(const a3d_conv_desc* d) {
  return d->stride_h == 1 && d->stride_w == 1 && d->ldy == d->K && d->K % 16 == 0 && d->C % 8 == 0 &&
         d->R - 1 - d->pad_t >= 0 && d->S - 1 - d->pad_l >= 0;
}
static bool dgrad_as_cols_ok(const a3d_conv_desc* d) {
  return d->K % 64 == 0 && (d->R * d->S * d->C) % 64 == 0 && d->ldy % 8 == 0 && d->C % 8 == 0;
}

__global__ void flip_filter_kernel(const uint16_t* __restrict__ w, uint16_t* __restrict__ wd, int K, int RS, int C) {
  // w[co][t][ci] -> wd[ci][RS-1-t][co]
  size_t total = (size_t)K * RS * C;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int co = (int)(i % K);
    size_t t2 = i / K;
    int tf = (int)(t2 % RS);
    int ci = (int)(t2 / RS);
    wd[i] = w[((size_t)co * RS + (RS - 1 - tf)) * C + ci];
  }
}

// dx[n,ih,iw,c8] = sum over taps (r,s) with (ih+pt-r) % sh == 0 ... of col[(n,p,q)][(r,s,c8)]
__global__ void col2im_kernel(const float* __restrict__ col, uint16_t* __restrict__ dx, int N, int H, int W, int C, int R,
                              int S, int sh, int sw, int pt, int pl, int P, int Q) {
  const int C8 = C / 8;
  const size_t J = (size_t)R * S * C;
  size_t total = (size_t)N * H * W * C8;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int n, ih, iw, c8;
    split_nhwc(i, H, W, C8, n, ih, iw, c8);
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int r = 0; r < R; ++r) {
      int ph = ih + pt - r;
      if (ph < 0 || ph % sh) continue;
      int p = ph / sh;
      if (p >= P) continue;
      for (int s = 0; s < S; ++s) {
        int qw = iw + pl - s;
        if (qw < 0 || qw % sw) continue;
        int q = qw / sw;
        if (q >= Q) continue;
        const float4* src =
            reinterpret_cast<const float4*>(col + (((size_t)n * P + p) * Q + q) * J + (size_t)(r * S + s) * C + c8 * 8);
        float4 a = __ldg(src), b = __ldg(src + 1);
        acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
        acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
      }
    }
    uint4 o = make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]), pack_bf16x2(acc[4], acc[5]),
                         pack_bf16x2(acc[6], acc[7]));
    reinterpret_cast<uint4*>(dx)[i] = o;
  }
}

// Single-filter convolution (K == 1, C % 64 == 0): one warp per output pixel, lanes split the channels
// (coalesced 128 B per tap), warp-shuffle reduction.  HBM/L2-bound; used for MSDN fine/third
// (src/models.py:250: 5x5x64 -> 1) where a 128-row tensor-core tile would be 127/128 padding.
__global__ void conv_k1_fwd_kernel(const uint16_t* __restrict__ x, const uint16_t* __restrict__ w,
                                   const float* __restrict__ bias, void* __restrict__ y, int y_f32, int N, int H, int W,
                                   int C, int R, int S, int sh, int sw, int pt, int pl, int P, int Q, int ldy,
                                   unsigned flags) {
  extern __shared__ float wsm[];           // R*S*C filter as f32
  for (int i = threadIdx.x; i < R * S * C; i += blockDim.x) wsm[i] = bf16_bits_to_f32(w[i]);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  const long long total = (long long)N * P * Q;
  for (long long m = (long long)blockIdx.x * warps_per_block + (threadIdx.x >> 5); m < total;
       m += (long long)gridDim.x * warps_per_block) {
    int q = (int)(m % Q);
    long long t = m / Q;
    int p = (int)(t % P);
    int n = (int)(t / P);
    float acc = 0.f;
    for (int r = 0; r < R; ++r) {
      int ih = p * sh - pt + r;
      if (ih < 0 || ih >= H) continue;
      for (int s = 0; s < S; ++s) {
        int iw = q * sw - pl + s;
        if (iw < 0 || iw >= W) continue;
        const uint16_t* px = x + (((size_t)n * H + ih) * W + iw) * C;
        const float* wf = wsm + (r * S + s) * C;
        for (int c = lane * 2; c < C; c += 64) {
          uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(px + c));
          acc = fmaf(__uint_as_float(v << 16), wf[c], acc);
          acc = fmaf(__uint_as_float(v & 0xffff0000u), wf[c + 1], acc);
        }
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      if (bias) acc += bias[0];
      if (flags & A3D_EPI_RELU) acc = fmaxf(acc, 0.f);
      if (y_f32) reinterpret_cast<float*>(y)[(size_t)m * ldy] = acc;
      else reinterpret_cast<uint16_t*>(y)[(size_t)m * ldy] = f32_to_bf16_bits(acc);
    }
  }
}

static size_t filt_bytes(const a3d_conv_desc* d) { return ((size_t)d->K * d->R * d->S * d->C * 2 + 255) & ~(size_t)255; }

// split-K (and with it the f32 accumulation buffer) is only chosen when the output has far fewer
// 128x128 tiles than the GPU has SMs (tc_gemm.cu pick_splits)
static size_t splitk_bytes(a3d_ctx* ctx, long long rows, int cols) {
  long long tiles = ((rows + 127) / 128) * ((cols + 127) / 128);
  int sms = ctx ? ctx->sm_count : 148;
  return tiles >= sms * 3 / 4 ? 0 : (size_t)rows * cols * sizeof(float);
}

extern "C" size_t a3d_conv2d_ws_bytes(a3d_ctx* ctx, const a3d_conv_desc* d, int op) {
  if (!d) return 0;
  if (op == A3D_OP_FWD) return splitk_bytes(ctx, (long long)d->N * d->P * d->Q, d->K);
  if (op == A3D_OP_DGRAD) {
    if (dgrad_as_fwd_ok(d)) return filt_bytes(d) + splitk_bytes(ctx, (long long)d->N * d->H * d->W, d->C);
    if (dgrad_as_cols_ok(d)) return (size_t)d->N * d->P * d->Q * d->R * d->S * d->C * sizeof(float);
    return 0;
  }
  return 0;
}

extern "C" int a3d_conv2d_fwd(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* x, const uint16_t* w,
                              const float* bias, void* y, int y_dtype, unsigned flags, void* ws, size_t ws_bytes,
                              void* stream) {
  A3D_REQUIRE(ctx && x && w && y, "conv fwd: null argument");
  int rc = check_desc(d);
  if (rc) return rc;
  cudaStream_t st = as_stream(stream);
  if (d->impl == A3D_IMPL_SIMT) return a3d_simt_conv_fwd(ctx, d, x, w, bias, y, y_dtype, flags, st);
  // single-filter 64-channel convolution (MSDN fine/third): tap products on mma.sync + stencil sum reads the
  // input once; as a BN = 16 tcgen05 GEMM the im2col operand traffic is 25x redundant (49 us vs the input's 17 MB).
  if (d->impl == A3D_IMPL_AUTO && a3d_conv_k1_tiled_ok(d)) return a3d_conv_k1_tiled(ctx, d, x, w, bias, y, y_dtype, flags, st);
  a3d_conv_desc v;
  const a3d_conv_desc* e = virtualize(d, &v) ? &v : d;
  if (a3d_tc_conv_fwd_supported(e)) return a3d_tc_conv_fwd(ctx, e, x, w, bias, y, y_dtype, flags, ws, ws_bytes, st);
  if (d->K == 1 && d->C % 64 == 0 && d->impl == A3D_IMPL_AUTO && (size_t)d->R * d->S * d->C * 4 <= 48 * 1024) {
    long long pixels = (long long)d->N * d->P * d->Q;
    int block = 256, grid = (int)((pixels + 7) / 8);
    if (grid > ctx->sm_count * 8) grid = ctx->sm_count * 8;
    conv_k1_fwd_kernel<<<grid, block, (size_t)d->R * d->S * d->C * 4, st>>>(
        x, w, bias, y, y_dtype == A3D_F32, d->N, d->H, d->W, d->C, d->R, d->S, d->stride_h, d->stride_w, d->pad_t,
        d->pad_l, d->P, d->Q, d->ldy, flags);
    A3D_LAUNCH_OK(ctx);
    return 0;
  }
  if (d->impl == A3D_IMPL_TC) {
    a3d_set_error("conv fwd: shape not supported by the tcgen05 path (C=%d K=%d)", d->C, d->K);
    return A3D_ENOTSUP;
  }
  return a3d_simt_conv_fwd(ctx, d, x, w, bias, y, y_dtype, flags, st);
}

static int dgrad_impl(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* dy, const uint16_t* w, uint16_t* dx,
                      const uint16_t* relu_src, bool* relu_done, void* ws, size_t ws_bytes, cudaStream_t st,
                      const uint16_t* wflip = nullptr);

static int launch_flip(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* w, uint16_t* wd, cudaStream_t st) {
  size_t total = (size_t)d->K * d->R * d->S * d->C;
  int grid = (int)((total + 255) / 256);
  if (grid > ctx->sm_count * 8) grid = ctx->sm_count * 8;
  flip_filter_kernel<<<grid, 256, 0, st>>>(w, wd, d->K, d->R * d->S, d->C);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// The dgrad of a stride-1 convolution runs as a forward convolution of dY with the spatially flipped,
// channel-transposed filter.  The flip depends only on the weights, so a training loop can take it off the
// backward critical path: prepare it (on any stream) once the weights of the step are final, then call
// a3d_conv2d_dgrad_prepared.  Returns A3D_ENOTSUP when this shape's dgrad does not use a flipped filter.
extern "C" int a3d_conv2d_dgrad_prepare(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* w, uint16_t* wflip,
                                        void* stream) {
  A3D_REQUIRE(ctx && w && wflip, "conv dgrad prepare: null argument");
  int rc = check_desc(d);
  if (rc) return rc;
  if (d->impl == A3D_IMPL_SIMT || !dgrad_as_fwd_ok(d)) {
    a3d_set_error("conv dgrad prepare: this shape's dgrad does not use a flipped filter");
    return A3D_ENOTSUP;
  }
  return launch_flip(ctx, d, w, wflip, as_stream(stream));
}

extern "C" int a3d_conv2d_dgrad_prepared(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* dy, const uint16_t* wflip,
                                         uint16_t* dx, const uint16_t* relu_src, void* ws, size_t ws_bytes,
                                         void* stream) {
  A3D_REQUIRE(ctx && dy && wflip && dx, "conv dgrad (prepared): null argument");
  int rc = check_desc(d);
  if (rc) return rc;
  A3D_REQUIRE(d->impl != A3D_IMPL_SIMT && dgrad_as_fwd_ok(d), "conv dgrad (prepared): shape has no flipped-filter dgrad");
  cudaStream_t st = as_stream(stream);
  bool relu_done = false;
  rc = dgrad_impl(ctx, d, dy, nullptr, dx, relu_src, &relu_done, ws, ws_bytes, st, wflip);
  if (rc) return rc;
  if (relu_src && !relu_done) {
    A3D_REQUIRE(d->C % 8 == 0, "conv dgrad: fused ReluGrad needs C %% 8 == 0");
    return a3d_relu_bwd(ctx, relu_src, dx, d->C, dx, (size_t)d->N * d->H * d->W, d->C, st);     // in place
  }
  return 0;
}

extern "C" int a3d_conv2d_dgrad(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* dy, const uint16_t* w,
                                uint16_t* dx, const uint16_t* relu_src, void* ws, size_t ws_bytes, void* stream) {
  A3D_REQUIRE(ctx && dy && w && dx, "conv dgrad: null argument");
  int rc = check_desc(d);
  if (rc) return rc;
  cudaStream_t st = as_stream(stream);
  bool relu_done = false;
  rc = dgrad_impl(ctx, d, dy, w, dx, relu_src, &relu_done, ws, ws_bytes, st);
  if (rc) return rc;
  if (relu_src && !relu_done) {
    A3D_REQUIRE(d->C % 8 == 0, "conv dgrad: fused ReluGrad needs C %% 8 == 0");
    return a3d_relu_bwd(ctx, relu_src, dx, d->C, dx, (size_t)d->N * d->H * d->W, d->C, st);     // in place
  }
  return 0;
}

static int dgrad_impl(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* dy, const uint16_t* w, uint16_t* dx,
                      const uint16_t* relu_src, bool* relu_done, void* ws, size_t ws_bytes, cudaStream_t st,
                      const uint16_t* wflip) {
  int rc = 0;
  const size_t filt = filt_bytes(d);
  if (wflip) {                                   // filter already flipped by a3d_conv2d_dgrad_prepare
    a3d_conv_desc e = *d;
    e.H = d->P; e.W = d->Q; e.C = d->K;          // "input" is dy
    e.K = d->C; e.P = d->H; e.Q = d->W; e.ldy = d->C;
    e.pad_t = d->R - 1 - d->pad_t; e.pad_l = d->S - 1 - d->pad_l;
    e.stride_h = e.stride_w = 1;
    return a3d_tc_conv_fwd(ctx, &e, dy, wflip, nullptr, dx, A3D_BF16, 0, ws, ws_bytes, st);
  }
  if (d->impl != A3D_IMPL_SIMT && dgrad_as_fwd_ok(d) && ws && ws_bytes >= filt) {
    uint16_t* wd = reinterpret_cast<uint16_t*>(ws);
    rc = launch_flip(ctx, d, w, wd, st);
    if (rc) return rc;
    a3d_conv_desc e = *d;
    e.H = d->P; e.W = d->Q; e.C = d->K;          // "input" is dy
    e.K = d->C; e.P = d->H; e.Q = d->W; e.ldy = d->C;
    e.pad_t = d->R - 1 - d->pad_t; e.pad_l = d->S - 1 - d->pad_l;
    e.stride_h = e.stride_w = 1;
    return a3d_tc_conv_fwd(ctx, &e, dy, wd, nullptr, dx, A3D_BF16, 0, reinterpret_cast<uint8_t*>(ws) + filt,
                           ws_bytes - filt, st);
  }
  const size_t col_bytes = (size_t)d->N * d->P * d->Q * d->R * d->S * d->C * sizeof(float);
  if (d->impl != A3D_IMPL_SIMT && dgrad_as_cols_ok(d) && ws && ws_bytes >= col_bytes) {
    // strided conv: GEMM into per-output-pixel columns, then gather them back (col2im)
    float* col = reinterpret_cast<float*>(ws);
    rc = a3d_tc_dgrad_cols(ctx, d, dy, w, col, st);
    if (rc) return rc;
    size_t total = (size_t)d->N * d->H * d->W * (d->C / 8);
    int grid = (int)((total + 255) / 256);
    if (grid > ctx->sm_count * 16) grid = ctx->sm_count * 16;
    col2im_kernel<<<grid, 256, 0, st>>>(col, dx, d->N, d->H, d->W, d->C, d->R, d->S, d->stride_h, d->stride_w, d->pad_t,
                                       d->pad_l, d->P, d->Q);
    A3D_LAUNCH_OK(ctx);
    return 0;
  }
  if (d->impl == A3D_IMPL_TC) {
    a3d_set_error("conv dgrad: shape not supported by the tcgen05 path (stride %d, K=%d, ws=%zu)", d->stride_h, d->K,
                  ws_bytes);
    return A3D_ENOTSUP;
  }
  return a3d_simt_conv_dgrad(ctx, d, dy, w, dx, st);
}

extern "C" int a3d_conv2d_wgrad(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* x, const uint16_t* dy, float* dw,
                                float* db, void* ws, size_t ws_bytes, void* stream) {
  A3D_REQUIRE(ctx && x && dy && dw, "conv wgrad: null argument");
  int rc = check_desc(d, true);
  if (rc) return rc;
  cudaStream_t st = as_stream(stream);
  if (db) {
    rc = a3d_colsum_bf16(ctx, dy, (size_t)d->N * d->P * d->Q, d->K, d->ldy, db, st);
    if (rc) return rc;
  }
  if (d->impl != A3D_IMPL_SIMT) {
    a3d_conv_desc v;
    const a3d_conv_desc* e = (!is_view(d) && virtualize(d, &v)) ? &v : d;
    if (a3d_tc_conv_wgrad_supported(e)) return a3d_tc_conv_wgrad(ctx, e, x, dy, dw, st);
    if (d->impl == A3D_IMPL_TC) {
      a3d_set_error("conv wgrad: shape not supported by the tcgen05 path (C=%d ldy=%d)", d->C, d->ldy);
      return A3D_ENOTSUP;
    }
  }
  return a3d_simt_conv_wgrad(ctx, d, x, dy, dw, st);
}

// ------------------------------------------------------------------------------------------ dense
extern "C" int a3d_dense_fwd(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* w, const float* bias,
                             const uint8_t* keep_mask, float drop_rate, void* y, int y_dtype, float* acc_ws, int M,
                             int N, int K, unsigned flags, int impl, void* stream) {
  A3D_REQUIRE(ctx && x && w && y && M > 0 && N > 0 && K > 0 && ldx >= K, "dense fwd: bad argument");
  cudaStream_t st = as_stream(stream);
  bool tc_ok = (K % 64 == 0) && (ldx % 8 == 0) && acc_ws;
  if (impl != A3D_IMPL_SIMT && tc_ok) {
    // the batch is the UMMA N dimension (<= 256): larger batches (inference sweep, bs 512) go in chunks of 256 rows
    const size_t ysz = y_dtype == A3D_F32 ? 4 : 2;
    for (int m0 = 0; m0 < M; m0 += 256) {
      const int mc = M - m0 < 256 ? M - m0 : 256;
      int rc = a3d_tc_dense_fwd(ctx, x + (size_t)m0 * ldx, ldx, w, bias, keep_mask ? keep_mask + (size_t)m0 * N : nullptr,
                                drop_rate, reinterpret_cast<uint8_t*>(y) + (size_t)m0 * N * ysz, y_dtype,
                                acc_ws + (size_t)m0 * N, mc, N, K, flags, st);
      if (rc) return rc;
    }
    return 0;
  }
  if (impl == A3D_IMPL_TC) {
    a3d_set_error("dense fwd: shape not supported by the tcgen05 path (M=%d N=%d K=%d)", M, N, K);
    return A3D_ENOTSUP;
  }
  return a3d_simt_dense_fwd(ctx, x, ldx, w, bias, keep_mask, drop_rate, y, y_dtype, M, N, K, flags, st);
}

extern "C" int a3d_dense_dgrad(a3d_ctx* ctx, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx,
                               float* acc_ws, int M, int N, int K, int impl, void* stream) {
  A3D_REQUIRE(ctx && dy && w && dx && M > 0 && N > 0 && K > 0 && lddy >= N, "dense dgrad: bad argument");
  cudaStream_t st = as_stream(stream);
  bool tc_ok = (K % 8 == 0) && (lddy % 8 == 0) && M <= 128 && acc_ws;
  if (impl != A3D_IMPL_SIMT && tc_ok) return a3d_tc_dense_dgrad(ctx, dy, lddy, w, dx, acc_ws, M, N, K, st);
  if (impl != A3D_IMPL_SIMT && M > 128 && N % 64 == 0 && K % 64 == 0 && lddy % 8 == 0)
    return a3d_tc_dense_dgrad_rows(ctx, dy, lddy, w, dx, M, N, K, st);       // long batch (DCNF patches)
  if (impl == A3D_IMPL_TC) {
    a3d_set_error("dense dgrad: shape not supported by the tcgen05 path (M=%d N=%d K=%d lddy=%d)", M, N, K, lddy);
    return A3D_ENOTSUP;
  }
  return a3d_simt_dense_dgrad(ctx, dy, lddy, w, dx, M, N, K, st);
}

// dgrad + the activation gradient of the layer that produced x (y_act = its stored post-activation / post-dropout
// output [M,K]): dx = act'(y_act) * keep_mask/(1-rate) * (dy . w) in the dgrad's own finishing pass.
extern "C" int a3d_dense_dgrad_act(a3d_ctx* ctx, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx,
                                   float* acc_ws, int M, int N, int K, int impl, const uint16_t* y_act,
                                   const uint8_t* keep_mask, float drop_rate, unsigned flags, void* stream) {
  A3D_REQUIRE(ctx && dy && w && dx && y_act && M > 0 && N > 0 && K > 0 && lddy >= N, "dense dgrad+act: bad argument");
  cudaStream_t st = as_stream(stream);
  bool tc_ok = (K % 8 == 0) && (lddy % 8 == 0) && M <= 128 && acc_ws;
  if (impl != A3D_IMPL_SIMT && tc_ok) {
    a3d_actbwd_args ab{y_act, keep_mask, drop_rate, flags};
    return a3d_tc_dense_dgrad(ctx, dy, lddy, w, dx, acc_ws, M, N, K, st, &ab);
  }
  if (impl == A3D_IMPL_TC) {
    a3d_set_error("dense dgrad+act: shape not supported by the tcgen05 path (M=%d N=%d K=%d lddy=%d)", M, N, K, lddy);
    return A3D_ENOTSUP;
  }
  int rc = a3d_simt_dense_dgrad(ctx, dy, lddy, w, dx, M, N, K, st);
  if (rc) return rc;
  return a3d_dense_epilogue_bwd(ctx, dx, y_act, keep_mask, drop_rate, dx, (size_t)M * K, flags, stream);     // in place
}

extern "C" int a3d_dense_wgrad(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* dw,
                               float* db, int M, int N, int K, int impl, void* stream) {
  A3D_REQUIRE(ctx && x && dy && dw && M > 0 && N > 0 && K > 0 && lddy >= N && ldx >= K, "dense wgrad: bad argument");
  cudaStream_t st = as_stream(stream);
  if (db) {
    int rc = a3d_colsum_bf16(ctx, dy, (size_t)M, N, lddy, db, st);
    if (rc) return rc;
  }
  bool tc_ok = (K % 64 == 0) && (ldx % 8 == 0) && (lddy % 8 == 0);
  if (impl != A3D_IMPL_SIMT && tc_ok) return a3d_tc_dense_wgrad(ctx, x, ldx, dy, lddy, dw, M, N, K, st);
  if (impl == A3D_IMPL_TC) {
    a3d_set_error("dense wgrad: shape not supported by the tcgen05 path (M=%d N=%d K=%d)", M, N, K);
    return A3D_ENOTSUP;
  }
  return a3d_simt_dense_wgrad(ctx, x, ldx, dy, lddy, dw, M, N, K, st);
}

// Dense weight gradient fused with the TF-Adam update of that weight matrix: the 128 x 256 gradient tiles
// are consumed from TMEM by the optimizer (w, m, v updated in place, bf16 mirror refreshed) and never
// written to HBM.  Single-GPU only (a data-parallel step must allreduce the gradient first).
// db (nullable) still receives the bias gradient for a separate (tiny) a3d_adam_tf launch.
extern "C" int a3d_dense_wgrad_adam(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* db,
                                    float* w, float* m, float* v, uint16_t* w_bf16, int M, int N, int K, float lr_t,
                                    float beta1, float beta2, float eps, float grad_scale, const float* lr_t_dev,
                                    void* stream) {
  A3D_REQUIRE(ctx && x && dy && w && m && v && M > 0 && N > 0 && K > 0 && lddy >= N && ldx >= K,
              "dense wgrad+adam: bad argument");
  A3D_REQUIRE(K % 64 == 0 && ldx % 8 == 0 && lddy % 8 == 0, "dense wgrad+adam: needs K %% 64 == 0 and aligned row pitches");
  cudaStream_t st = as_stream(stream);
  if (db) {
    int rc = a3d_colsum_bf16(ctx, dy, (size_t)M, N, lddy, db, st);
    if (rc) return rc;
  }
  // The optimizer-shaped streaming kernel that forms the rank-M gradient with warp-level mma.sync (batch <= 32).  (Two
  // other forms were measured and removed: the 32 FMAs per parameter on the CUDA cores, 381 us, and a tcgen05 GEMM with
  // a TF-Adam epilogue, 535 us, against 277 us.)
  int rc = a3d_mma_dense_wgrad_adam(ctx, x, ldx, dy, lddy, w, m, v, w_bf16, M, N, K, lr_t, beta1, beta2, eps, grad_scale,
                                    lr_t_dev, st);
  if (rc == A3D_ENOTSUP)
    a3d_set_error("dense wgrad+adam: needs batch <= %d, K %% 256 == 0 and 16-byte aligned w/m/v (batch %d, K %d)",
                  A3D_DENSE_WGRAD_ADAM_MAX_M, M, K);
  return rc;
}

// Convolution + bias + activation + 2x2/2 max-pool in one tcgen05 GEMM.  The caller supplies the "pool-embedded"
// filter: for every pooled output pixel the four conv outputs of its window are four groups of Kc = 64 filters
// (K = 256, filter index g*64 + c, g = 2*a + b for window position (a, b)) over a common receptive field, so
// that the pool is a max over four accumulator columns of one GEMM row (tc::EPI_POOL4_BF16).
// y bf16 [N,P,Q,ldy] (64 channels), idx u8 [N,P,Q,64] (nullable): first arg-max group, for a3d_pool4_bwd.
__global__ void pool4_reduce_kernel(const float* __restrict__ acc, const float* __restrict__ bias, uint16_t* __restrict__ y,
                                    int ldy, uint8_t* __restrict__ idx, size_t rows, unsigned flags) {
  const size_t total = rows * 64;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t row = i >> 6;
    const int c = (int)(i & 63);
    const float* a = acc + row * 256 + c;
    float m = a[0];
    int g = 0;
    if (a[64] > m) { m = a[64]; g = 1; }
    if (a[128] > m) { m = a[128]; g = 2; }
    if (a[192] > m) { m = a[192]; g = 3; }
    if (bias) m += bias[c];
    if (flags & A3D_EPI_RELU) m = fmaxf(m, 0.f);
    y[row * ldy + c] = f32_to_bf16_bits(m);
    if (idx) idx[i] = (uint8_t)g;
  }
}

extern "C" int a3d_conv2d_pool4_fwd(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* x, const uint16_t* w,
                                    const float* bias, uint16_t* y, uint8_t* idx, unsigned flags, void* ws,
                                    size_t ws_bytes, void* stream) {
  A3D_REQUIRE(ctx && x && w && y && d, "conv pool4 fwd: null argument");
  A3D_REQUIRE(d->K == 256 && d->ldy >= 64, "conv pool4 fwd: K must be 4 x 64 and ldy >= 64");
  a3d_conv_desc chk = *d;
  chk.ldy = d->K;                      // ldy describes the POOLED output (64 channels), not the 256 GEMM columns
  int rc = check_desc(&chk, true);
  if (rc) return rc;
  cudaStream_t st = as_stream(stream);
  if (d->impl == A3D_IMPL_SIMT) {
    // CUDA-core cross-check: plain convolution into an f32 scratch [rows][256], then the group max
    const size_t rows = (size_t)d->N * d->P * d->Q;
    A3D_REQUIRE(ws && ws_bytes >= rows * 256 * sizeof(float), "conv pool4 fwd (simt): needs rows*256*4 bytes of scratch");
    a3d_conv_desc e = *d;
    e.ldy = 256;
    rc = a3d_simt_conv_fwd(ctx, &e, x, w, nullptr, ws, A3D_F32, 0, st);
    if (rc) return rc;
    size_t total = rows * 64;
    int grid = (int)((total + 255) / 256);
    if (grid > ctx->sm_count * 16) grid = ctx->sm_count * 16;
    pool4_reduce_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const float*>(ws), bias, y, d->ldy, idx, rows, flags);
    A3D_LAUNCH_OK(ctx);
    return 0;
  }
  return a3d_tc_conv_fwd(ctx, d, x, w, bias, y, A3D_BF16, (flags & (A3D_EPI_RELU)) | A3D_EPI_POOL4, nullptr, 0, st, idx);
}

// elementwise.cu -- the HBM-bound kernels of the MSDN/DCNF step: bilinear resize, 2x2 max-pool
// (fwd / bwd fused with ReLU-grad), scale-invariant log loss (+grad), TF-Adam / SGD, casts.
// All are coalesced, 128-bit vectorised where the layout allows, and sized as grid-stride loops
// over a multiple of the SM count.
#include "common.cuh"

static inline int grid_for(a3d_ctx* ctx, size_t work_items, int block, int max_waves = 8) {
  size_t blocks = (work_items + block - 1) / block;
  size_t cap = (size_t)ctx->sm_count * max_waves * (2048 / block);
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// ------------------------------------------------------------------------------------ resize
// TF1 legacy bilinear (tf1_coord / tf1_lerp, common.cuh).  One thread per output pixel; the <= 4 channels of a pixel are adjacent so a warp reads a
// contiguous strip of each of the two source rows.
template <bool OUT_BF16>
__global__ void resize_bilinear_tf1_kernel(const float* __restrict__ src, int B, int H, int W, int C,
                                           void* __restrict__ dst, int OH, int OW, int dstC, float sy, float sx) {
  size_t total = (size_t)B * OH * OW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int ox = (int)(i % OW);
    size_t t = i / OW;
    int oy = (int)(t % OH);
    int b = (int)(t / OH);
    int y0, y1, x0, x1;
    float ly, lx;
    tf1_coord(oy, sy, H, y0, y1, ly);
    tf1_coord(ox, sx, W, x0, x1, lx);
    const float* r0 = src + ((size_t)b * H + y0) * W * C;
    const float* r1 = src + ((size_t)b * H + y1) * W * C;
    for (int c = 0; c < dstC; ++c) {
      float v = 0.f;
      if (c < C) {
        float tl = __ldg(r0 + (size_t)x0 * C + c), tr = __ldg(r0 + (size_t)x1 * C + c);
        float bl = __ldg(r1 + (size_t)x0 * C + c), br = __ldg(r1 + (size_t)x1 * C + c);
        v = tf1_lerp(tl, tr, bl, br, ly, lx);
      }
      if (OUT_BF16) reinterpret_cast<uint16_t*>(dst)[i * dstC + c] = f32_to_bf16_bits(v);
      else reinterpret_cast<float*>(dst)[i * dstC + c] = v;
    }
  }
}

extern "C" int a3d_resize_bilinear_tf1(a3d_ctx* ctx, const float* src, int B, int H, int W, int C, void* dst,
                                       int OH, int OW, int dstC, int dst_dtype, void* stream) {
  A3D_REQUIRE(ctx && src && dst, "resize: null argument");
  A3D_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0 && OH > 0 && OW > 0 && dstC >= C, "resize: bad shape");
  size_t total = (size_t)B * OH * OW;
  int block = 256, grid = grid_for(ctx, total, block);
  // the scale is formed in float like TF's CalculateResizeScale (in/out as float division)
  float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  if (dst_dtype == A3D_BF16)
    resize_bilinear_tf1_kernel<true><<<grid, block, 0, as_stream(stream)>>>(src, B, H, W, C, dst, OH, OW, dstC, sy, sx);
  else
    resize_bilinear_tf1_kernel<false><<<grid, block, 0, as_stream(stream)>>>(src, B, H, W, C, dst, OH, OW, dstC, sy, sx);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ max-pool
__device__ __forceinline__ uint4 max_bf16x8(uint4 a, uint4 b) {
  uint4 r;
  __nv_bfloat162* ra = reinterpret_cast<__nv_bfloat162*>(&a);
  __nv_bfloat162* rb = reinterpret_cast<__nv_bfloat162*>(&b);
  __nv_bfloat162* rr = reinterpret_cast<__nv_bfloat162*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) rr[i] = __hmax2(ra[i], rb[i]);
  return r;
}

// one thread = one output pixel x 8 channels (16 B loads/stores)
__global__ void maxpool2x2_fwd_kernel(const uint4* __restrict__ x, int N, int H, int W, int C8, uint4* __restrict__ y,
                                      int ldy8) {
  int OH = H / 2, OW = W / 2;
  size_t total = (size_t)N * OH * OW * C8;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int n, oh, ow, c;
    split_nhwc(i, OH, OW, C8, n, oh, ow, c);
    const uint4* p = x + (((size_t)n * H + 2 * oh) * W + 2 * ow) * C8 + c;
    uint4 a = __ldg(p), b = __ldg(p + C8), d = __ldg(p + (size_t)W * C8), e = __ldg(p + (size_t)W * C8 + C8);
    y[(((size_t)n * OH + oh) * OW + ow) * ldy8 + c] = max_bf16x8(max_bf16x8(a, b), max_bf16x8(d, e));
  }
}

extern "C" int a3d_maxpool2x2_fwd(a3d_ctx* ctx, const uint16_t* x, int N, int H, int W, int C, uint16_t* y, int ldy,
                                  void* stream) {
  A3D_REQUIRE(ctx && x && y, "maxpool: null argument");
  A3D_REQUIRE(C % 8 == 0 && ldy % 8 == 0 && ldy >= C && H >= 2 && W >= 2, "maxpool: C and ldy must be multiples of 8");
  size_t total = (size_t)N * (H / 2) * (W / 2) * (C / 8);
  int block = 256, grid = grid_for(ctx, total, block);
  maxpool2x2_fwd_kernel<<<grid, block, 0, as_stream(stream)>>>(reinterpret_cast<const uint4*>(x), N, H, W, C / 8,
                                                             reinterpret_cast<uint4*>(y), ldy / 8);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// one thread = one 2x2 window (or an uncovered edge cell group) x 8 channels.
// Gradient goes to the FIRST arg-max in (0,0),(0,1),(1,0),(1,1) order and only where x > 0 (ReLU).
__global__ void maxpool2x2_relu_bwd_kernel(const uint4* __restrict__ x, const uint4* __restrict__ dy, int lddy8, int N,
                                           int H, int W, int C8, uint4* __restrict__ dx) {
  int OH = H / 2, OW = W / 2;
  int GH = (H + 1) / 2, GW = (W + 1) / 2;   // windows incl. the partial ones on the odd edge
  size_t total = (size_t)N * GH * GW * C8;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int n, gh, gw, c;
    split_nhwc(i, GH, GW, C8, n, gh, gw, c);
    int h0 = 2 * gh, w0 = 2 * gw;
    bool covered = (gh < OH) && (gw < OW);
    size_t base = (((size_t)n * H + h0) * W + w0) * C8 + c;
    uint4 zero = make_uint4(0, 0, 0, 0);
    if (!covered) {
      dx[base] = zero;
      if (w0 + 1 < W) dx[base + C8] = zero;
      if (h0 + 1 < H) {
        dx[base + (size_t)W * C8] = zero;
        if (w0 + 1 < W) dx[base + (size_t)W * C8 + C8] = zero;
      }
      continue;
    }
    uint4 xv[4] = {__ldg(x + base), __ldg(x + base + C8), __ldg(x + base + (size_t)W * C8),
                   __ldg(x + base + (size_t)W * C8 + C8)};
    uint4 g = __ldg(dy + (((size_t)n * OH + gh) * OW + gw) * lddy8 + c);
    uint4 out[4];
    const uint16_t* gv = reinterpret_cast<const uint16_t*>(&g);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = bf16_bits_to_f32(reinterpret_cast<const uint16_t*>(&xv[k])[e]);
      int arg = 0;
      float m = v[0];
#pragma unroll
      for (int k = 1; k < 4; ++k)
        if (v[k] > m) { m = v[k]; arg = k; }
      uint16_t gg = (m > 0.f) ? gv[e] : (uint16_t)0;
#pragma unroll
      for (int k = 0; k < 4; ++k) reinterpret_cast<uint16_t*>(&out[k])[e] = (k == arg) ? gg : (uint16_t)0;
    }
    dx[base] = out[0];
    dx[base + C8] = out[1];
    dx[base + (size_t)W * C8] = out[2];
    dx[base + (size_t)W * C8 + C8] = out[3];
  }
}

extern "C" int a3d_maxpool2x2_relu_bwd(a3d_ctx* ctx, const uint16_t* x, const uint16_t* dy, int lddy, int N, int H,
                                       int W, int C, uint16_t* dx, void* stream) {
  A3D_REQUIRE(ctx && x && dy && dx, "maxpool_bwd: null argument");
  A3D_REQUIRE(C % 8 == 0 && lddy % 8 == 0 && lddy >= C, "maxpool_bwd: C and lddy must be multiples of 8");
  size_t total = (size_t)N * ((H + 1) / 2) * ((W + 1) / 2) * (C / 8);
  int block = 256, grid = grid_for(ctx, total, block);
  maxpool2x2_relu_bwd_kernel<<<grid, block, 0, as_stream(stream)>>>(
      reinterpret_cast<const uint4*>(x), reinterpret_cast<const uint4*>(dy), lddy / 8, N, H, W, C / 8,
      reinterpret_cast<uint4*>(dx));
  A3D_LAUNCH_OK(ctx);
  return 0;
}

__global__ void relu_bwd_kernel(const uint4* __restrict__ y, const uint4* __restrict__ dy, int lddy8, uint4* __restrict__ dx,
                                size_t rows, int C8) {
  size_t total = rows * C8;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    size_t r; int c;
    split_rc(i, C8, r, c);
    uint4 yv = __ldg(y + i), g = __ldg(dy + r * lddy8 + c), o;
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float v = bf16_bits_to_f32(reinterpret_cast<const uint16_t*>(&yv)[e]);
      reinterpret_cast<uint16_t*>(&o)[e] = v > 0.f ? reinterpret_cast<const uint16_t*>(&g)[e] : (uint16_t)0;
    }
    dx[i] = o;
  }
}

extern "C" int a3d_relu_bwd(a3d_ctx* ctx, const uint16_t* y, const uint16_t* dy, int lddy, uint16_t* dx, size_t rows,
                            int C, void* stream) {
  A3D_REQUIRE(ctx && y && dy && dx, "relu_bwd: null argument");
  A3D_REQUIRE(C % 8 == 0 && lddy % 8 == 0, "relu_bwd: C and lddy must be multiples of 8");
  int block = 256, grid = grid_for(ctx, rows * (C / 8), block);
  relu_bwd_kernel<<<grid, block, 0, as_stream(stream)>>>(reinterpret_cast<const uint4*>(y),
                                                       reinterpret_cast<const uint4*>(dy), lddy / 8,
                                                       reinterpret_cast<uint4*>(dx), rows, C / 8);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

__global__ void dense_epilogue_bwd_kernel(const uint16_t* __restrict__ g_post, const uint16_t* __restrict__ y,
                                          const uint8_t* __restrict__ mask, float scale, uint16_t* __restrict__ g_pre,
                                          size_t n, unsigned flags) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float g = bf16_bits_to_f32(g_post[i]);
    if (mask) g = mask[i] ? g * scale : 0.f;
    float yv = bf16_bits_to_f32(y[i]);
    if (flags & A3D_EPI_RELU) g = yv > 0.f ? g : 0.f;
    if (flags & A3D_EPI_SIGMOID) g = g * yv * (1.f - yv);
    g_pre[i] = f32_to_bf16_bits(g);
  }
}

extern "C" int a3d_dense_epilogue_bwd(a3d_ctx* ctx, const uint16_t* g_post, const uint16_t* y, const uint8_t* keep_mask,
                                      float drop_rate, uint16_t* g_pre, size_t n, unsigned flags, void* stream) {
  A3D_REQUIRE(ctx && g_post && y && g_pre, "dense_epilogue_bwd: null argument");
  int block = 256, grid = grid_for(ctx, n, block);
  dense_epilogue_bwd_kernel<<<grid, block, 0, as_stream(stream)>>>(g_post, y, keep_mask, 1.f / (1.f - drop_rate), g_pre,
                                                                 n, flags);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ loss
// One CTA per sample.  Pass 1: d_i = nan0(log(out+eps)) - nan0(log(tar+eps)), block-reduce sum d and
// sum d^2 with warp shuffles.  Pass 2: gradient (2 d_i - 2*lon*sum d) / (out_i+eps) / B, 0 on the NaN branch.
__global__ void silog_loss_kernel(const float* __restrict__ out, const float* __restrict__ tar, int n, int B,
                                  float lambda_over_n, float* __restrict__ loss_ps, float* __restrict__ dout_f32,
                                  uint16_t* __restrict__ dout_bf16, int ld) {
  extern __shared__ float sd[];          // n floats: cached d_i
  __shared__ float red[2][32];
  const float eps = 1e-8f;
  int b = blockIdx.x;
  const float* o = out + (size_t)b * n;
  const float* t = tar + (size_t)b * n;
  float s1 = 0.f, s2 = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float lo = logf(o[i] + eps);
    lo = isnan(lo) ? 0.f : lo;
    float lt = logf(t[i] + eps);
    lt = isnan(lt) ? 0.f : lt;
    float d = lo - lt;
    sd[i] = d;
    s1 += d;
    s2 += d * d;
  }
  s1 = warp_sum(s1);
  s2 = warp_sum(s2);
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if (lane == 0) { red[0][wid] = s1; red[1][wid] = s2; }
  __syncthreads();
  if (wid == 0) {
    s1 = lane < nw ? red[0][lane] : 0.f;
    s2 = lane < nw ? red[1][lane] : 0.f;
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    if (lane == 0) { red[0][0] = s1; red[1][0] = s2; }
  }
  __syncthreads();
  s1 = red[0][0];
  s2 = red[1][0];
  if (threadIdx.x == 0) loss_ps[b] = s2 - lambda_over_n * s1 * s1;
  if (dout_f32 || dout_bf16) {
    float invB = 1.f / (float)B;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
      float arg = o[i] + eps;
      float g = 0.f;
      if (!isnan(logf(arg))) g = (2.f * sd[i] - 2.f * lambda_over_n * s1) / arg * invB;
      if (dout_f32) dout_f32[(size_t)b * ld + i] = g;
      if (dout_bf16) dout_bf16[(size_t)b * ld + i] = f32_to_bf16_bits(g);
    }
  }
}

__global__ void mean_kernel(const float* __restrict__ v, int n, float* __restrict__ out) {
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += 32) s += v[i];
  s = warp_sum(s);
  if (threadIdx.x == 0) *out = s / (float)n;
}

extern "C" int a3d_silog_loss(a3d_ctx* ctx, const float* out, const float* tar, int B, int n, float lambda_over_n,
                              float* loss_per_sample, float* loss, float* dout_f32, uint16_t* dout_bf16, int dout_ld,
                              void* stream) {
  A3D_REQUIRE(ctx && out && tar && loss_per_sample && loss, "silog_loss: null argument");
  A3D_REQUIRE(B > 0 && n > 0 && (size_t)n * sizeof(float) <= 200 * 1024, "silog_loss: bad shape");
  size_t smem = (size_t)n * sizeof(float);
  if (smem > 48 * 1024)
    A3D_CHECK_CUDA(cudaFuncSetAttribute(silog_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (dout_ld <= 0) dout_ld = n;
  A3D_REQUIRE(dout_ld >= n, "silog_loss: dout_ld < n");
  silog_loss_kernel<<<B, 512, smem, as_stream(stream)>>>(out, tar, n, B, lambda_over_n, loss_per_sample, dout_f32,
                                                        dout_bf16, dout_ld);
  A3D_LAUNCH_OK(ctx);
  mean_kernel<<<1, 32, 0, as_stream(stream)>>>(loss_per_sample, B, loss);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ scale-and-shift-invariant loss
// The formula is stated in include/a3d.h (a3d_ssi_loss).  One CTA per image, p and g staged in shared memory.
// Pass 1: double moments + min/max of p, then the fit (s, t).  Pass 2: sum r^2, the weighted sum of |D| over the
// scales' pairs, and Q.  Pass 3: the gradient; each pixel gathers the signs of its own <= 4 pairs per scale.
// Residuals are recomputed from p and g wherever a pass needs one (three float32 roundings, so every thread
// that touches pixel j gets the same r_j).  Every reduction runs in a fixed order and there are no atomics.
constexpr int SSI_THREADS = 512;
constexpr int SSI_MAX_SCALES = 4;

// v[] summed over the block; every thread receives the totals.  The shuffle tree and the pass over the warp partials
// have a fixed order, so the result does not depend on scheduling.
template <int NV>
__device__ __forceinline__ void ssi_block_sum(double (&v)[NV], double (*red)[SSI_THREADS / 32]) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[j] += __shfl_xor_sync(0xffffffffu, v[j], o);
    if (lane == 0) red[j][wid] = v[j];
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    double s = 0.0;
    for (int w = 0; w < SSI_THREADS / 32; ++w) s += red[j][w];
    v[j] = s;
  }
  __syncthreads();
}

__device__ __forceinline__ float ssi_residual(float s, float t, float p, float g) {
  return __fsub_rn(__fadd_rn(__fmul_rn(s, p), t), g);          // no contraction into an FMA
}

__device__ __forceinline__ double ssi_sign(float d) { return d > 0.f ? 1.0 : (d < 0.f ? -1.0 : 0.0); }

__global__ void __launch_bounds__(SSI_THREADS, 1)
ssi_loss_kernel(const float* __restrict__ out, const float* __restrict__ tar, int H, int W, int B, float alpha,
                int scales, float* __restrict__ loss_ps, float* __restrict__ dout_f32, uint16_t* __restrict__ dout_bf16,
                int ld) {
  extern __shared__ float ssi_sm[];                       // p [n] | g [n]
  __shared__ double red[4][SSI_THREADS / 32];
  __shared__ float redf[2][SSI_THREADS / 32];
  const int n = H * W, b = blockIdx.x;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  float* sp = ssi_sm;
  float* sg = ssi_sm + n;
  const float* o = out + (size_t)b * n;
  const float* t = tar + (size_t)b * n;
  // pass 1: Sp, Sg, Spp, Spg and the range of p
  double m[4] = {0.0, 0.0, 0.0, 0.0};
  float mn = INFINITY, mx = -INFINITY;
  for (int i = threadIdx.x; i < n; i += SSI_THREADS) {
    const float p = o[i], g = t[i];
    sp[i] = p;
    sg[i] = g;
    const double pd = p, gd = g;
    m[0] += pd;
    m[1] += gd;
    m[2] += pd * pd;
    m[3] += pd * gd;
    mn = fminf(mn, p);
    mx = fmaxf(mx, p);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
  }
  if (lane == 0) { redf[0][wid] = mn; redf[1][wid] = mx; }
  ssi_block_sum(m, red);                                  // its barrier also publishes sp, sg and redf
  for (int w = 0; w < SSI_THREADS / 32; ++w) { mn = fminf(mn, redf[0][w]); mx = fmaxf(mx, redf[1][w]); }
  const double nd = (double)n, Sp = m[0], Sg = m[1];
  const double D = m[2] - Sp * Sp / nd, N = m[3] - Sp * Sg / nd;
  const bool flat = !(mn < mx) || !(D > 0.0);             // constant prediction: s = 0, t = mean g, gradient 0
  const double sd = flat ? 0.0 : N / D;
  const float s = (float)sd;
  const float tt = (float)(__dsub_rn(Sg, __dmul_rn(sd, Sp)) / nd);
  double inv_nk[SSI_MAX_SCALES];
#pragma unroll
  for (int k = 0; k < SSI_MAX_SCALES; ++k) {
    const int h = 1 << k;
    inv_nk[k] = 1.0 / ((double)((H + h - 1) >> k) * (double)((W + h - 1) >> k));
  }
  // pass 2: sum r^2, sum_k (1/n_k) sum |D|, Q
  double a[3] = {0.0, 0.0, 0.0};
  for (int i = threadIdx.x; i < n; i += SSI_THREADS) {
    const int y = i / W, x = i - y * W;
    const float ri = ssi_residual(s, tt, sp[i], sg[i]);
    a[0] += (double)ri * (double)ri;
#pragma unroll
    for (int k = 0; k < SSI_MAX_SCALES; ++k) {
      const int h = 1 << k;
      if (k >= scales || ((y | x) & (h - 1))) break;      // off grid k means off every coarser grid too
      if (x + h < W) {
        const float d = __fsub_rn(ri, ssi_residual(s, tt, sp[i + h], sg[i + h]));
        a[1] += inv_nk[k] * fabs((double)d);
        a[2] += inv_nk[k] * ssi_sign(d) * ((double)sp[i] - (double)sp[i + h]);
      }
      if (y + h < H) {
        const float d = __fsub_rn(ri, ssi_residual(s, tt, sp[i + h * W], sg[i + h * W]));
        a[1] += inv_nk[k] * fabs((double)d);
        a[2] += inv_nk[k] * ssi_sign(d) * ((double)sp[i] - (double)sp[i + h * W]);
      }
    }
  }
  ssi_block_sum(a, red);
  const double al = (double)alpha;
  if (threadIdx.x == 0) loss_ps[b] = (float)(a[0] / (2.0 * nd) + al * a[1]);
  if (!dout_f32 && !dout_bf16) return;
  // pass 3: dL/dp_i / B
  const double Q = a[2], mp = Sp / nd, mg = Sg / nd, sf = (double)s;
  for (int i = threadIdx.x; i < n; i += SSI_THREADS) {
    double gr = 0.0;
    if (!flat) {
      const int y = i / W, x = i - y * W;
      const float ri = ssi_residual(s, tt, sp[i], sg[i]);
      double c = 0.0;
#pragma unroll
      for (int k = 0; k < SSI_MAX_SCALES; ++k) {
        const int h = 1 << k;
        if (k >= scales || ((y | x) & (h - 1))) break;
        double ck = 0.0;                                  // i is the first point (a) of its right / lower pair ...
        if (x + h < W) ck += ssi_sign(__fsub_rn(ri, ssi_residual(s, tt, sp[i + h], sg[i + h])));
        if (y + h < H) ck += ssi_sign(__fsub_rn(ri, ssi_residual(s, tt, sp[i + h * W], sg[i + h * W])));
        if (x >= h) ck -= ssi_sign(__fsub_rn(ssi_residual(s, tt, sp[i - h], sg[i - h]), ri));   // ... the second (b)
        if (y >= h) ck -= ssi_sign(__fsub_rn(ssi_residual(s, tt, sp[i - h * W], sg[i - h * W]), ri));
        c += inv_nk[k] * ck;
      }
      const double ds = (((double)sg[i] - mg) - 2.0 * sd * ((double)sp[i] - mp)) / D;
      gr = (sf * (double)ri / nd + al * (sf * c + Q * ds)) / (double)B;
    }
    const float gv = (float)gr;
    if (dout_f32) dout_f32[(size_t)b * ld + i] = gv;
    if (dout_bf16) dout_bf16[(size_t)b * ld + i] = f32_to_bf16_bits(gv);
  }
}

extern "C" int a3d_ssi_loss(a3d_ctx* ctx, const float* out, const float* tar, int B, int H, int W, float alpha,
                            int scales, float* loss_per_sample, float* loss, float* dout_f32, uint16_t* dout_bf16,
                            int dout_ld, void* stream) {
  A3D_REQUIRE(ctx, "ssi_loss: null context");
  A3D_REQUIRE(out, "ssi_loss: out is null");
  A3D_REQUIRE(tar, "ssi_loss: tar is null");
  A3D_REQUIRE(loss_per_sample, "ssi_loss: loss_per_sample is null");
  A3D_REQUIRE(loss, "ssi_loss: loss is null");
  A3D_REQUIRE(B > 0 && H > 0 && W > 0, "ssi_loss: bad shape B=%d H=%d W=%d", B, H, W);
  const size_t n = (size_t)H * (size_t)W, smem = 2 * n * sizeof(float);
  A3D_REQUIRE(smem <= 200 * 1024, "ssi_loss: H*W = %zu exceeds the shared-memory bound of %d pixels", n,
              200 * 1024 / (int)(2 * sizeof(float)));
  if (dout_ld <= 0) dout_ld = (int)n;
  A3D_REQUIRE((size_t)dout_ld >= n, "ssi_loss: dout_ld = %d < H*W = %zu", dout_ld, n);
  A3D_REQUIRE(alpha >= 0.f, "ssi_loss: alpha = %g must be >= 0", (double)alpha);
  A3D_REQUIRE(scales >= 1 && scales <= SSI_MAX_SCALES, "ssi_loss: scales = %d outside 1..%d", scales, SSI_MAX_SCALES);
  if (smem > 48 * 1024)
    A3D_CHECK_CUDA(cudaFuncSetAttribute(ssi_loss_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  ssi_loss_kernel<<<B, SSI_THREADS, smem, as_stream(stream)>>>(out, tar, H, W, B, alpha, scales, loss_per_sample,
                                                              dout_f32, dout_bf16, dout_ld);
  A3D_LAUNCH_OK(ctx);
  mean_kernel<<<1, 32, 0, as_stream(stream)>>>(loss_per_sample, B, loss);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ optimizers
// TF1 ApplyAdam; one pass, 128-bit loads/stores: 16 B read + 12 B written per parameter (+2 B bf16 mirror).
__global__ void adam_tf_kernel(float4* __restrict__ w, const float4* __restrict__ g, float4* __restrict__ m,
                               float4* __restrict__ v, uint2* __restrict__ wb, size_t n4, float lr_t, float b1, float b2,
                               float eps, float gs, const float* __restrict__ lr_dev) {
  if (lr_dev) lr_t = __ldg(lr_dev);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 W = w[i], G = __ldg(g + i), M = m[i], V = v[i];
    float* pw = &W.x; float* pg = &G.x; float* pm = &M.x; float* pv = &V.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float gk = pg[k] * gs;
      pm[k] = b1 * pm[k] + (1.f - b1) * gk;
      pv[k] = b2 * pv[k] + (1.f - b2) * gk * gk;
      pw[k] = pw[k] - lr_t * pm[k] / (sqrtf(pv[k]) + eps);
    }
    w[i] = W; m[i] = M; v[i] = V;
    if (wb) wb[i] = make_uint2(pack_bf16x2(W.x, W.y), pack_bf16x2(W.z, W.w));
  }
}
__global__ void adam_tf_tail_kernel(float* w, const float* g, float* m, float* v, uint16_t* wb, size_t start, size_t n,
                                    float lr_t, float b1, float b2, float eps, float gs, const float* lr_dev) {
  if (lr_dev) lr_t = __ldg(lr_dev);
  size_t i = start + blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) {
    float gk = g[i] * gs;
    float mm = b1 * m[i] + (1.f - b1) * gk;
    float vv = b2 * v[i] + (1.f - b2) * gk * gk;
    float ww = w[i] - lr_t * mm / (sqrtf(vv) + eps);
    m[i] = mm; v[i] = vv; w[i] = ww;
    if (wb) wb[i] = f32_to_bf16_bits(ww);
  }
}

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

extern "C" int a3d_adam_tf(a3d_ctx* ctx, float* w, const float* g, float* m, float* v, uint16_t* w_bf16, size_t n,
                           float lr_t, float beta1, float beta2, float eps, float grad_scale, const float* lr_t_dev,
                           void* stream) {
  A3D_REQUIRE(ctx && w && g && m && v, "adam: null argument");
  if (n == 0) return 0;
  bool vec = aligned16(w) && aligned16(g) && aligned16(m) && aligned16(v) &&
             (!w_bf16 || (reinterpret_cast<uintptr_t>(w_bf16) & 7) == 0);
  size_t n4 = vec ? n / 4 : 0;
  if (n4) {
    int block = 256, grid = grid_for(ctx, n4, block);
    adam_tf_kernel<<<grid, block, 0, as_stream(stream)>>>(reinterpret_cast<float4*>(w), reinterpret_cast<const float4*>(g),
                                                        reinterpret_cast<float4*>(m), reinterpret_cast<float4*>(v),
                                                        reinterpret_cast<uint2*>(w_bf16), n4, lr_t, beta1, beta2, eps,
                                                        grad_scale, lr_t_dev);
    A3D_LAUNCH_OK(ctx);
  }
  size_t done = n4 * 4;
  if (done < n) {
    size_t rem = n - done;
    adam_tf_tail_kernel<<<ceil_div(rem, 256), 256, 0, as_stream(stream)>>>(w, g, m, v, w_bf16, done, n, lr_t, beta1, beta2,
                                                                          eps, grad_scale, lr_t_dev);
    A3D_LAUNCH_OK(ctx);
  }
  return 0;
}

__global__ void sgd_kernel(float* __restrict__ w, const float* __restrict__ g, uint16_t* __restrict__ wb, size_t n, float lr,
                           float gs) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float ww = w[i] - lr * (g[i] * gs);
    w[i] = ww;
    if (wb) wb[i] = f32_to_bf16_bits(ww);
  }
}
extern "C" int a3d_sgd(a3d_ctx* ctx, float* w, const float* g, uint16_t* w_bf16, size_t n, float lr, float grad_scale,
                       void* stream) {
  A3D_REQUIRE(ctx && w && g, "sgd: null argument");
  if (n == 0) return 0;
  int block = 256, grid = grid_for(ctx, n, block);
  sgd_kernel<<<grid, block, 0, as_stream(stream)>>>(w, g, w_bf16, n, lr, grad_scale);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ s, uint16_t* __restrict__ d, size_t n) {
  size_t n4 = n / 4;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 f = __ldg(reinterpret_cast<const float4*>(s) + i);
    reinterpret_cast<uint2*>(d)[i] = make_uint2(pack_bf16x2(f.x, f.y), pack_bf16x2(f.z, f.w));
  }
  size_t i = n4 * 4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) d[i] = f32_to_bf16_bits(s[i]);
}
__global__ void cast_f32_bf16_scalar_kernel(const float* __restrict__ s, uint16_t* __restrict__ d, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    d[i] = f32_to_bf16_bits(s[i]);
}
extern "C" int a3d_cast_f32_bf16(a3d_ctx* ctx, const float* src, uint16_t* dst, size_t n, void* stream) {
  A3D_REQUIRE(ctx && src && dst, "cast: null argument");
  if (n == 0) return 0;
  int block = 256;
  if (aligned16(src) && (reinterpret_cast<uintptr_t>(dst) & 7) == 0) {
    int grid = grid_for(ctx, n / 4 + 1, block);
    cast_f32_bf16_kernel<<<grid, block, 0, as_stream(stream)>>>(src, dst, n);
  } else {
    cast_f32_bf16_scalar_kernel<<<grid_for(ctx, n, block), block, 0, as_stream(stream)>>>(src, dst, n);
  }
  A3D_LAUNCH_OK(ctx);
  return 0;
}

__global__ void scatter_channel_kernel(const float* __restrict__ s, uint16_t* __restrict__ d, size_t rows, int ld, int ch) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < rows; i += (size_t)gridDim.x * blockDim.x)
    d[i * ld + ch] = f32_to_bf16_bits(s[i]);
}
extern "C" int a3d_scatter_channel_bf16(a3d_ctx* ctx, const float* src, uint16_t* dst, size_t rows, int ld, int ch,
                                        void* stream) {
  A3D_REQUIRE(ctx && src && dst && ch >= 0 && ch < ld, "scatter_channel: bad argument");
  int block = 256, grid = grid_for(ctx, rows, block);
  scatter_channel_kernel<<<grid, block, 0, as_stream(stream)>>>(src, dst, rows, ld, ch);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

extern "C" int a3d_fill_zero(a3d_ctx* ctx, void* p, size_t bytes, void* stream) {
  A3D_REQUIRE(ctx && p, "fill_zero: null argument");
  A3D_CHECK_CUDA(cudaMemsetAsync(p, 0, bytes, as_stream(stream)));
  return 0;
}

__global__ void apply_mask_kernel(float* __restrict__ g, const uint8_t* __restrict__ keep, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    if (!keep[i]) g[i] = 0.f;
}
extern "C" int a3d_apply_mask_f32(a3d_ctx* ctx, float* g, const uint8_t* keep, size_t n, void* stream) {
  A3D_REQUIRE(ctx && g && keep, "apply_mask: null argument");
  if (n == 0) return 0;
  int block = 256, grid = grid_for(ctx, n, block);
  apply_mask_kernel<<<grid, block, 0, as_stream(stream)>>>(g, keep, n);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

__device__ __forceinline__ uint64_t mix64(uint64_t x) {   // splitmix64 finaliser
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
__global__ void bernoulli_mask_kernel(uint8_t* __restrict__ keep, size_t n, float keep_prob, uint64_t seed,
                                      const int64_t* __restrict__ counter) {
  uint64_t base = mix64(seed ^ mix64((uint64_t)(counter ? *counter : 0)));
  uint32_t thresh = (uint32_t)fminf(keep_prob * 4294967296.f, 4294967295.f);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    keep[i] = ((uint32_t)(mix64(base + i) >> 32) < thresh) ? 1 : 0;
}
extern "C" int a3d_bernoulli_mask(a3d_ctx* ctx, uint8_t* keep, size_t n, float keep_prob, uint64_t seed,
                                  const int64_t* counter_dev, void* stream) {
  A3D_REQUIRE(ctx && keep, "bernoulli_mask: null argument");
  if (n == 0) return 0;
  int block = 256, grid = grid_for(ctx, n, block);
  bernoulli_mask_kernel<<<grid, block, 0, as_stream(stream)>>>(keep, n, keep_prob, seed, counter_dev);
  A3D_LAUNCH_OK(ctx);
  return 0;
}
// ---- in-graph timeline: one thread writes the GPU's global nanosecond timer; captured in a CUDA graph like any kernel
__global__ void stamp_kernel(unsigned long long* slot) {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  *slot = t;
}
extern "C" int a3d_stamp(a3d_ctx* ctx, uint64_t* slot, void* stream) {
  A3D_REQUIRE(ctx && slot, "stamp: null argument");
  stamp_kernel<<<1, 1, 0, as_stream(stream)>>>(reinterpret_cast<unsigned long long*>(slot));
  A3D_CHECK_CUDA(cudaGetLastError());
  return 0;
}
__global__ void increment_i64_kernel(int64_t* p) { *p += 1; }
extern "C" int a3d_increment_i64(a3d_ctx* ctx, int64_t* p, void* stream) {
  A3D_REQUIRE(ctx && p, "increment: null argument");
  increment_i64_kernel<<<1, 1, 0, as_stream(stream)>>>(p);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ f32 pool + routing index
// one thread = one output pixel x 4 channels (16 B f32 loads, 8 B bf16 store, 4 B index store)
__global__ void maxpool2x2_fwd_f32_kernel(const float4* __restrict__ x, int N, int H, int W, int C4,
                                          uint2* __restrict__ y, int ldy4, uint32_t* __restrict__ idx) {
  int OH = H / 2, OW = W / 2;
  size_t total = (size_t)N * OH * OW * C4;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int n, oh, ow, c;
    split_nhwc(i, OH, OW, C4, n, oh, ow, c);
    const float4* p = x + (((size_t)n * H + 2 * oh) * W + 2 * ow) * C4 + c;
    float4 v[4] = {__ldg(p), __ldg(p + C4), __ldg(p + (size_t)W * C4), __ldg(p + (size_t)W * C4 + C4)};
    float m[4];
    uint32_t packed = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float best = (&v[0].x)[e];
      int arg = 0;
#pragma unroll
      for (int k = 1; k < 4; ++k) {
        float val = (&v[k].x)[e];
        if (val > best) { best = val; arg = k; }
      }
      m[e] = best;
      packed |= (uint32_t)(best > 0.f ? arg : 4) << (8 * e);
    }
    size_t o = ((size_t)n * OH + oh) * OW + ow;
    y[o * ldy4 + c] = make_uint2(pack_bf16x2(m[0], m[1]), pack_bf16x2(m[2], m[3]));
    if (idx) idx[o * C4 + c] = packed;
  }
}

extern "C" int a3d_maxpool2x2_fwd_f32(a3d_ctx* ctx, const float* x, int N, int H, int W, int C, uint16_t* y, int ldy,
                                      uint8_t* idx, void* stream) {
  A3D_REQUIRE(ctx && x && y, "maxpool_f32: null argument");
  A3D_REQUIRE(C % 4 == 0 && ldy % 4 == 0 && ldy >= C && H >= 2 && W >= 2, "maxpool_f32: C and ldy must be multiples of 4");
  size_t total = (size_t)N * (H / 2) * (W / 2) * (C / 4);
  int block = 256, grid = grid_for(ctx, total, block);
  maxpool2x2_fwd_f32_kernel<<<grid, block, 0, as_stream(stream)>>>(reinterpret_cast<const float4*>(x), N, H, W, C / 4,
                                                                 reinterpret_cast<uint2*>(y), ldy / 4,
                                                                 reinterpret_cast<uint32_t*>(idx));
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// one thread = one (possibly partial) 2x2 window x 4 channels
__global__ void maxpool2x2_idx_bwd_kernel(const uint32_t* __restrict__ idx, const uint2* __restrict__ dy, int lddy4, int N,
                                          int H, int W, int C4, uint2* __restrict__ dx) {
  int OH = H / 2, OW = W / 2;
  int GH = (H + 1) / 2, GW = (W + 1) / 2;
  size_t total = (size_t)N * GH * GW * C4;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int n, gh, gw, c;
    split_nhwc(i, GH, GW, C4, n, gh, gw, c);
    int h0 = 2 * gh, w0 = 2 * gw;
    bool covered = (gh < OH) && (gw < OW);
    size_t base = (((size_t)n * H + h0) * W + w0) * C4 + c;
    uint2 out[4] = {make_uint2(0, 0), make_uint2(0, 0), make_uint2(0, 0), make_uint2(0, 0)};
    if (covered) {
      size_t o = ((size_t)n * OH + gh) * OW + gw;
      uint32_t packed = __ldg(idx + o * C4 + c);
      uint2 g = __ldg(dy + o * lddy4 + c);
      const uint16_t* gv = reinterpret_cast<const uint16_t*>(&g);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        uint32_t a = (packed >> (8 * e)) & 0xff;
        if (a < 4) reinterpret_cast<uint16_t*>(&out[a])[e] = gv[e];
      }
    }
    dx[base] = out[0];
    if (w0 + 1 < W) dx[base + C4] = out[1];
    if (h0 + 1 < H) {
      dx[base + (size_t)W * C4] = out[2];
      if (w0 + 1 < W) dx[base + (size_t)W * C4 + C4] = out[3];
    }
  }
}

// the same with 8 channels per thread: 16-byte stores (a warp writes 512 contiguous bytes per input row)
__global__ void maxpool2x2_idx_bwd8_kernel(const uint2* __restrict__ idx, const uint4* __restrict__ dy, int lddy8, int N,
                                           int H, int W, int C8, uint4* __restrict__ dx) {
  int OH = H / 2, OW = W / 2;
  int GH = (H + 1) / 2, GW = (W + 1) / 2;
  size_t total = (size_t)N * GH * GW * C8;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int n, gh, gw, c;
    split_nhwc(i, GH, GW, C8, n, gh, gw, c);
    int h0 = 2 * gh, w0 = 2 * gw;
    bool covered = (gh < OH) && (gw < OW);
    size_t base = (((size_t)n * H + h0) * W + w0) * C8 + c;
    uint4 out[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) out[a] = make_uint4(0, 0, 0, 0);
    if (covered) {
      size_t o = ((size_t)n * OH + gh) * OW + gw;
      const uint2 packed = __ldg(idx + o * C8 + c);
      const uint4 g = __ldg(dy + o * lddy8 + c);
      const uint16_t* gv = reinterpret_cast<const uint16_t*>(&g);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const uint32_t a = ((e < 4 ? packed.x : packed.y) >> (8 * (e & 3))) & 0xff;
#pragma unroll
        for (int q = 0; q < 4; ++q)                     // constant indices: the four outputs stay in registers
          if (a == (uint32_t)q) reinterpret_cast<uint16_t*>(&out[q])[e] = gv[e];
      }
    }
    dx[base] = out[0];
    if (w0 + 1 < W) dx[base + C8] = out[1];
    if (h0 + 1 < H) {
      dx[base + (size_t)W * C8] = out[2];
      if (w0 + 1 < W) dx[base + (size_t)W * C8 + C8] = out[3];
    }
  }
}

extern "C" int a3d_maxpool2x2_idx_bwd(a3d_ctx* ctx, const uint8_t* idx, const uint16_t* dy, int lddy, int N, int H, int W,
                                      int C, uint16_t* dx, void* stream) {
  A3D_REQUIRE(ctx && idx && dy && dx, "maxpool_idx_bwd: null argument");
  A3D_REQUIRE(C % 4 == 0 && lddy % 4 == 0 && lddy >= C, "maxpool_idx_bwd: C and lddy must be multiples of 4");
  if (C % 8 == 0 && lddy % 8 == 0 && ((reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx)) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(idx) & 7) == 0) {
    size_t total8 = (size_t)N * ((H + 1) / 2) * ((W + 1) / 2) * (C / 8);
    int grid8 = grid_for(ctx, total8, 256);
    maxpool2x2_idx_bwd8_kernel<<<grid8, 256, 0, as_stream(stream)>>>(reinterpret_cast<const uint2*>(idx),
                                                                    reinterpret_cast<const uint4*>(dy), lddy / 8, N, H, W,
                                                                    C / 8, reinterpret_cast<uint4*>(dx));
    A3D_LAUNCH_OK(ctx);
    return 0;
  }
  size_t total = (size_t)N * ((H + 1) / 2) * ((W + 1) / 2) * (C / 4);
  int block = 256, grid = grid_for(ctx, total, block);
  maxpool2x2_idx_bwd_kernel<<<grid, block, 0, as_stream(stream)>>>(reinterpret_cast<const uint32_t*>(idx),
                                                                 reinterpret_cast<const uint2*>(dy), lddy / 4, N, H, W,
                                                                 C / 4, reinterpret_cast<uint2*>(dx));
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// TF-Adam with a bf16 gradient (data-parallel exchange dtype): 14 B read + 14 B written per parameter.
__global__ void adam_tf_bf16g_kernel(float4* __restrict__ w, const uint2* __restrict__ g, float4* __restrict__ m,
                                     float4* __restrict__ v, uint2* __restrict__ wb, size_t n4, float lr_t, float b1,
                                     float b2, float eps, float gs, const float* __restrict__ lr_dev) {
  if (lr_dev) lr_t = __ldg(lr_dev);
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    float4 W = w[i], M = m[i], V = v[i];
    uint2 G = __ldg(g + i);
    float gk[4] = {__uint_as_float(G.x << 16), __uint_as_float(G.x & 0xffff0000u), __uint_as_float(G.y << 16),
                   __uint_as_float(G.y & 0xffff0000u)};
    float* pw = &W.x; float* pm = &M.x; float* pv = &V.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float gg = gk[k] * gs;
      pm[k] = b1 * pm[k] + (1.f - b1) * gg;
      pv[k] = b2 * pv[k] + (1.f - b2) * gg * gg;
      pw[k] = pw[k] - lr_t * pm[k] / (sqrtf(pv[k]) + eps);
    }
    w[i] = W; m[i] = M; v[i] = V;
    if (wb) wb[i] = make_uint2(pack_bf16x2(W.x, W.y), pack_bf16x2(W.z, W.w));
  }
}
extern "C" int a3d_adam_tf_bf16g(a3d_ctx* ctx, float* w, const uint16_t* g, float* m, float* v, uint16_t* w_bf16, size_t n,
                                 float lr_t, float beta1, float beta2, float eps, float grad_scale, const float* lr_t_dev,
                                 void* stream) {
  A3D_REQUIRE(ctx && w && g && m && v, "adam_bf16g: null argument");
  A3D_REQUIRE(n % 4 == 0 && aligned16(w) && aligned16(m) && aligned16(v) && (reinterpret_cast<uintptr_t>(g) & 7) == 0 &&
                  (!w_bf16 || (reinterpret_cast<uintptr_t>(w_bf16) & 7) == 0),
              "adam_bf16g: segment must be a multiple of 4 elements and 16-byte aligned");
  if (n == 0) return 0;
  int block = 256, grid = grid_for(ctx, n / 4, block);
  adam_tf_bf16g_kernel<<<grid, block, 0, as_stream(stream)>>>(
      reinterpret_cast<float4*>(w), reinterpret_cast<const uint2*>(g), reinterpret_cast<float4*>(m),
      reinterpret_cast<float4*>(v), reinterpret_cast<uint2*>(w_bf16), n / 4, lr_t, beta1, beta2, eps, grad_scale, lr_t_dev);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// one thread = one source pixel of 4 channels (8 bytes)
__global__ void space_to_depth2_kernel(const uint2* __restrict__ src, int N, int H, int W, int C4, uint2* __restrict__ dst) {
  size_t total = (size_t)N * H * W * C4;
  const int H2 = H / 2, W2 = W / 2;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    int n, h, w, c;
    split_nhwc(i, H, W, C4, n, h, w, c);
    size_t o = ((((size_t)n * H2 + h / 2) * W2 + w / 2) * 4 + (h & 1) * 2 + (w & 1)) * C4 + c;
    dst[o] = __ldg(src + i);
  }
}
extern "C" int a3d_space_to_depth2(a3d_ctx* ctx, const uint16_t* src, int N, int H, int W, int C, uint16_t* dst,
                                   void* stream) {
  A3D_REQUIRE(ctx && src && dst && C % 4 == 0 && H % 2 == 0 && W % 2 == 0, "space_to_depth2: bad argument");
  size_t total = (size_t)N * H * W * (C / 4);
  int block = 256, grid = grid_for(ctx, total, block);
  space_to_depth2_kernel<<<grid, block, 0, as_stream(stream)>>>(reinterpret_cast<const uint2*>(src), N, H, W, C / 4,
                                                              reinterpret_cast<uint2*>(dst));
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ resize -> space-to-depth
// Bilinear resize (TF1 legacy mapping, as above) written directly in space-to-depth layout: an s x s block
// of resized pixels becomes ONE pixel of s*s*C channels, dst[b][Y][X][(dy*s+dx)*C + c] = resized[b][s*Y+dy][s*X+dx][c],
// channels >= s*s*C are zero.  One thread writes 8 consecutive bf16 channels (16 bytes), so consecutive
// threads fill whole 128-byte pixel rows.  (MSDN: 228x304x3 -> 57x76x64, the input of the stride-4 11x11
// coarse/conv2d_0 and of the pool-fused stride-2 9x9 fine/first, both 3x3 stride-1 convolutions in this layout.)
__global__ void resize_bilinear_tf1_s2d_kernel(const float* __restrict__ src, int B, int H, int W, int C,
                                               uint4* __restrict__ dst, int OHs, int OWs, int s, int dstC8, float sy,
                                               float sx) {
  const size_t total = (size_t)B * OHs * OWs * dstC8;
  const int real = s * s * C;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int q = (int)(i % dstC8);
    size_t t = i / dstC8;
    const int X = (int)(t % OWs);
    t /= OWs;
    const int Y = (int)(t % OHs);
    const int b = (int)(t / OHs);
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = q * 8 + j;
      float r = 0.f;
      if (k < real) {
        const int pix = k / C, c = k - pix * C;
        const int dy = pix / s, dx = pix - dy * s;
        const int oy = Y * s + dy, ox = X * s + dx;
        const float fy = oy * sy, fx = ox * sx;
        const int y0 = (int)floorf(fy), x0 = (int)floorf(fx);
        const int y1 = min(y0 + 1, H - 1), x1 = min(x0 + 1, W - 1);
        const float ly = fy - y0, lx = fx - x0;
        const float* r0 = src + ((size_t)b * H + y0) * W * C;
        const float* r1 = src + ((size_t)b * H + y1) * W * C;
        const float tl = __ldg(r0 + (size_t)x0 * C + c), tr = __ldg(r0 + (size_t)x1 * C + c);
        const float bl = __ldg(r1 + (size_t)x0 * C + c), br = __ldg(r1 + (size_t)x1 * C + c);
        const float top = tl + (tr - tl) * lx;
        const float bot = bl + (br - bl) * lx;
        r = top + (bot - top) * ly;
      }
      v[j] = r;
    }
    dst[i] = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  }
}

// s = 4, C = 3 (the MSDN image): one thread = one row of a 4x4 block = 4 resized pixels x 3 channels = 24 contiguous
// output bytes; neighbouring threads read neighbouring source strips.  The zero channels [48, dstC) are written by
// the dy == 0 thread (40 bytes when dstC = 64).
__global__ void resize_bilinear_tf1_s2d4c3_kernel(const float* __restrict__ src, int B, int H, int W,
                                                  uint16_t* __restrict__ dst, int OH, int OWs, int dstC, float sy, float sx) {
  const size_t total = (size_t)B * OH * OWs;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int X = (int)(i % OWs);
    size_t t = i / OWs;
    const int oy = (int)(t % OH);
    const int b = (int)(t / OH);
    const float fy = oy * sy;
    const int y0 = (int)floorf(fy);
    const int y1 = min(y0 + 1, H - 1);
    const float ly = fy - y0;
    const float* r0 = src + ((size_t)b * H + y0) * W * 3;
    const float* r1 = src + ((size_t)b * H + y1) * W * 3;
    float v[12];
#pragma unroll
    for (int dx = 0; dx < 4; ++dx) {
      const float fx = (X * 4 + dx) * sx;
      const int x0 = (int)floorf(fx);
      const int x1 = min(x0 + 1, W - 1);
      const float lx = fx - x0;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float tl = __ldg(r0 + (size_t)x0 * 3 + c), tr = __ldg(r0 + (size_t)x1 * 3 + c);
        const float bl = __ldg(r1 + (size_t)x0 * 3 + c), br = __ldg(r1 + (size_t)x1 * 3 + c);
        const float top = tl + (tr - tl) * lx;
        const float bot = bl + (br - bl) * lx;
        v[dx * 3 + c] = top + (bot - top) * ly;
      }
    }
    const int Y = oy >> 2, dy = oy & 3;
    uint16_t* o = dst + (((size_t)b * (OH >> 2) + Y) * OWs + X) * dstC;
    uint2* o8 = reinterpret_cast<uint2*>(o + dy * 12);
    o8[0] = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
    o8[1] = make_uint2(pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
    o8[2] = make_uint2(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]));
    if (dy == 0)
      for (int k = 48; k < dstC; k += 4) *reinterpret_cast<uint2*>(o + k) = make_uint2(0u, 0u);
  }
}

// Row-staged resize (used when two pairs of source rows fit in shared memory): the two source rows an output row
// interpolates between are loaded ONCE with coalesced 16-byte copies (every source byte crosses HBM -> SM a single time:
// 118 MB for the MSDN batch).  Persistent blocks, each walks over output rows and copies the two source rows of its
// NEXT output row into the other half of shared memory (cp.async, 16 bytes per thread and instruction) while it
// interpolates the current one, so every resident block always has loads in flight (a one-shot kernel with one block
// per output row spent half of each block's life in its compute/store phase: 2.9 TB/s).
// T = float (the reference's tensor contract, src/data.py:82-86) or uint8_t (8-bit wire format: value / 255,
// i.e. the pixels before tools/data_tf_converter.py:36-37 turned them into floats; `scale` = 1/255).
template <typename T>
__global__ void __launch_bounds__(256)
resize_s2d4c3_rows_pipelined_kernel(const T* __restrict__ src, int H, int W, uint16_t* __restrict__ dst, int OH, int OWs,
                                    int dstC, float sy, float sx, int total_rows, float scale) {
  extern __shared__ __align__(16) uint8_t rp_sm[];      // [2 buffers][2 rows][W*3*sizeof(T)]
  const int row_bytes = W * 3 * (int)sizeof(T);
  const int row_ch = row_bytes / 16;                    // 16-byte chunks per source row
  const uint32_t sm_base = static_cast<uint32_t>(__cvta_generic_to_shared(rp_sm));
  auto issue = [&](int r, int buf) {
    const int oy = r % OH, b = r / OH;
    const int y0 = (int)floorf(oy * sy);
    const int y1 = min(y0 + 1, H - 1);
    const uint8_t* r0 = reinterpret_cast<const uint8_t*>(src + ((size_t)b * H + y0) * W * 3);
    const uint8_t* r1 = reinterpret_cast<const uint8_t*>(src + ((size_t)b * H + y1) * W * 3);
    const uint32_t d0 = sm_base + (uint32_t)(buf * 2 * row_bytes);
    for (int i = threadIdx.x; i < 2 * row_ch; i += blockDim.x) {
      const int which = i >= row_ch;
      const int j = i - which * row_ch;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d0 + (uint32_t)(which * row_bytes + j * 16)),
                   "l"((which ? r1 : r0) + (size_t)j * 16)
                   : "memory");
    }
  };
  int r = blockIdx.x, buf = 0;
  if (r < total_rows) issue(r, 0);
  asm volatile("cp.async.commit_group;" ::: "memory");
  for (; r < total_rows; r += gridDim.x) {
    const int nxt = r + gridDim.x;
    if (nxt < total_rows) issue(nxt, buf ^ 1);
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 1;" ::: "memory");       // the rows of r have landed (this thread's copies)
    __syncthreads();                                           // ... and everybody else's
    const T* a0 = reinterpret_cast<const T*>(rp_sm + (size_t)buf * 2 * row_bytes);
    const T* a1 = reinterpret_cast<const T*>(rp_sm + (size_t)buf * 2 * row_bytes + row_bytes);
    const int oy = r % OH, b = r / OH;
    const float fy = oy * sy;
    const float ly = fy - floorf(fy);
    const int Y = oy >> 2, dy = oy & 3;
    uint16_t* orow = dst + ((size_t)b * (OH >> 2) + Y) * OWs * dstC;
    for (int t = threadIdx.x; t < OWs * 3; t += blockDim.x) {
      const int X = t / 3, p = t - X * 3;               // piece p = values 4p .. 4p+3 of the 12 (dx, c) values
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = p * 4 + j;
        const int dx = k / 3, c = k - dx * 3;
        const float fx = (X * 4 + dx) * sx;
        const int x0 = (int)floorf(fx);
        const int x1 = min(x0 + 1, W - 1);
        const float lx = fx - x0;
        const float tl = (float)a0[x0 * 3 + c], tr = (float)a0[x1 * 3 + c], bl = (float)a1[x0 * 3 + c],
                    br = (float)a1[x1 * 3 + c];
        const float top = tl + (tr - tl) * lx;
        const float bot = bl + (br - bl) * lx;
        v[j] = (top + (bot - top) * ly) * scale;
      }
      *reinterpret_cast<uint2*>(orow + (size_t)X * dstC + dy * 12 + p * 4) =
          make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
    }
    if (dy == 0) {
      const int padq = (dstC - 48) / 4;                  // uint2 pieces of zero padding per pixel
      for (int t = threadIdx.x; t < OWs * padq; t += blockDim.x) {
        const int X = t / padq, q = t - X * padq;
        *reinterpret_cast<uint2*>(orow + (size_t)X * dstC + 48 + q * 4) = make_uint2(0u, 0u);
      }
    }
    __syncthreads();                                           // buffer `buf` is refilled in the next iteration
    buf ^= 1;
  }
}

template <typename T>
static int launch_resize_pipelined(a3d_ctx* ctx, const T* src, int B, int H, int W, uint16_t* dst, int OH, int OW,
                                   int dstC, float scale, cudaStream_t st) {
  const size_t smem = (size_t)W * 3 * sizeof(T) * 4;
  static int blocks_per_sm = 0;
  static size_t smem_set = 0;
  if (smem > smem_set) {
    A3D_CHECK_CUDA(cudaFuncSetAttribute(resize_s2d4c3_rows_pipelined_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem));
    A3D_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, resize_s2d4c3_rows_pipelined_kernel<T>,
                                                                 256, smem));
    smem_set = smem;
  }
  const int total = B * OH;
  int grid = ctx->sm_count * (blocks_per_sm > 0 ? blocks_per_sm : 1);
  if (grid > total) grid = total;
  resize_s2d4c3_rows_pipelined_kernel<T><<<grid, 256, smem, st>>>(src, H, W, dst, OH, OW / 4, dstC, (float)H / (float)OH,
                                                                 (float)W / (float)OW, total, scale);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// 8-bit images: dst = space-to-depth(4) of resize(src / 255).  Same kernel as the float path, a quarter of the
// bytes over PCIe and HBM.
extern "C" int a3d_resize_bilinear_tf1_s2d_u8(a3d_ctx* ctx, const uint8_t* src, int B, int H, int W, int C, uint16_t* dst,
                                              int OH, int OW, int s, int dstC, void* stream) {
  A3D_REQUIRE(ctx && src && dst, "resize_s2d_u8: null argument");
  A3D_REQUIRE(B > 0 && H > 0 && W > 0 && C == 3 && s == 4 && OH % 4 == 0 && OW % 4 == 0 && dstC % 8 == 0 && dstC >= 48 &&
                  (reinterpret_cast<uintptr_t>(dst) & 15) == 0 && (W * 3) % 16 == 0 &&
                  (reinterpret_cast<uintptr_t>(src) & 15) == 0 && (size_t)W * 3 * 4 <= 200 * 1024,
              "resize_s2d_u8: needs C == 3, s == 4, 16-byte aligned source rows (W*3 %% 16 == 0)");
  return launch_resize_pipelined<uint8_t>(ctx, src, B, H, W, dst, OH, OW, dstC, 1.f / 255.f, as_stream(stream));
}

extern "C" int a3d_resize_bilinear_tf1_s2d(a3d_ctx* ctx, const float* src, int B, int H, int W, int C, uint16_t* dst,
                                           int OH, int OW, int s, int dstC, void* stream) {
  A3D_REQUIRE(ctx && src && dst, "resize_s2d: null argument");
  A3D_REQUIRE(B > 0 && H > 0 && W > 0 && C > 0 && s > 0 && OH % s == 0 && OW % s == 0 && dstC % 8 == 0 &&
                  dstC >= s * s * C && (reinterpret_cast<uintptr_t>(dst) & 15) == 0,
              "resize_s2d: bad shape (OH, OW multiples of s; dstC %% 8 == 0 and >= s*s*C)");
  float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  if (s == 4 && C == 3 && (W * 3) % 4 == 0 && (size_t)W * 3 * 4 * sizeof(float) <= 100 * 1024 && dstC % 4 == 0 &&
      (reinterpret_cast<uintptr_t>(src) & 15) == 0)
    return launch_resize_pipelined<float>(ctx, src, B, H, W, dst, OH, OW, dstC, 1.f, as_stream(stream));
  if (s == 4 && C == 3) {
    const size_t rows = (size_t)B * OH * (OW / 4);
    int block = 256, grid = grid_for(ctx, rows, block);
    resize_bilinear_tf1_s2d4c3_kernel<<<grid, block, 0, as_stream(stream)>>>(src, B, H, W, dst, OH, OW / 4, dstC, sy, sx);
    A3D_LAUNCH_OK(ctx);
    return 0;
  }
  const size_t total = (size_t)B * (OH / s) * (OW / s) * (dstC / 8);
  int block = 256, grid = grid_for(ctx, total, block);
  resize_bilinear_tf1_s2d_kernel<<<grid, block, 0, as_stream(stream)>>>(src, B, H, W, C, reinterpret_cast<uint4*>(dst),
                                                                      OH / s, OW / s, s, dstC / 8, sy, sx);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ pool4 backward
// Backward of the pool-fused convolution (a3d_conv2d_pool4_fwd): MaxPoolGrad + ReluGrad expressed on the GEMM
// columns, dybig[row][g*64 + c] = (idx[row][c] == g && y[row][c] > 0) ? dy[row][c] : 0.
__global__ void pool4_bwd_kernel(const uint16_t* __restrict__ dy, int lddy, const uint16_t* __restrict__ y, int ldy,
                                 const uint8_t* __restrict__ idx, uint4* __restrict__ dybig, size_t rows) {
  const size_t total = rows * 32;               // one thread = 8 of the 256 columns
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t row = i >> 5;
    const int col = (int)(i & 31) * 8;
    const int g = col >> 6, c = col & 63;
    const uint4 d = __ldg(reinterpret_cast<const uint4*>(dy + row * lddy + c));
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(y + row * ldy + c));
    const uint2 k = __ldg(reinterpret_cast<const uint2*>(idx + row * 64 + c));
    const uint16_t* dv = reinterpret_cast<const uint16_t*>(&d);
    const uint16_t* av = reinterpret_cast<const uint16_t*>(&a);
    const uint8_t* kv = reinterpret_cast<const uint8_t*>(&k);
    uint16_t o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = (kv[j] == g && bf16_bits_to_f32(av[j]) > 0.f) ? dv[j] : (uint16_t)0;
    dybig[i] = make_uint4(o[0] | ((uint32_t)o[1] << 16), o[2] | ((uint32_t)o[3] << 16), o[4] | ((uint32_t)o[5] << 16),
                          o[6] | ((uint32_t)o[7] << 16));
  }
}

extern "C" int a3d_pool4_bwd(a3d_ctx* ctx, const uint16_t* dy, int lddy, const uint16_t* y, int ldy, const uint8_t* idx,
                             uint16_t* dybig, size_t rows, void* stream) {
  A3D_REQUIRE(ctx && dy && y && idx && dybig && rows > 0, "pool4_bwd: null argument");
  A3D_REQUIRE(lddy % 8 == 0 && ldy % 8 == 0 && lddy >= 64 && ldy >= 64, "pool4_bwd: row pitches must be multiples of 8 elements");
  int block = 256, grid = grid_for(ctx, rows * 32, block);
  pool4_bwd_kernel<<<grid, block, 0, as_stream(stream)>>>(dy, lddy, y, ldy, idx, reinterpret_cast<uint4*>(dybig), rows);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ embedded-filter maps
// A filter that is stored several times inside a larger (derived) filter -- the four shifted copies of the 9x9
// fine/first filter inside the pool-fused 3x3x64 -> 256 filter -- keeps ONE canonical copy in the parameter arena.
// idx[g][e] (int32, -1 = none) is the position of canonical element e in copy g of the derived tensor.
//   gather_sum:   dst[e] = sum_g src[idx[g][e]]              (fold the derived filter's gradient)
//   scatter_cast: dst[idx[g][e]] = bf16(src[e])              (refresh the derived filter after an update)
__global__ void gather_sum_f32_kernel(const float* __restrict__ src, const int* __restrict__ idx, int G, size_t n,
                                      float* __restrict__ dst) {
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int g = 0; g < G; ++g) {
      const int k = __ldg(idx + (size_t)g * n + e);
      if (k >= 0) acc += __ldg(src + k);
    }
    dst[e] = acc;
  }
}
__global__ void scatter_cast_bf16_kernel(const float* __restrict__ src, const int* __restrict__ idx, int G, size_t n,
                                         uint16_t* __restrict__ dst) {
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < n; e += (size_t)gridDim.x * blockDim.x) {
    const uint16_t v = f32_to_bf16_bits(__ldg(src + e));
    for (int g = 0; g < G; ++g) {
      const int k = __ldg(idx + (size_t)g * n + e);
      if (k >= 0) dst[k] = v;
    }
  }
}
extern "C" int a3d_gather_sum_f32(a3d_ctx* ctx, const float* src, const int* idx, int G, size_t n, float* dst, void* stream) {
  A3D_REQUIRE(ctx && src && idx && dst && G > 0 && n > 0, "gather_sum: bad argument");
  int block = 256, grid = grid_for(ctx, n, block);
  gather_sum_f32_kernel<<<grid, block, 0, as_stream(stream)>>>(src, idx, G, n, dst);
  A3D_LAUNCH_OK(ctx);
  return 0;
}
extern "C" int a3d_scatter_cast_bf16(a3d_ctx* ctx, const float* src, const int* idx, int G, size_t n, uint16_t* dst,
                                     void* stream) {
  A3D_REQUIRE(ctx && src && idx && dst && G > 0 && n > 0, "scatter_cast: bad argument");
  int block = 256, grid = grid_for(ctx, n, block);
  scatter_cast_bf16_kernel<<<grid, block, 0, as_stream(stream)>>>(src, idx, G, n, dst);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// ------------------------------------------------------------------------------------ dense wgrad + TF-Adam, one pass
// For the batch-32 dense layers the weight gradient dw[n][k] = sum_b dy[b][n] * x[b][k] is 32 FMAs per parameter,
// while the optimizer moves 26 bytes per parameter: the update is HBM-bound and the gradient is cheap enough to be
// recomputed from the two small activation matrices INSIDE the optimizer pass.  The f32 gradient (4 B written + 4 B
// read per parameter, 536 MB for MSDN's 67 M dense parameters) then never exists in HBM.
// ------------------------------------------------------------------------------------ dense wgrad + TF-Adam (mma.sync)
// The 32-term dot products run on the tensor cores (warp-level mma.sync m16n8k16, bf16 -> f32; on the CUDA cores the
// same pass was issue-bound at 381 us against 277 us):
// the kernel keeps the shape of the plain optimizer pass -- many resident warps streaming w/m/v -- and the gradient
// costs 8 MMAs per 512 parameters instead of 512 FMAs per 16.  No shared memory, no block-level synchronisation.
//   MMA M = 16 weight rows n, K = batch b (2 steps of 16), N = 8 weight columns k per tile
//   A[n][b] = dy[b][n], B[b][k] = x[b][k], D[n][k] = dw[n][k]
// A warp owns 16 rows x 32 columns: 4 MMA column tiles whose columns are PERMUTED so that a thread's accumulators
// of a tile pair are 4 consecutive weight columns (one float4 of w/m/v per row): MMA column c of tile j (pair q =
// j/2) is weight column 16q + 4(c/2) + 2(j%2) + c%2.  The B fragments depend only on the warp's columns and are
// loaded once; row tiles are dealt round-robin over gridDim.y (one resident wave, compact live footprint).
__device__ __forceinline__ void mma_bf16_16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// kAdamQN = column groups of 16 per warp (warp tile 16 rows x 16*QN columns), kAdamBPS = resident blocks per SM the
// register budget is compiled for, kAdamPF = prefetch the next row tile's w/m/v lines into L2 while this one is updated.
constexpr int kAdamQN = 2, kAdamBPS = 3;
constexpr bool kAdamPF = true;
__global__ void __launch_bounds__(256, kAdamBPS)
dense_wgrad_adam_mma_kernel(const uint16_t* __restrict__ x, int ldx, const uint16_t* __restrict__ dy, int lddy,
                            float* __restrict__ w, float* __restrict__ m, float* __restrict__ v, uint16_t* __restrict__ wb,
                            int M, int N, int K, float lr_t, float b1, float b2, float eps, float gs,
                            const float* __restrict__ lr_dev) {
  if (lr_dev) lr_t = __ldg(lr_dev);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int kc0 = blockIdx.x * (128 * kAdamQN) + warp * (16 * kAdamQN);          // first weight column of this warp
  // B fragments: bfrag[j][kb][0/1], tile j = 2q + h
  uint32_t bfrag[2 * kAdamQN][2][2];
#pragma unroll
  for (int j = 0; j < 2 * kAdamQN; ++j) {
    const int col = kc0 + 16 * (j >> 1) + 4 * (g >> 1) + 2 * (j & 1) + (g & 1);
#pragma unroll
    for (int kb = 0; kb < 2; ++kb)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int b0 = kb * 16 + h * 8 + 2 * t;
        const uint32_t lo = b0 < M ? __ldg(x + (size_t)b0 * ldx + col) : 0u;
        const uint32_t hi = b0 + 1 < M ? __ldg(x + (size_t)(b0 + 1) * ldx + col) : 0u;
        bfrag[j][kb][h] = lo | (hi << 16);
      }
  }
  const int nstep = gridDim.y * 16;
  for (int n0 = blockIdx.y * 16; n0 < N; n0 += nstep) {
    const int r0 = n0 + g, r1 = n0 + g + 8;
    if (kAdamPF && t == 0) {
      // the 4 lanes of a quad cover 64 contiguous bytes per (row, column group): one prefetch per quad
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int row = (half ? r1 : r0) + nstep;
        if (row < N) {
#pragma unroll
          for (int q = 0; q < kAdamQN; ++q) {
            const size_t off = (size_t)row * K + kc0 + 16 * q;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(w + off));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(m + off));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(v + off));
          }
        }
      }
    }
    // A fragments for both batch halves
    uint32_t afrag[2][4];
#pragma unroll
    for (int kb = 0; kb < 2; ++kb)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int row = (i & 1) ? r1 : r0;
        const int b0 = kb * 16 + (i >> 1) * 8 + 2 * t;
        const uint32_t lo = (row < N && b0 < M) ? __ldg(dy + (size_t)b0 * lddy + row) : 0u;
        const uint32_t hi = (row < N && b0 + 1 < M) ? __ldg(dy + (size_t)(b0 + 1) * lddy + row) : 0u;
        afrag[kb][i] = lo | (hi << 16);
      }
    float acc[2 * kAdamQN][4];
#pragma unroll
    for (int j = 0; j < 2 * kAdamQN; ++j) {
      acc[j][0] = acc[j][1] = acc[j][2] = acc[j][3] = 0.f;
      mma_bf16_16816(acc[j], afrag[0], bfrag[j][0]);
      mma_bf16_16816(acc[j], afrag[1], bfrag[j][1]);
    }
    // this thread: rows r0 / r1, column groups q -> float4 at column kc0 + 16q + 4t
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int row = half ? r1 : r0;
      if (row < N) {
        float4 W[kAdamQN], Mo[kAdamQN], V[kAdamQN];
#pragma unroll
        for (int q = 0; q < kAdamQN; ++q) {
          const size_t off = (size_t)row * K + kc0 + 16 * q + 4 * t;
          W[q] = *reinterpret_cast<const float4*>(w + off);
          Mo[q] = *reinterpret_cast<const float4*>(m + off);
          V[q] = *reinterpret_cast<const float4*>(v + off);
        }
#pragma unroll
        for (int q = 0; q < kAdamQN; ++q) {
          const float gr[4] = {acc[2 * q][half * 2], acc[2 * q][half * 2 + 1], acc[2 * q + 1][half * 2],
                               acc[2 * q + 1][half * 2 + 1]};
          float* pw = &W[q].x; float* pm = &Mo[q].x; float* pv = &V[q].x;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float gk = gr[j] * gs;
            pm[j] = b1 * pm[j] + (1.f - b1) * gk;
            pv[j] = b2 * pv[j] + (1.f - b2) * gk * gk;
            pw[j] = pw[j] - lr_t * pm[j] / (sqrtf(pv[j]) + eps);
          }
          const size_t off = (size_t)row * K + kc0 + 16 * q + 4 * t;
          *reinterpret_cast<float4*>(w + off) = W[q];
          *reinterpret_cast<float4*>(m + off) = Mo[q];
          *reinterpret_cast<float4*>(v + off) = V[q];
          if (wb) *reinterpret_cast<uint2*>(wb + off) = make_uint2(pack_bf16x2(W[q].x, W[q].y), pack_bf16x2(W[q].z, W[q].w));
        }
      }
    }
  }
}

int a3d_mma_dense_wgrad_adam(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* w, float* m,
                             float* v, uint16_t* wb, int M, int N, int K, float lr_t, float beta1, float beta2, float eps,
                             float grad_scale, const float* lr_t_dev, cudaStream_t st) {
  if (M > A3D_DENSE_WGRAD_ADAM_MAX_M || K % 256 || !aligned16(w) || !aligned16(m) || !aligned16(v) || (wb && (reinterpret_cast<uintptr_t>(wb) & 7)))
    return A3D_ENOTSUP;
  const int kblocks = K / (128 * kAdamQN);
  int gy = kAdamBPS * ctx->sm_count / kblocks;       // one resident wave
  if (gy < 1) gy = 1;
  if (gy > ceil_div(N, 16)) gy = ceil_div(N, 16);
  dense_wgrad_adam_mma_kernel<<<dim3(kblocks, gy), 256, 0, st>>>(x, ldx, dy, lddy, w, m, v, wb, M, N, K, lr_t, beta1, beta2,
                                                                 eps, grad_scale, lr_t_dev);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// BiasAddGrad alone: db[c] = sum_rows dy[row][c]  (dy bf16 [rows][ld]; group_rows > 0: rows in blocks of group_rows,
// block i at dy + i * group_stride)
extern "C" int a3d_bias_grad_bf16(a3d_ctx* ctx, const uint16_t* dy, size_t rows, int C, int ld, float* db, int group_rows,
                                  size_t group_stride, void* stream) {
  A3D_REQUIRE(ctx && dy && db && rows > 0 && C > 0 && ld >= C, "bias grad: bad argument");
  if (group_rows > 0) return a3d_colsum_bf16_grouped(ctx, dy, (int)rows, C, ld, group_rows, group_stride, db, as_stream(stream));
  return a3d_colsum_bf16(ctx, dy, rows, C, ld, db, as_stream(stream));
}

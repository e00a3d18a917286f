// fp8.cu -- the FP8 inference mode (include/a3d.h "FP8 inference"): E4M3 operands with one scale per weight row and one
// per image, tcgen05.mma kind::f8f6f4 (tc_gemm.cu), and the kernels that produce the E4M3 tensors -- the weight-row
// quantiser, the per-image activation quantiser (optionally fused with the 2x2 max-pool) and the image resize.
//
// Quantisation rule (weights per row, activations per image):  amax = max |x|,  s = amax / 448,  inv = 448 / amax,
// code = e4m3_rn_satfinite(x * inv);  amax == 0 gives s = 0 and all codes 0.  Every step is one float32 operation, so
// oracle/fp8.py restates it bit for bit.  Nothing here synchronises with the host: the whole forward is capturable.
#include "common.cuh"
#include "ptx.cuh"

int a3d_tc_conv_fwd_fp8(a3d_ctx*, const a3d_conv_desc*, const uint8_t* x, const float* x_scale, const uint8_t* w,
                        const float* w_scale, const float* bias, void* y, int y_dtype, unsigned flags, void* ws,
                        size_t ws_bytes, cudaStream_t st, int pool4);
int a3d_tc_dense_fwd_fp8(a3d_ctx*, const uint8_t* x, int ldx, const float* x_scale, const uint8_t* w, const float* w_scale,
                         const float* bias, void* y, int y_dtype, float* acc_ws, int M, int N, int K, unsigned flags,
                         cudaStream_t st);

namespace {

constexpr int kQBlock = 256;            // threads per quantiser block; each thread handles 8 elements per iteration
constexpr int kQMaxParts = 64;          // blocks (partial maxima) per image

__device__ __forceinline__ float e4m3_inv(float amax) { return amax > 0.f ? __fdiv_rn(448.f, amax) : 0.f; }

__device__ __forceinline__ uint2 quant8(const float (&v)[8], float inv) {
  uint32_t w[2];
#pragma unroll
  for (int h = 0; h < 2; ++h)
    w[h] = (uint32_t)ptx::cvt_e4m3x2(__fmul_rn(v[4 * h], inv), __fmul_rn(v[4 * h + 1], inv)) |
           ((uint32_t)ptx::cvt_e4m3x2(__fmul_rn(v[4 * h + 2], inv), __fmul_rn(v[4 * h + 3], inv)) << 16);
  return make_uint2(w[0], w[1]);
}

__device__ __forceinline__ void unpack8(uint4 u, float (&v)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = bf16_bits_to_f32((uint16_t)(w[i] & 0xffffu));
    v[2 * i + 1] = bf16_bits_to_f32((uint16_t)(w[i] >> 16));
  }
}

// Sources of the per-image quantiser: 8 consecutive bf16 values of image b at element e (a multiple of 8).
struct PlainSrc {
  const uint16_t* x;
  size_t n;                              // elements per image
  __device__ void load(int b, size_t e, float (&v)[8]) const {
    unpack8(__ldg(reinterpret_cast<const uint4*>(x + (size_t)b * n + e)), v);
  }
};
// 2x2/2 max-pool of x bf16 [B,H,W,C] on the fly; the pooled image is [H/2, W/2, ldy], channels C..ldy-1 are zero
struct PoolSrc {
  const uint16_t* x;
  int H, W, C, ldy;
  __device__ void load(int b, size_t e, float (&v)[8]) const {
    const int c = (int)(e % ldy);
    if (c >= C) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = 0.f;
      return;
    }
    const size_t pix = e / ldy;
    const int OW = W / 2, ow = (int)(pix % OW), oh = (int)(pix / OW);
    const uint16_t* p = x + (((size_t)b * H + 2 * oh) * W + 2 * ow) * C + c;
    float a[8], t[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(p)), a);
    const size_t offs[3] = {(size_t)C, (size_t)W * C, (size_t)W * C + C};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      unpack8(__ldg(reinterpret_cast<const uint4*>(p + offs[k])), t);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] = fmaxf(a[j], t[j]);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = a[j];
  }
};

// pass 1: part[b][blockIdx.x] = max |x| over the block's share of image b
template <class S>
__global__ void __launch_bounds__(kQBlock) amax_kernel(S src, size_t n, float* __restrict__ part) {
  const int b = blockIdx.y;
  float m = 0.f;
  for (size_t e = ((size_t)blockIdx.x * kQBlock + threadIdx.x) * 8; e < n; e += (size_t)gridDim.x * kQBlock * 8) {
    float v[8];
    src.load(b, e, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) m = fmaxf(m, fabsf(v[j]));
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float red[kQBlock / 32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int i = 1; i < kQBlock / 32; ++i) m = fmaxf(m, red[i]);
    part[(size_t)b * gridDim.x + blockIdx.x] = m;
  }
}

// pass 2: amax of image b from its partial maxima, then codes; block 0 of each image writes the scale
template <class S>
__global__ void __launch_bounds__(kQBlock) quant_kernel(S src, size_t n, const float* __restrict__ part, int nparts,
                                                        uint8_t* __restrict__ y, float* __restrict__ scale) {
  const int b = blockIdx.y;
  float amax = 0.f;
  for (int i = 0; i < nparts; ++i) amax = fmaxf(amax, __ldg(part + (size_t)b * nparts + i));
  const float inv = e4m3_inv(amax);
  if (blockIdx.x == 0 && threadIdx.x == 0) scale[b] = __fdiv_rn(amax, 448.f);
  for (size_t e = ((size_t)blockIdx.x * kQBlock + threadIdx.x) * 8; e < n; e += (size_t)gridDim.x * kQBlock * 8) {
    float v[8];
    src.load(b, e, v);
    *reinterpret_cast<uint2*>(y + (size_t)b * n + e) = quant8(v, inv);
  }
}

int parts_for(size_t n) {
  const size_t p = (n + 16383) / 16384;
  return p < 1 ? 1 : p > kQMaxParts ? kQMaxParts : (int)p;
}

template <class S>
int quantize_images(a3d_ctx* ctx, S src, int B, size_t n, uint8_t* y, float* y_scale, void* ws, size_t ws_bytes,
                    cudaStream_t st) {
  const int parts = parts_for(n);
  A3D_REQUIRE(ws && ws_bytes >= (size_t)B * parts * sizeof(float), "quantize e4m3: workspace too small (%zu B, need %zu)",
              ws_bytes, (size_t)B * parts * sizeof(float));
  float* part = reinterpret_cast<float*>(ws);
  amax_kernel<S><<<dim3(parts, B), kQBlock, 0, st>>>(src, n, part);
  A3D_LAUNCH_OK(ctx);
  quant_kernel<S><<<dim3(parts, B), kQBlock, 0, st>>>(src, n, part, parts, y, y_scale);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// one block per row: amax, scale, codes
__global__ void __launch_bounds__(kQBlock) quant_rows_kernel(const uint16_t* __restrict__ x, int cols, long long ldx,
                                                             uint8_t* __restrict__ q, float* __restrict__ scale) {
  const uint16_t* row = x + (size_t)blockIdx.x * ldx;
  float m = 0.f;
  for (int e = threadIdx.x * 8; e < cols; e += kQBlock * 8) {
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(row + e)), v);
#pragma unroll
    for (int j = 0; j < 8; ++j) m = fmaxf(m, fabsf(v[j]));
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __shared__ float red[kQBlock / 32];
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  float amax = red[0];
  for (int i = 1; i < kQBlock / 32; ++i) amax = fmaxf(amax, red[i]);
  const float inv = e4m3_inv(amax);
  if (threadIdx.x == 0) scale[blockIdx.x] = __fdiv_rn(amax, 448.f);
  for (int e = threadIdx.x * 8; e < cols; e += kQBlock * 8) {
    float v[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(row + e)), v);
    *reinterpret_cast<uint2*>(q + (size_t)blockIdx.x * cols + e) = quant8(v, inv);
  }
}

// TF1 bilinear resize (align_corners = false, as a3d_resize_bilinear_tf1_s2d_f32) + space-to-depth(4) of a 3-channel
// image into E4M3 codes of x * 256: dst [B, OH/4, OW/4, 64], channel dy*12 + dx*3 + c, channels 48..63 zero.
// One thread = one (pixel block, dy): 12 values.  uint8 sources are read as pixel / 255 (one float32 division per tap,
// so they equal a float32 image holding k / 255).
template <typename T>
__global__ void resize_s2d_e4m3_kernel(const T* __restrict__ src, int B, int H, int W, uint8_t* __restrict__ dst, int OHs,
                                       int OWs, float sy, float sx) {
  const size_t total = (size_t)B * OHs * OWs * 4;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int dy = (int)(i & 3);
    size_t t = i >> 2;
    const int X = (int)(t % OWs);
    t /= OWs;
    const int Y = (int)(t % OHs);
    const int b = (int)(t / OHs);
    const int oy = Y * 4 + dy;
    const float fy = oy * sy;
    const int y0 = (int)floorf(fy), y1 = min(y0 + 1, H - 1);
    const float ly = fy - y0;
    const T* r0 = src + ((size_t)b * H + y0) * W * 3;
    const T* r1 = src + ((size_t)b * H + y1) * W * 3;
    float v[12];
#pragma unroll
    for (int dx = 0; dx < 4; ++dx) {
      const float fx = (X * 4 + dx) * sx;
      const int x0 = (int)floorf(fx), x1 = min(x0 + 1, W - 1);
      const float lx = fx - x0;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float tl, tr, bl, br;
        if constexpr (sizeof(T) == 1) {
          tl = __fdiv_rn((float)r0[x0 * 3 + c], 255.f); tr = __fdiv_rn((float)r0[x1 * 3 + c], 255.f);
          bl = __fdiv_rn((float)r1[x0 * 3 + c], 255.f); br = __fdiv_rn((float)r1[x1 * 3 + c], 255.f);
        } else {
          tl = __ldg(r0 + x0 * 3 + c); tr = __ldg(r0 + x1 * 3 + c);
          bl = __ldg(r1 + x0 * 3 + c); br = __ldg(r1 + x1 * 3 + c);
        }
        const float top = tl + (tr - tl) * lx;
        const float bot = bl + (br - bl) * lx;
        v[dx * 3 + c] = (top + (bot - top) * ly) * 256.f;
      }
    }
    uint8_t* o = dst + (((size_t)b * OHs + Y) * OWs + X) * 64;
    uint32_t w[3];
#pragma unroll
    for (int k = 0; k < 3; ++k)
      w[k] = (uint32_t)ptx::cvt_e4m3x2(v[4 * k], v[4 * k + 1]) | ((uint32_t)ptx::cvt_e4m3x2(v[4 * k + 2], v[4 * k + 3]) << 16);
    uint32_t* o32 = reinterpret_cast<uint32_t*>(o + dy * 12);
    o32[0] = w[0]; o32[1] = w[1]; o32[2] = w[2];
    if (dy == 0) *reinterpret_cast<uint4*>(o + 48) = make_uint4(0u, 0u, 0u, 0u);
  }
}

int check_desc_fp8(const a3d_conv_desc* d) {
  A3D_REQUIRE(d, "conv fp8: null descriptor");
  A3D_REQUIRE(d->N > 0 && d->H > 0 && d->W > 0 && d->C > 0 && d->K > 0 && d->R > 0 && d->S > 0, "conv fp8: bad dims");
  A3D_REQUIRE(d->stride_h > 0 && d->stride_w > 0 && d->pad_t >= 0 && d->pad_l >= 0 && d->P > 0 && d->Q > 0,
              "conv fp8: bad stride / pad / output dims");
  A3D_REQUIRE((d->P - 1) * d->stride_h - d->pad_t < d->H && (d->Q - 1) * d->stride_w - d->pad_l < d->W,
              "conv fp8: output larger than the input supports");
  return 0;
}

}  // namespace

extern "C" size_t a3d_quantize_ws_bytes_e4m3(int B, size_t n) { return (size_t)B * parts_for(n) * sizeof(float); }

extern "C" int a3d_quantize_rows_e4m3(a3d_ctx* ctx, const uint16_t* x, int rows, int cols, long long ldx, uint8_t* q,
                                      float* scale, void* stream) {
  A3D_REQUIRE(ctx && x && q && scale && rows > 0 && cols > 0 && cols % 8 == 0 && ldx >= cols && ldx % 8 == 0 &&
                  (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(q) & 7) == 0,
              "quantize rows e4m3: needs cols %% 8 == 0, ldx %% 8 == 0, 16-byte aligned x, 8-byte aligned q");
  quant_rows_kernel<<<rows, kQBlock, 0, as_stream(stream)>>>(x, cols, ldx, q, scale);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

extern "C" int a3d_quantize_e4m3(a3d_ctx* ctx, const uint16_t* x, int B, size_t n, uint8_t* y, float* y_scale, void* ws,
                                 size_t ws_bytes, void* stream) {
  A3D_REQUIRE(ctx && x && y && y_scale && B > 0 && n > 0 && n % 8 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                  (reinterpret_cast<uintptr_t>(y) & 7) == 0,
              "quantize e4m3: needs n %% 8 == 0, 16-byte aligned x, 8-byte aligned y");
  return quantize_images(ctx, PlainSrc{x, n}, B, n, y, y_scale, ws, ws_bytes, as_stream(stream));
}

extern "C" int a3d_maxpool2x2_quantize_e4m3(a3d_ctx* ctx, const uint16_t* x, int B, int H, int W, int C, uint8_t* y, int ldy,
                                            float* y_scale, void* ws, size_t ws_bytes, void* stream) {
  A3D_REQUIRE(ctx && x && y && y_scale && B > 0 && H >= 2 && W >= 2 && C % 8 == 0 && ldy >= C && ldy % 8 == 0 &&
                  (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 7) == 0,
              "maxpool quantize e4m3: needs C %% 8 == 0, ldy >= C, ldy %% 8 == 0, aligned x / y");
  const size_t n = (size_t)(H / 2) * (W / 2) * ldy;
  return quantize_images(ctx, PoolSrc{x, H, W, C, ldy}, B, n, y, y_scale, ws, ws_bytes, as_stream(stream));
}

extern "C" int a3d_resize_bilinear_tf1_s2d_e4m3(a3d_ctx* ctx, const void* src, int src_dtype, int B, int H, int W, int C,
                                                uint8_t* dst, int OH, int OW, int s, int dstC, void* stream) {
  A3D_REQUIRE(ctx && src && dst && B > 0 && H > 0 && W > 0 && C == 3 && s == 4 && dstC == 64 && OH % 4 == 0 &&
                  OW % 4 == 0 && (src_dtype == A3D_F32 || src_dtype == A3D_U8) && (reinterpret_cast<uintptr_t>(dst) & 15) == 0,
              "resize s2d e4m3: needs C == 3, s == 4, dstC == 64, OH / OW multiples of 4, f32 or u8 source");
  const float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  const size_t total = (size_t)B * (OH / 4) * (OW / 4) * 4;
  const int block = 256;
  const size_t want = (total + block - 1) / block, cap = (size_t)ctx->sm_count * 8;
  const int grid = (int)(want < cap ? want : cap);
  cudaStream_t st = as_stream(stream);
  if (src_dtype == A3D_U8)
    resize_s2d_e4m3_kernel<uint8_t><<<grid, block, 0, st>>>(reinterpret_cast<const uint8_t*>(src), B, H, W, dst, OH / 4,
                                                           OW / 4, sy, sx);
  else
    resize_s2d_e4m3_kernel<float><<<grid, block, 0, st>>>(reinterpret_cast<const float*>(src), B, H, W, dst, OH / 4, OW / 4,
                                                         sy, sx);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

extern "C" int a3d_conv2d_fwd_fp8(a3d_ctx* ctx, const a3d_conv_desc* d, const uint8_t* x, const float* x_scale,
                                  const uint8_t* w, const float* w_scale, const float* bias, void* y, int y_dtype,
                                  unsigned flags, void* ws, size_t ws_bytes, void* stream) {
  A3D_REQUIRE(ctx && x && x_scale && w && w_scale && y, "conv fwd fp8: null argument");
  int rc = check_desc_fp8(d);
  if (rc) return rc;
  A3D_REQUIRE(d->ldy >= d->K && (y_dtype == A3D_BF16 || y_dtype == A3D_F32), "conv fwd fp8: ldy >= K, bf16 or f32 output");
  return a3d_tc_conv_fwd_fp8(ctx, d, x, x_scale, w, w_scale, bias, y, y_dtype, flags, ws, ws_bytes, as_stream(stream), 0);
}

extern "C" int a3d_conv2d_pool4_fwd_fp8(a3d_ctx* ctx, const a3d_conv_desc* d, const uint8_t* x, const float* x_scale,
                                        const uint8_t* w, const float* w_scale, const float* bias, uint16_t* y, unsigned flags,
                                        void* stream) {
  A3D_REQUIRE(ctx && x && x_scale && w && w_scale && y, "conv pool4 fwd fp8: null argument");
  int rc = check_desc_fp8(d);
  if (rc) return rc;
  A3D_REQUIRE(d->K == 256 && d->ldy >= 64, "conv pool4 fwd fp8: K must be 4 x 64 and ldy >= 64");
  return a3d_tc_conv_fwd_fp8(ctx, d, x, x_scale, w, w_scale, bias, y, A3D_BF16, flags, nullptr, 0, as_stream(stream), 1);
}

extern "C" int a3d_dense_fwd_fp8(a3d_ctx* ctx, const uint8_t* x, int ldx, const float* x_scale, const uint8_t* w,
                                 const float* w_scale, const float* bias, void* y, int y_dtype, float* acc_ws, int M, int N,
                                 int K, unsigned flags, void* stream) {
  A3D_REQUIRE(ctx && x && x_scale && w && w_scale && y && acc_ws && M > 0 && N > 0 && K > 0 && ldx >= K &&
                  (y_dtype == A3D_BF16 || y_dtype == A3D_F32),
              "dense fwd fp8: bad argument");
  cudaStream_t st = as_stream(stream);
  const size_t esz = y_dtype == A3D_F32 ? 4 : 2;
  for (int m0 = 0; m0 < M; m0 += 256) {          // the batch is the UMMA N dimension (<= 256)
    const int mc = M - m0 < 256 ? M - m0 : 256;
    int rc = a3d_tc_dense_fwd_fp8(ctx, x + (size_t)m0 * ldx, ldx, x_scale + m0, w, w_scale, bias,
                                  reinterpret_cast<uint8_t*>(y) + (size_t)m0 * N * esz, y_dtype, acc_ws + (size_t)m0 * N, mc,
                                  N, K, flags, st);
    if (rc) return rc;
  }
  return 0;
}

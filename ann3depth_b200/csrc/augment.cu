// augment.cu -- training-time augmentation (Eigen et al. 2014, section 3.3), beyond the reference (it has none).  See
// a3d_augment_desc in include/a3d.h for the transform contract; oracle/augment.py restates it in float64.
//
// a3d_augment_draw: one thread per image, float64, writes the packed [B][16] parameter rows.
// a3d_resize_affine_tf1_s2d / a3d_resize_affine_tf1: the TF1 resizes with the source position of every output pixel passed
// through the image's affine map.  The normalised matrix is folded into per-tensor pixel coefficients
//   x = M00 u + M01 (W/H) v + M02 W,   y = M10 (H/W) u + M11 v + M12 H
// evaluated as two fmaf, so identity parameters give x = u, y = v exactly and the kernels reproduce the plain resizes bit
// for bit (same tf1_lerp, same value scaling order).  A rotated window has no row structure to stage, so every output
// pixel gathers its four neighbours through L1: neighbouring threads sample neighbouring source positions.
#include "common.cuh"
#include <math.h>

namespace {

__device__ __forceinline__ uint64_t aug_mix64(uint64_t x) {   // splitmix64 finaliser (as bernoulli_mask_kernel)
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

constexpr int kDraws = 8;            // uniforms per image: scale, theta, c_x, c_y, flip, c_r, c_g, c_b

__global__ void augment_draw_kernel(a3d_augment_desc d, int B, uint64_t seed, const int64_t* __restrict__ counter,
                                    float* __restrict__ params) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const uint64_t base = aug_mix64(seed ^ aug_mix64((uint64_t)(counter ? *counter : 0)));
  double u[kDraws];
#pragma unroll
  for (int j = 0; j < kDraws; ++j)
    u[j] = (double)(aug_mix64(base + (uint64_t)b * kDraws + j) >> 11) * 0x1.0p-53;   // [0, 1), 53 bits
  const double s = (double)d.scale_lo + ((double)d.scale_hi - (double)d.scale_lo) * u[0];
  const double theta = (double)d.max_rotation_deg * (2.0 * u[1] - 1.0);
  const double k = (double)d.crop_fraction / s;
  const double half = 0.5 * (1.0 - k);
  const double cx = 0.5 + half * (2.0 * u[2] - 1.0), cy = 0.5 + half * (2.0 * u[3] - 1.0);
  const bool flip = u[4] < (double)d.flip_prob;
  const double fl = flip ? -1.0 : 1.0;
  const double rad = theta * (M_PI / 180.0);
  const double cs = cos(rad), sn = sin(rad), a = (double)d.aspect;
  const double m00 = cs * fl * k, m01 = -sn * a * k;
  const double m10 = sn / a * fl * k, m11 = cs * k;
  float* p = params + (size_t)b * A3D_AUG_PARAMS;
  p[A3D_AUG_M00] = (float)m00;
  p[A3D_AUG_M01] = (float)m01;
  p[A3D_AUG_M02] = (float)(cx - 0.5 * (m00 + m01));
  p[A3D_AUG_M10] = (float)m10;
  p[A3D_AUG_M11] = (float)m11;
  p[A3D_AUG_M12] = (float)(cy - 0.5 * (m10 + m11));
  for (int c = 0; c < 3; ++c)
    p[A3D_AUG_COLOR + c] = (float)((double)d.color_lo + ((double)d.color_hi - (double)d.color_lo) * u[5 + c]);
  p[A3D_AUG_INV_SCALE] = (float)(1.0 / s);
  p[A3D_AUG_SCALE] = (float)s;
  p[A3D_AUG_THETA] = (float)theta;
  p[A3D_AUG_FLIP] = flip ? 1.f : 0.f;
  p[A3D_AUG_CX] = (float)cx;
  p[A3D_AUG_CY] = (float)cy;
  p[A3D_AUG_CROP] = d.crop_fraction;
}

// The image's map in this tensor's source pixels: x = ax u + bx v + cx, y = ay u + by v + cy.
struct PixelMap {
  float ax, bx, cx, ay, by, cy;
  __device__ __forceinline__ PixelMap(const float* __restrict__ p, int H, int W) {
    const float wh = (float)W / (float)H, hw = (float)H / (float)W;
    ax = __ldg(p + A3D_AUG_M00);
    bx = __ldg(p + A3D_AUG_M01) * wh;
    cx = __ldg(p + A3D_AUG_M02) * (float)W;
    ay = __ldg(p + A3D_AUG_M10) * hw;
    by = __ldg(p + A3D_AUG_M11);
    cy = __ldg(p + A3D_AUG_M12) * (float)H;
  }
};

// TF1 bilinear sample position of (u, v) after the map: corner indices and weights, border clamped.
struct Tap {
  int x0, x1, y0, y1;
  float lx, ly;
  __device__ __forceinline__ Tap(const PixelMap& m, float u, float v, int H, int W) {
    float x = fmaf(m.ax, u, fmaf(m.bx, v, m.cx));
    float y = fmaf(m.ay, u, fmaf(m.by, v, m.cy));
    x = fminf(fmaxf(x, 0.f), (float)(W - 1));
    y = fminf(fmaxf(y, 0.f), (float)(H - 1));
    x0 = (int)floorf(x);
    y0 = (int)floorf(y);
    x1 = min(x0 + 1, W - 1);
    y1 = min(y0 + 1, H - 1);
    lx = x - x0;
    ly = y - y0;
  }
};

template <typename T>
__device__ __forceinline__ float ld_src(const T* p) { return (float)__ldg(p); }

// One thread = one row of a 4x4 space-to-depth block: 4 resized pixels x 3 channels (as resize_bilinear_tf1_s2d4c3_kernel).
// The dy == 0 thread zeroes the padding channels [48, dstC).
template <typename TS, bool OUT_BF16>
__global__ void __launch_bounds__(256)
resize_affine_s2d4c3_kernel(const TS* __restrict__ src, int B, int H, int W, void* __restrict__ dst, int OH, int OWs,
                            int dstC, float sy, float sx, float scale, const float* __restrict__ params) {
  const size_t total = (size_t)B * OH * OWs;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int X = (int)(i % OWs);
    const size_t t = i / OWs;
    const int oy = (int)(t % OH);
    const int b = (int)(t / OH);
    const float* p = params + (size_t)b * A3D_AUG_PARAMS;
    const PixelMap m(p, H, W);
    const float col[3] = {__ldg(p + A3D_AUG_COLOR) , __ldg(p + A3D_AUG_COLOR + 1), __ldg(p + A3D_AUG_COLOR + 2)};
    const float v = oy * sy;
    const TS* img = src + (size_t)b * H * W * 3;
    float r[12];
#pragma unroll
    for (int dx = 0; dx < 4; ++dx) {
      const Tap q(m, (X * 4 + dx) * sx, v, H, W);
      const TS* r0 = img + (size_t)q.y0 * W * 3;
      const TS* r1 = img + (size_t)q.y1 * W * 3;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float tl = ld_src(r0 + q.x0 * 3 + c), tr = ld_src(r0 + q.x1 * 3 + c);
        const float bl = ld_src(r1 + q.x0 * 3 + c), br = ld_src(r1 + q.x1 * 3 + c);
        r[dx * 3 + c] = (tf1_lerp(tl, tr, bl, br, q.ly, q.lx) * scale) * col[c];
      }
    }
    const int Y = oy >> 2, dy = oy & 3;
    const size_t pix = ((size_t)b * (OH >> 2) + Y) * OWs + X;
    if (OUT_BF16) {
      uint16_t* o = reinterpret_cast<uint16_t*>(dst) + pix * dstC;
      uint2* o8 = reinterpret_cast<uint2*>(o + dy * 12);
      o8[0] = make_uint2(pack_bf16x2(r[0], r[1]), pack_bf16x2(r[2], r[3]));
      o8[1] = make_uint2(pack_bf16x2(r[4], r[5]), pack_bf16x2(r[6], r[7]));
      o8[2] = make_uint2(pack_bf16x2(r[8], r[9]), pack_bf16x2(r[10], r[11]));
      if (dy == 0)
        for (int k = 48; k < dstC; k += 4) *reinterpret_cast<uint2*>(o + k) = make_uint2(0u, 0u);
    } else {
      float* o = reinterpret_cast<float*>(dst) + pix * dstC;
      float4* o4 = reinterpret_cast<float4*>(o + dy * 12);
      o4[0] = make_float4(r[0], r[1], r[2], r[3]);
      o4[1] = make_float4(r[4], r[5], r[6], r[7]);
      o4[2] = make_float4(r[8], r[9], r[10], r[11]);
      if (dy == 0)
        for (int k = 48; k < dstC; k += 4) *reinterpret_cast<float4*>(o + k) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
}

// Generic NHWC, C <= 4, one thread per output pixel (as resize_bilinear_tf1_kernel).
template <bool DEPTH>
__global__ void __launch_bounds__(256)
resize_affine_kernel(const float* __restrict__ src, int B, int H, int W, int C, float* __restrict__ dst, int OH, int OW,
                     float sy, float sx, const float* __restrict__ params) {
  const size_t total = (size_t)B * OH * OW;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int ox = (int)(i % OW);
    const size_t t = i / OW;
    const int oy = (int)(t % OH);
    const int b = (int)(t / OH);
    const float* p = params + (size_t)b * A3D_AUG_PARAMS;
    const PixelMap m(p, H, W);
    const Tap q(m, ox * sx, oy * sy, H, W);
    const float* r0 = src + ((size_t)b * H + q.y0) * W * C;
    const float* r1 = src + ((size_t)b * H + q.y1) * W * C;
    for (int c = 0; c < C; ++c) {
      const float tl = __ldg(r0 + (size_t)q.x0 * C + c), tr = __ldg(r0 + (size_t)q.x1 * C + c);
      const float bl = __ldg(r1 + (size_t)q.x0 * C + c), br = __ldg(r1 + (size_t)q.x1 * C + c);
      const float f = DEPTH ? __ldg(p + A3D_AUG_INV_SCALE) : __ldg(p + A3D_AUG_COLOR + c);
      dst[i * C + c] = tf1_lerp(tl, tr, bl, br, q.ly, q.lx) * f;
    }
  }
}

int grid_for_aug(a3d_ctx* ctx, size_t work, int block) {
  size_t blocks = (work + block - 1) / block, cap = (size_t)ctx->sm_count * 8 * (2048 / block);
  if (blocks > cap) blocks = cap;
  return (int)(blocks < 1 ? 1 : blocks);
}

}  // namespace

extern "C" int a3d_augment_draw(a3d_ctx* ctx, const a3d_augment_desc* desc, int B, uint64_t seed,
                                const int64_t* counter_dev, float* params, void* stream) {
  A3D_REQUIRE(ctx && desc && params && B > 0, "augment_draw: bad argument");
  const a3d_augment_desc d = *desc;
  A3D_REQUIRE(d.scale_lo > 0.f && d.scale_lo <= d.scale_hi && d.crop_fraction > 0.f && d.crop_fraction <= 1.f &&
                  d.flip_prob >= 0.f && d.flip_prob <= 1.f && d.color_lo <= d.color_hi && d.max_rotation_deg >= 0.f &&
                  d.aspect > 0.f,
              "augment_draw: bad ranges (0 < scale_lo <= scale_hi, 0 < crop_fraction <= 1, flip_prob in [0, 1], "
              "color_lo <= color_hi, max_rotation_deg >= 0, aspect > 0)");
  augment_draw_kernel<<<ceil_div(B, 128), 128, 0, as_stream(stream)>>>(d, B, seed, counter_dev, params);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

extern "C" int a3d_resize_affine_tf1_s2d(a3d_ctx* ctx, const void* src, int src_dtype, int B, int H, int W, int C,
                                         void* dst, int dst_dtype, int OH, int OW, int s, int dstC, const float* params,
                                         void* stream) {
  A3D_REQUIRE(ctx && src && dst && params, "resize_affine_s2d: null argument");
  A3D_REQUIRE(B > 0 && H > 0 && W > 0 && C == 3 && s == 4 && OH % 4 == 0 && OW % 4 == 0 && dstC % 4 == 0 &&
                  dstC >= 48 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0 &&
                  (src_dtype == A3D_F32 || src_dtype == A3D_U8) && (dst_dtype == A3D_F32 || dst_dtype == A3D_BF16),
              "resize_affine_s2d: needs C == 3, s == 4, OH and OW multiples of 4, dstC %% 4 == 0 and >= 48, 16-byte "
              "aligned dst, src F32|U8, dst BF16|F32");
  const size_t rows = (size_t)B * OH * (OW / 4);
  const int block = 256, grid = grid_for_aug(ctx, rows, block);
  // the scale is formed in float like TF's CalculateResizeScale (as the plain kernels)
  const float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  cudaStream_t st = as_stream(stream);
  if (src_dtype == A3D_U8) {
    if (dst_dtype == A3D_BF16)
      resize_affine_s2d4c3_kernel<uint8_t, true><<<grid, block, 0, st>>>(
          static_cast<const uint8_t*>(src), B, H, W, dst, OH, OW / 4, dstC, sy, sx, 1.f / 255.f, params);
    else
      resize_affine_s2d4c3_kernel<uint8_t, false><<<grid, block, 0, st>>>(
          static_cast<const uint8_t*>(src), B, H, W, dst, OH, OW / 4, dstC, sy, sx, 1.f / 255.f, params);
  } else {
    if (dst_dtype == A3D_BF16)
      resize_affine_s2d4c3_kernel<float, true><<<grid, block, 0, st>>>(
          static_cast<const float*>(src), B, H, W, dst, OH, OW / 4, dstC, sy, sx, 1.f, params);
    else
      resize_affine_s2d4c3_kernel<float, false><<<grid, block, 0, st>>>(
          static_cast<const float*>(src), B, H, W, dst, OH, OW / 4, dstC, sy, sx, 1.f, params);
  }
  A3D_LAUNCH_OK(ctx);
  return 0;
}

extern "C" int a3d_resize_affine_tf1(a3d_ctx* ctx, const float* src, int B, int H, int W, int C, float* dst, int OH,
                                     int OW, const float* params, int value_mode, void* stream) {
  A3D_REQUIRE(ctx && src && dst && params, "resize_affine: null argument");
  A3D_REQUIRE(B > 0 && H > 0 && W > 0 && OH > 0 && OW > 0 && C > 0 && C <= 4 &&
                  (value_mode == A3D_AUG_VALUE_DEPTH || (value_mode == A3D_AUG_VALUE_COLOR && C <= 3)),
              "resize_affine: needs 0 < C <= 4 (C <= 3 for the colour rule) and value_mode COLOR|DEPTH");
  const size_t total = (size_t)B * OH * OW;
  const int block = 256, grid = grid_for_aug(ctx, total, block);
  const float sy = (float)H / (float)OH, sx = (float)W / (float)OW;
  if (value_mode == A3D_AUG_VALUE_DEPTH)
    resize_affine_kernel<true><<<grid, block, 0, as_stream(stream)>>>(src, B, H, W, C, dst, OH, OW, sy, sx, params);
  else
    resize_affine_kernel<false><<<grid, block, 0, as_stream(stream)>>>(src, B, H, W, C, dst, OH, OW, sy, sx, params);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

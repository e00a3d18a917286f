// common.cuh -- context, error plumbing and small device helpers shared by all liba3d sources.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/a3d.h"

struct a3d_ctx {
  int device;
  int sm_count;
  uint64_t launches;
  // driver entry points (resolved with cudaGetDriverEntryPoint; no link-time libcuda dependency)
  void* fn_encode_tiled;
  void* fn_encode_im2col;
  int driver_version;
  // NCCL (dlopen)
  void* nccl_lib;
  void* nccl_comm;
  int nranks;
};

void a3d_set_error(const char* fmt, ...);

#define A3D_CHECK_CUDA(expr)                                                            \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      a3d_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return (int)_e;                                                                   \
    }                                                                                   \
  } while (0)

#define A3D_REQUIRE(cond, ...)                                                          \
  do {                                                                                  \
    if (!(cond)) {                                                                      \
      a3d_set_error(__VA_ARGS__);                                                       \
      return A3D_EINVAL;                                                                \
    }                                                                                   \
  } while (0)

// after a kernel launch
#define A3D_LAUNCH_OK(ctx)                                                              \
  do {                                                                                  \
    (ctx)->launches++;                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) {                                                            \
      a3d_set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return (int)_e;                                                                   \
    }                                                                                   \
  } while (0)

static inline cudaStream_t as_stream(void* s) { return (cudaStream_t)s; }
static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ float bf16_bits_to_f32(uint16_t b) {
  return __uint_as_float(((uint32_t)b) << 16);
}
__device__ __forceinline__ uint16_t f32_to_bf16_bits(float f) {
  __nv_bfloat16 h = __float2bfloat16_rn(f);
  return *reinterpret_cast<uint16_t*>(&h);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  return (uint32_t)f32_to_bf16_bits(lo) | ((uint32_t)f32_to_bf16_bits(hi) << 16);
}

// Flat index -> (n, h, w, c) of an [N][H][W][C] grid.  64-bit div/mod costs ~100 instructions each and made the
// pool / col2im kernels index-math-bound (pool backward: 21 us for 33 MB); every MSDN tensor has < 2^32 elements,
// so the 32-bit path is the one taken.
__device__ __forceinline__ void split_nhwc(size_t i, int H, int W, int C, int& n, int& h, int& w, int& c) {
  if (i <= 0xffffffffull) {
    uint32_t u = (uint32_t)i;
    uint32_t q = u / (uint32_t)C; c = (int)(u - q * (uint32_t)C); u = q;
    q = u / (uint32_t)W; w = (int)(u - q * (uint32_t)W); u = q;
    q = u / (uint32_t)H; h = (int)(u - q * (uint32_t)H); n = (int)q;
  } else {
    c = (int)(i % C); size_t t = i / C;
    w = (int)(t % W); t /= W;
    h = (int)(t % H); n = (int)(t / H);
  }
}
__device__ __forceinline__ void split_rc(size_t i, int C, size_t& r, int& c) {
  if (i <= 0xffffffffull) {
    uint32_t u = (uint32_t)i, q = u / (uint32_t)C;
    r = q; c = (int)(u - q * (uint32_t)C);
  } else {
    r = i / C; c = (int)(i - r * C);
  }
}

// TF1 legacy bilinear mapping (tf.image.resize_images, align_corners=False): source coordinate = dst * (in/out),
// lo = floor, hi = min(lo+1, in-1), weight = coordinate - lo.  Shared by a3d_resize_bilinear_tf1 and
// a3d_depth_metrics, which samples the prediction at ground-truth pixels and must see the resize's values bit for bit.
__device__ __forceinline__ void tf1_coord(int o, float scale, int in, int& lo, int& hi, float& w) {
  float f = o * scale;
  lo = (int)floorf(f);
  hi = min(lo + 1, in - 1);
  w = f - lo;
}
__device__ __forceinline__ float tf1_lerp(float tl, float tr, float bl, float br, float ly, float lx) {
  float top = tl + (tr - tl) * lx;
  float bot = bl + (br - bl) * lx;
  return top + (bot - top) * ly;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// internal cross-file entry points
int a3d_tc_conv_fwd_supported(const a3d_conv_desc* d);
int a3d_simt_conv_fwd(a3d_ctx*, const a3d_conv_desc*, const uint16_t* x, const uint16_t* w, const float* bias,
                      void* y, int y_dtype, unsigned flags, cudaStream_t st);
int a3d_simt_conv_dgrad(a3d_ctx*, const a3d_conv_desc*, const uint16_t* dy, const uint16_t* w, uint16_t* dx,
                        cudaStream_t st);
int a3d_simt_conv_wgrad(a3d_ctx*, const a3d_conv_desc*, const uint16_t* x, const uint16_t* dy, float* dw,
                        cudaStream_t st);
int a3d_colsum_bf16(a3d_ctx*, const uint16_t* a, size_t rows, int C, int ld, float* out, cudaStream_t st);
int a3d_colsum_bf16_grouped(a3d_ctx*, const uint16_t* a, int rows, int C, int ld, int gb, size_t gs, float* out,
                            cudaStream_t st);
int a3d_simt_dense_fwd(a3d_ctx*, const uint16_t* x, int ldx, const uint16_t* w, const float* bias, const uint8_t* mask,
                       float drop_rate, void* y, int y_dtype, int M, int N, int K, unsigned flags, cudaStream_t st);
int a3d_simt_dense_dgrad(a3d_ctx*, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx, int M, int N, int K,
                         cudaStream_t st);
int a3d_simt_dense_wgrad(a3d_ctx*, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* dw, int M, int N,
                         int K, cudaStream_t st);

// dense_stream.cu: weight-streaming mma.sync kernels (batch <= 32 dense layers, single-filter convolution)
bool a3d_stream_dense_fwd_ok(int M, int N, int K, int ldx);
bool a3d_stream_dense_dgrad_ok(int M, int N, int K, int lddy);
int a3d_stream_dense_fwd(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* w, float* acc, int M, int N, int K,
                         int ctas, cudaStream_t st);
int a3d_stream_dense_dgrad(a3d_ctx* ctx, const uint16_t* dy, int lddy, const uint16_t* w, float* acc, int M, int N, int K,
                           int ctas, cudaStream_t st);
bool a3d_conv_k1_tiled_ok(const a3d_conv_desc* d);
int a3d_conv_k1_tiled(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* x, const uint16_t* w, const float* bias,
                      void* y, int y_dtype, unsigned flags, cudaStream_t st);

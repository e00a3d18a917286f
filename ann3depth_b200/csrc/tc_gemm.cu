// tc_gemm.cu -- host side of the tcgen05 GEMM engine: tensor-map construction, tile/split selection
// and the launchers used by the convolution / dense entry points.
#include "tc_gemm.cuh"
#include "tc_pair.cuh"
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                   CUtensorMapFloatOOBfill);

CUtensorMapSwizzle swizzle_for(int row_bytes) {
  return row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
         : row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
         : row_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                           : CU_TENSOR_MAP_SWIZZLE_NONE;
}

// Operand element type of a tensor map: 2 = bf16; 1 = E4M3; 4 = f32 read as TFLOAT32 -- the TMA unit rounds the low 13 mantissa
// bits away (round to nearest) on the way into shared memory, so kind::tf32 MMAs see properly rounded TF32 values
// instead of truncated ones.
CUtensorMapDataType tmap_dtype(int elt) {
  if (elt == 2) return CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  if (elt == 1) return CU_TENSOR_MAP_DATA_TYPE_UINT8;       // E4M3 codes: the TMA unit only moves the bytes
  return CU_TENSOR_MAP_DATA_TYPE_TFLOAT32;
}

// 2-D operand tensor [rows][cols] (cols contiguous, row pitch ld elements of `elt` bytes); box = box_cols x box_rows.
// mn_major: the operand is consumed MN-major; for 4-byte elements that needs the 32-byte-atom variant of the 128-byte swizzle.
int make_tmap_2d(a3d_ctx* ctx, CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                 uint32_t box_cols, uint32_t box_rows, int elt = 2, bool mn_major = false) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * (uint64_t)elt};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides[0] & 15)) {
    a3d_set_error("tensor map: base %p / row pitch %llu B not 16-byte aligned", base, (unsigned long long)strides[0]);
    return A3D_EINVAL;
  }
  CUresult r = reinterpret_cast<EncodeTiledFn>(ctx->fn_encode_tiled)(
      tm, tmap_dtype(elt), 2, const_cast<void*>(base), dims, strides, box, estr,
      CU_TENSOR_MAP_INTERLEAVE_NONE, (elt == 4 && mn_major) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : swizzle_for(box_cols * elt),
      CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    a3d_set_error("cuTensorMapEncodeTiled failed (%d): rows=%llu cols=%llu ld=%llu box=%ux%u", (int)r,
                  (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_cols, box_rows);
    return A3D_ETMAP;
  }
  return 0;
}

// Weight matrix [rows][ktot] viewed as {8, rows, ktot/8}: one box = 8 chunks x box_rows rows x 8 elements,
// landing chunk-major in shared memory (the "chunked" no-swizzle K-major layout of tc_gemm.cuh).
int make_tmap_chunked(a3d_ctx* ctx, CUtensorMap* tm, const void* base, uint64_t rows, uint64_t ktot, uint32_t box_rows) {
  cuuint64_t dims[3] = {8, rows, ktot / 8};
  cuuint64_t strides[2] = {ktot * 2, 16};
  cuuint32_t box[3] = {8, box_rows, 8};
  cuuint32_t estr[3] = {1, 1, 1};
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides[0] & 15) || (ktot % 8)) {
    a3d_set_error("chunked tensor map: base / row pitch not 16-byte aligned (ktot=%llu)", (unsigned long long)ktot);
    return A3D_EINVAL;
  }
  CUresult r = reinterpret_cast<EncodeTiledFn>(ctx->fn_encode_tiled)(
      tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    a3d_set_error("cuTensorMapEncodeTiled(chunked) failed (%d): rows=%llu ktot=%llu", (int)r, (unsigned long long)rows,
                  (unsigned long long)ktot);
    return A3D_ETMAP;
  }
  return 0;
}

// NHWC activation tensor (bf16, or f32 read as TF32) in im2col mode.  Base pixels run over lower + {0..P-1} * stride per axis.
// pix_pitch (elements, 0 = C): pixel pitch of an overlapped view -- pixel w's C channels start at w * pix_pitch, so
// consecutive pixels share C - pix_pitch channels (a3d_conv_desc::pix_pitch); rows and images are W and H*W pitches apart
int make_tmap_im2col(a3d_ctx* ctx, CUtensorMap* tm, const void* base, int N, int H, int W, int C, int lower_h,
                     int lower_w, int P, int Q, int sh, int sw, uint32_t chan_box, uint32_t pixels, int elt = 2,
                     bool mn_major = false, int pix_pitch = 0) {
  const cuuint64_t pp = pix_pitch > 0 ? pix_pitch : C;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {pp * elt, (cuuint64_t)W * pp * elt, (cuuint64_t)H * W * pp * elt};
  // tightest bounding box that still contains the last base pixel (see DESIGN.md "im2col corners")
  int upper_w = lower_w + (Q - 1) * sw + 1 - W;
  int upper_h = lower_h + (P - 1) * sh + 1 - H;
  int lower[2] = {lower_w, lower_h};
  int upper[2] = {upper_w, upper_h};
  cuuint32_t estr[4] = {1, (cuuint32_t)sw, (cuuint32_t)sh, 1};
  for (int i = 0; i < 2; ++i)
    if (lower[i] < -128 || lower[i] > 127 || upper[i] < -128 || upper[i] > 127) {
      a3d_set_error("im2col tensor map: corner out of [-128,127] (lower %d,%d upper %d,%d)", lower_w, lower_h, upper_w,
                    upper_h);
      return A3D_ENOTSUP;
    }
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides[0] & 15)) {
    a3d_set_error("im2col tensor map: base/pixel pitch not 16-byte aligned (C=%d)", C);
    return A3D_EINVAL;
  }
  CUresult r = reinterpret_cast<EncodeIm2colFn>(ctx->fn_encode_im2col)(
      tm, tmap_dtype(elt), 4, const_cast<void*>(base), dims, strides, lower, upper, chan_box, pixels,
      estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
      (elt == 4 && mn_major) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : swizzle_for(chan_box * elt), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    a3d_set_error("cuTensorMapEncodeIm2col failed (%d): NHWC=%d,%d,%d,%d lower=%d,%d upper=%d,%d box=%u x %u", (int)r, N,
                  H, W, C, lower_w, lower_h, upper_w, upper_h, chan_box, pixels);
    return A3D_ETMAP;
  }
  // Driver quirk also worked around by CUTLASS (copy_traits_sm90_im2col.hpp): for tensors smaller
  // than 128 KiB, drivers <= 13.1 set a descriptor bit that makes im2col loads fault.
  if (ctx->driver_version <= 13010) {
    size_t bytes = (size_t)N * H * W * C * elt;
    if (bytes < 131072) reinterpret_cast<uint64_t*>(tm)[1] &= ~(1ull << 21);
  }
  return 0;
}

// f32 output matrix [rows][cols] (row pitch ld elements) for the TMA epilogue: box = 32 columns x 32 rows,
// SWIZZLE_128B (the staging slabs of tc::EPI_TMA_F32).
int make_tmap_out_f32(a3d_ctx* ctx, CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint64_t ld) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = reinterpret_cast<EncodeTiledFn>(ctx->fn_encode_tiled)(
      tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    a3d_set_error("cuTensorMapEncodeTiled(out f32) failed (%d): rows=%llu cols=%llu ld=%llu", (int)r,
                  (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld);
    return A3D_ETMAP;
  }
  return 0;
}

// bf16 output matrix for the TMA epilogue: box = 64 columns (128 bytes) x 32 rows, SWIZZLE_128B
int make_tmap_out_bf16(a3d_ctx* ctx, CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint64_t ld) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {64, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = reinterpret_cast<EncodeTiledFn>(ctx->fn_encode_tiled)(
      tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    a3d_set_error("cuTensorMapEncodeTiled(out bf16) failed (%d): rows=%llu cols=%llu ld=%llu", (int)r,
                  (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld);
    return A3D_ETMAP;
  }
  return 0;
}

// The TMA epilogue wherever the output is an f32 row-major matrix with 16-byte aligned rows; the per-thread register
// epilogue otherwise.
bool epi_tma_ok(const void* out, long long ldo) {
  return (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (ldo % 4) == 0;
}
// switch a row-major f32 epilogue to the TMA epilogue when possible; builds the output map
int maybe_tma_out(a3d_ctx* ctx, tc::Params& p, CUtensorMap* tmC, bool* use) {
  *use = false;
  if (p.epi == tc::EPI_POOL4_BF16) {           // 64 pooled columns; the caller checked alignment
    int rc = make_tmap_out_bf16(ctx, tmC, p.out, (uint64_t)p.M, 64, (uint64_t)p.ldo);
    if (rc) return rc;
    *use = true;
    return 0;
  }
  if (p.epi == tc::EPI_ROW_F32 && epi_tma_ok(p.out, p.ldo)) {
    int rc = make_tmap_out_f32(ctx, tmC, p.out, (uint64_t)p.M, (uint64_t)p.N, (uint64_t)p.ldo);
    if (rc) return rc;
    p.epi = tc::EPI_TMA_F32;
    *use = true;
  } else if (p.epi == tc::EPI_ROW_BF16 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0 &&
             (p.ldo % 8) == 0) {
    int rc = make_tmap_out_bf16(ctx, tmC, p.out, (uint64_t)p.M, (uint64_t)p.N, (uint64_t)p.ldo);
    if (rc) return rc;
    p.epi = tc::EPI_TMA_BF16;
    *use = true;
  }
  return 0;
}

template <class C>
int launch_cfg(a3d_ctx* ctx, const CUtensorMap& tmA, const CUtensorMap& tmB, const tc::Params& p_in, int splits,
               cudaStream_t st) {
  static_assert(C::STAGES * C::STAGE_BYTES >= 4 * 8192, "the TMA epilogue stages 4 x 8 KB in the ring");
  static bool attr_set = false;
  if (!attr_set) {
    A3D_CHECK_CUDA(cudaFuncSetAttribute(tc::gemm_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set = true;
  }
  tc::Params p = p_in;
  CUtensorMap tmC;
  bool use_c = false;
  int rc = maybe_tma_out(ctx, p, &tmC, &use_c);
  if (rc) return rc;
  dim3 grid(ceil_div(p.M, C::BM), ceil_div(p.N, C::BN), splits);
  tc::gemm_kernel<C><<<grid, 192, C::SMEM_BYTES, st>>>(tmA, tmB, use_c ? tmC : tmA, p);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// K-major x K-major dispatch over (BN, KCB) and the tile variant:
//   0  128-row tile, default ring (tc_gemm.cuh A3D_RING_KB / A3D_MIN_STAGES: most CTAs per SM)
//   1  128-row tile, one stage more (long main loops -- conv2d_1 dgrad has 100 k-blocks -- want the deeper pipeline)
//   2  256-row tile (two accumulators sharing every B stage: less L2->SM operand traffic), default ring
//   3  256-row tile, three stages
//   4..10 (removed) round-1 experiments that lost on every MSDN layer once measured on hardware: a persistent tile loop
//         with double-buffered TMEM accumulators, and a cluster kernel that TMA-multicast the weight tile to 2 / 4 CTAs
//   11,12 CTA-pair kernel (tc_pair.cuh): tcgen05.mma.cta_group::2, 256 x BN tile per pair, each CTA holds half the
//         weight tile; 11 = short ring (two CTAs per SM), 12 = deep ring (one CTA per SM).  tmB box = BN / 2 rows.
enum { V_BASE = 0, V_DEEP = 1, V_BM256 = 2, V_BM256_DEEP = 3, V_PAIR = 11, V_PAIR_DEEP = 12, V_COUNT = 13 };
// CTAs that share one B tile: the pair kernel's tensor map for B has a box of BN / 2 rows
int mcast_cl(int variant) { return variant == V_PAIR || variant == V_PAIR_DEEP ? 2 : 1; }
template <class C>
int launch_pair(a3d_ctx* ctx, const CUtensorMap& tmA, const CUtensorMap& tmB_half, const tc::Params& p_in, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    A3D_CHECK_CUDA(cudaFuncSetAttribute(tc::gemm_pair_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
    attr_set = true;
  }
  tc::Params p = p_in;
  if (p.atomic || p.kb_per_split < p.num_kb) { a3d_set_error("pair gemm: no split-K"); return A3D_ENOTSUP; }
  CUtensorMap tmC;
  bool use_c = false;
  int rc = maybe_tma_out(ctx, p, &tmC, &use_c);
  if (rc) return rc;
  const bool ok = use_c && ((p.epi == tc::EPI_TMA_F32 && C::BN % 32 == 0) || (p.epi == tc::EPI_TMA_BF16 && C::BN % 64 == 0) ||
                           (p.epi == tc::EPI_POOL4_BF16 && C::BN == 256));
  if (!ok) { a3d_set_error("pair gemm: needs a TMA-store epilogue (f32: BN %% 32, bf16: BN %% 64)"); return A3D_ENOTSUP; }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(ceil_div(ceil_div(p.M, 128), 2) * 2, ceil_div(p.N, C::BN), 1);
  cfg.blockDim = dim3(192, 1, 1);
  cfg.dynamicSmemBytes = C::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  A3D_CHECK_CUDA(cudaLaunchKernelEx(&cfg, tc::gemm_pair_kernel<C>, tmA, tmB_half, tmC, p));
  A3D_LAUNCH_OK(ctx);
  return 0;
}

int launch_kk(a3d_ctx* ctx, int bn, int kcb, const CUtensorMap& tmA, const CUtensorMap& tmB, const tc::Params& p,
              int splits, cudaStream_t st, int variant = V_BASE) {
  if (variant == V_BASE) {
#define A3D_CASE(BN, KCB) \
  if (bn == BN && kcb == KCB) return launch_cfg<tc::Cfg<BN, KCB, false, false>>(ctx, tmA, tmB, p, splits, st);
    A3D_CASE(32, 128) A3D_CASE(64, 128) A3D_CASE(96, 128) A3D_CASE(128, 128) A3D_CASE(192, 128) A3D_CASE(256, 128)
    A3D_CASE(32, 64) A3D_CASE(64, 64) A3D_CASE(96, 64) A3D_CASE(128, 64) A3D_CASE(192, 64) A3D_CASE(256, 64)
    A3D_CASE(32, 32) A3D_CASE(64, 32) A3D_CASE(96, 32) A3D_CASE(128, 32) A3D_CASE(256, 32)
    A3D_CASE(16, 128) A3D_CASE(16, 64) A3D_CASE(16, 32)
    A3D_CASE(32, 16) A3D_CASE(64, 16) A3D_CASE(96, 16) A3D_CASE(128, 16)
#undef A3D_CASE
  } else if (kcb == 128) {
#define A3D_CASEV(V, BN, MS, BM) \
  if (variant == V && bn == BN) \
    return launch_cfg<tc::Cfg<BN, 128, false, false, 64, MS, false, BM>>(ctx, tmA, tmB, p, splits, st);
    A3D_CASEV(V_DEEP, 64, 4, 128) A3D_CASEV(V_DEEP, 96, 3, 128) A3D_CASEV(V_DEEP, 128, 3, 128)
    A3D_CASEV(V_DEEP, 192, 3, 128) A3D_CASEV(V_DEEP, 256, 3, 128)
    A3D_CASEV(V_BM256, 64, 2, 256) A3D_CASEV(V_BM256, 96, 2, 256) A3D_CASEV(V_BM256, 128, 2, 256)
    A3D_CASEV(V_BM256, 256, 2, 256)
    A3D_CASEV(V_BM256_DEEP, 64, 3, 256) A3D_CASEV(V_BM256_DEEP, 96, 3, 256) A3D_CASEV(V_BM256_DEEP, 128, 3, 256)
    A3D_CASEV(V_BM256_DEEP, 256, 3, 256)
#undef A3D_CASEV
#define A3D_CASE2(BN, NS, ND) \
  if (bn == BN) { \
    if (variant == V_PAIR) return launch_pair<tc::PairCfg<BN, 128, NS>>(ctx, tmA, tmB, p, st); \
    return launch_pair<tc::PairCfg<BN, 128, ND>>(ctx, tmA, tmB, p, st); \
  }
    if ((variant == V_PAIR || variant == V_PAIR_DEEP) && splits == 1) {
      A3D_CASE2(64, 4, 8) A3D_CASE2(96, 4, 8) A3D_CASE2(128, 4, 8) A3D_CASE2(192, 3, 7) A3D_CASE2(256, 3, 6)
    }
#undef A3D_CASE2
  }
  a3d_set_error("tc gemm: no kernel for BN=%d KCB=%d variant=%d", bn, kcb, variant);
  return A3D_ENOTSUP;
}
bool variant_exists(int bn, int kcb, int variant) {
  if (variant == V_BASE) return true;
  if (kcb != 128) return false;
  if (variant == V_DEEP) return bn == 64 || bn == 96 || bn == 128 || bn == 192 || bn == 256;
  if (variant == V_PAIR || variant == V_PAIR_DEEP) return bn == 64 || bn == 96 || bn == 128 || bn == 192 || bn == 256;
  if (variant > V_BM256_DEEP) return false;
  return bn == 64 || bn == 96 || bn == 128 || bn == 256;
}

int pick_bn(int n) {
  if (n <= 16) return 16;
  if (n <= 32) return 32;
  if (n <= 64) return 64;
  if (n <= 96) return 96;
  if (n <= 128) return 128;
  if (n % 192 == 0 && n % 128 != 0) return 192;
  return 128;
}

// how many K splits give roughly >= 1 wave of CTAs without starving each split
int pick_splits(a3d_ctx* ctx, int tiles, int num_kb, int min_kb_per_split) {
  if (tiles >= ctx->sm_count * 3 / 4) return 1;
  int s = (ctx->sm_count + tiles - 1) / tiles;
  int max_s = num_kb / min_kb_per_split;
  if (max_s < 1) max_s = 1;
  if (s > max_s) s = max_s;
  return s < 1 ? 1 : s;
}

__global__ void bias_act_cast_kernel(const float* __restrict__ acc, const float* __restrict__ bias,
                                     const uint8_t* __restrict__ mask, float drop_scale, void* __restrict__ y, int y_f32,
                                     size_t rows, int n, long long ldy, unsigned flags) {
  size_t total = rows * n;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    size_t r; int c;
    split_rc(i, n, r, c);
    float v = acc[i];
    if (bias) v += bias[c];
    if (flags & A3D_EPI_RELU) v = fmaxf(v, 0.f);
    if (flags & A3D_EPI_SIGMOID) v = 1.f / (1.f + expf(-v));
    if (mask) v = mask[i] ? v * drop_scale : 0.f;
    if (y_f32) reinterpret_cast<float*>(y)[r * ldy + c] = v;
    else reinterpret_cast<uint16_t*>(y)[r * ldy + c] = f32_to_bf16_bits(v);
  }
}

// dense dgrad finish with the producer layer's activation gradient folded in (DropoutGrad, then ReluGrad / SigmoidGrad on
// the stored post-activation value y): dx = bf16(act'(y) * mask/(1-rate) * acc).  Same arithmetic as the separate
// dense_epilogue_bwd pass it replaces (x 1/(1-rate) = x2 is exact in bf16), one kernel and one bf16 round trip less.
__global__ void act_bwd_cast_kernel(const float* __restrict__ acc, const uint16_t* __restrict__ y,
                                    const uint8_t* __restrict__ mask, float scale, uint16_t* __restrict__ dx, size_t n,
                                    unsigned flags) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float g = bf16_bits_to_f32(f32_to_bf16_bits(acc[i]));      // the separate pass saw the bf16-rounded dgrad
    if (mask) g = mask[i] ? g * scale : 0.f;
    const float yv = bf16_bits_to_f32(y[i]);
    if (flags & A3D_EPI_RELU) g = yv > 0.f ? g : 0.f;
    if (flags & A3D_EPI_SIGMOID) g = g * yv * (1.f - yv);
    dx[i] = f32_to_bf16_bits(g);
  }
}

int finish(a3d_ctx* ctx, const float* acc, const float* bias, const uint8_t* mask, float drop_rate, void* y, int y_f32,
           size_t rows, int n, long long ldy, unsigned flags, cudaStream_t st) {
  size_t total = rows * n;
  int block = 256;
  size_t blocks = (total + block - 1) / block;
  if (blocks > (size_t)ctx->sm_count * 16) blocks = (size_t)ctx->sm_count * 16;
  bias_act_cast_kernel<<<(int)blocks, block, 0, st>>>(acc, bias, mask, 1.f / (1.f - drop_rate), y, y_f32, rows, n, ldy,
                                                     flags);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

}  // namespace

// y[r][c] = act(acc[r][c] + bias[c]) (x dropout mask), f32 -- the finishing pass of the 3xTF32 sums (tf32_conv.cu)
int a3d_tc_finish_f32(a3d_ctx* ctx, const float* acc, const float* bias, const uint8_t* mask, float drop_rate, float* y,
                      size_t rows, int n, long long ldy, unsigned flags, cudaStream_t st) {
  return finish(ctx, acc, bias, mask, drop_rate, y, 1, rows, n, ldy, flags, st);
}

// ---- first-use autotuning -------------------------------------------------------------------------
// The best tile width / split-K factor of the small MSDN layers depends on how many CTAs end up co-resident
// and on wave quantisation in ways the closed-form heuristics above miss by up to 1.8x (profiles/sweep_r01_*).
// The first launch of a shape (outside stream capture) therefore times every candidate configuration with CUDA
// events on the launching stream and caches the winner; later launches -- including the captured ones of the
// CUDA graph -- reuse it.  Candidate runs overwrite the same output, so tuning has no side effects.
namespace {
struct TuneKey { int v[16]; };
struct TuneEntry { TuneKey key; int choice; };
TuneEntry g_tune[256];
int g_tune_n = 0;

// A3D_TUNE_CACHE=<file>: choices are appended to the file and read back by later processes, so that a run under a
// profiler (whose launch overhead distorts the candidate timings) uses exactly the configuration of the plain run.
// One line per shape: the 16 key integers, the number of candidates and the chosen index.
void tune_cache_load() {
  static bool loaded = false;
  if (loaded) return;
  loaded = true;
  const char* path = getenv("A3D_TUNE_CACHE");
  if (!path) return;
  FILE* f = fopen(path, "r");
  if (!f) return;
  TuneKey k;
  int ncand, choice;
  while (g_tune_n < 256) {
    int got = 0;
    for (int i = 0; i < 16; ++i) got += fscanf(f, "%d", &k.v[i]) == 1;
    if (got != 16 || fscanf(f, "%d %d", &ncand, &choice) != 2) break;
    g_tune[g_tune_n].key = k;
    g_tune[g_tune_n].choice = choice;
    ++g_tune_n;
  }
  fclose(f);
}
void tune_cache_store(const TuneKey& key, int ncand, int choice) {
  const char* path = getenv("A3D_TUNE_CACHE");
  if (!path) return;
  FILE* f = fopen(path, "a");
  if (!f) return;
  for (int i = 0; i < 16; ++i) fprintf(f, "%d ", key.v[i]);
  fprintf(f, "%d %d\n", ncand, choice);
  fclose(f);
}

// run(c) launches candidate c on `st`; returns the index of the fastest candidate (0 when tuning is unavailable).
// A3D_TUNE_PICK=i (read on every call, for tests that run every candidate of a shape): return i without timing, and
// neither read nor write the in-process or file cache.  i outside [0, ncand) returns -1 with the error set; the call
// site returns A3D_EINVAL.
template <class F>
int autotune(const TuneKey& key, int ncand, F run, cudaStream_t st) {
  if (const char* pick = getenv("A3D_TUNE_PICK")) {
    const int i = atoi(pick);
    if (i < 0 || i >= ncand) {
      a3d_set_error("A3D_TUNE_PICK=%d out of range: tuner kind %d has %d candidates for this shape", i, key.v[0], ncand);
      return -1;
    }
    return i;
  }
  tune_cache_load();
  for (int i = 0; i < g_tune_n; ++i)
    if (memcmp(&g_tune[i].key, &key, sizeof(TuneKey)) == 0) return g_tune[i].choice < ncand ? g_tune[i].choice : 0;
  if (ncand <= 1) return 0;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) return 0;
  cudaEvent_t e0, e1;
  if (cudaEventCreate(&e0) != cudaSuccess || cudaEventCreate(&e1) != cudaSuccess) return 0;
  int best = 0;
  float best_ms = 1e30f;
  constexpr int kReps = 10;                        // 3 repetitions left the choice between near-ties to timer noise
  const bool verbose = getenv("A3D_AUTOTUNE_VERBOSE") && atoi(getenv("A3D_AUTOTUNE_VERBOSE")) >= 2;
  for (int c = 0; c < ncand; ++c) {
    if (run(c) != 0) continue;                     // warm-up (function attributes, L2)
    cudaEventRecord(e0, st);
    bool ok = true;
    for (int r = 0; r < kReps && ok; ++r) ok = run(c) == 0;
    cudaEventRecord(e1, st);
    if (cudaEventSynchronize(e1) != cudaSuccess || !ok) continue;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    if (verbose) fprintf(stderr, "a3d autotune:   kind %d candidate %d: %.1f us\n", key.v[0], c, ms * 1e3f / kReps);
    if (ms < best_ms) { best_ms = ms; best = c; }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (g_tune_n < 256) { g_tune[g_tune_n].key = key; g_tune[g_tune_n].choice = best; ++g_tune_n; }
  tune_cache_store(key, ncand, best);
  if (getenv("A3D_AUTOTUNE_VERBOSE"))
    fprintf(stderr, "a3d autotune: kind %d [%d %d %d %d %d %d %d %d %d] -> candidate %d of %d (%.1f us)\n", key.v[0],
            key.v[1], key.v[2], key.v[3], key.v[4], key.v[5], key.v[6], key.v[7], key.v[8], key.v[9], best, ncand,
            best_ms * 1e3f / kReps);
  return best;
}
// split-K candidates for the weight-streaming dense kernels: the heuristic first, then CTA counts of
// 1, 1.5 and 2 x SM count (two CTAs are co-resident per SM; a partial extra wave doubles the time)
int split_candidates(a3d_ctx* ctx, int tiles, int num_kb, int heuristic, int* out) {
  int n = 0;
  out[n++] = heuristic;
  const int targets[4] = {ctx->sm_count, ctx->sm_count * 3 / 2, ctx->sm_count * 2, ctx->sm_count * 5 / 2};
  for (int t = 0; t < 4; ++t) {
    int s = targets[t] / tiles;
    const int max_s = num_kb / 4 > 0 ? num_kb / 4 : 1;
    if (s > max_s) s = max_s;
    if (s < 1) s = 1;
    bool dup = false;
    for (int k = 0; k < n; ++k) dup |= out[k] == s;
    if (!dup) out[n++] = s;
  }
  return n;
}
}  // namespace

// ------------------------------------------------------------------------------------------------
// convolution forward as an implicit GEMM: M = N*P*Q output pixels, N = K filters, K = R*S*C
int a3d_tc_conv_fwd_supported(const a3d_conv_desc* d) {
  if (d->C % 8) return 0;                        // im2col box needs >= 16 B of channels per pixel
  if (d->C % 16 && d->K > 128) return 0;         // 8-channel "chunked" kernels exist for K <= 128 only
  if (d->stride_h > 8 || d->stride_w > 8) return 0;
  if (d->R > 256 || d->S > 256) return 0;
  return 1;
}

size_t a3d_tc_conv_fwd_ws_bytes(a3d_ctx* ctx, const a3d_conv_desc* d) {
  // split-K accumulation buffer (only used when the tile count is far below one wave)
  return (size_t)d->N * d->P * d->Q * d->K * sizeof(float);
}

int a3d_tc_conv_fwd(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* x, const uint16_t* w, const float* bias,
                    void* y, int y_dtype, unsigned flags, void* ws, size_t ws_bytes, cudaStream_t st,
                    uint8_t* pool_idx) {
  if (flags & A3D_EPI_POOL4) {
    // conv + bias + act + 2x2 max-pool: the four window positions are four groups of 64 filters (K = 256)
    if (d->K != 256 || d->C % 64 || y_dtype != A3D_BF16 || d->ldy % 8 || (reinterpret_cast<uintptr_t>(y) & 15)) {
      a3d_set_error("tc conv pool4 fwd: needs K == 256 (4 x 64), C %% 64 == 0, bf16 output with 16-byte aligned rows");
      return A3D_ENOTSUP;
    }
    const int cblocks = d->C / 64;
    const long long M = (long long)d->N * d->P * d->Q;
    CUtensorMap tmA, tmB;
    int rc = make_tmap_im2col(ctx, &tmA, x, d->N, d->H, d->W, d->C, -d->pad_t, -d->pad_l, d->P, d->Q, d->stride_h,
                              d->stride_w, 64, 128, 2, false, d->pix_pitch);
    if (rc) return rc;
    rc = make_tmap_2d(ctx, &tmB, w, 256, (uint64_t)d->R * d->S * d->C, (uint64_t)d->R * d->S * d->C, 64, 256);
    if (rc) return rc;
    tc::Params p{};
    p.M = (int)M; p.N = 256; p.num_kb = d->R * d->S * cblocks; p.kb_per_split = p.num_kb;
    p.a_mode = tc::A_IM2COL;
    p.PQ = d->P * d->Q; p.Q = d->Q; p.sh = d->stride_h; p.sw = d->stride_w; p.lower_h = -d->pad_t; p.lower_w = -d->pad_l;
    p.S = d->S; p.cblocks = cblocks; p.dil_w = d->dil_w > 1 ? d->dil_w : 1;
    p.epi = tc::EPI_POOL4_BF16; p.out = y; p.ldo = d->ldy; p.bias = bias; p.flags = flags; p.pool_idx = pool_idx;
    // 128-row tiles with two stages of 48 KB (two CTAs per SM, one CTA's epilogue under the other's main loop),
    // the same with three stages, or 256-row tiles (both accumulators fill the 512 TMEM columns)
    auto run = [&](int c) -> int {
      if (c == 6 || c == 7) {                      // CTA pair (tc_pair.cuh): each CTA holds 128 of the 256 filter rows
        CUtensorMap tmBh;
        int r = make_tmap_2d(ctx, &tmBh, w, 256, (uint64_t)d->R * d->S * d->C, (uint64_t)d->R * d->S * d->C, 64, 128);
        if (r) return r;
        if (c == 6) return launch_pair<tc::PairCfg<256, 128, 3>>(ctx, tmA, tmBh, p, st);
        return launch_pair<tc::PairCfg<256, 128, 6>>(ctx, tmA, tmBh, p, st);
      }
      if (c == 1) return launch_cfg<tc::Cfg<256, 128, false, false, 64, 3>>(ctx, tmA, tmB, p, 1, st);
      if (c == 2) return launch_cfg<tc::Cfg<256, 128, false, false, 64, 2, false, 256>>(ctx, tmA, tmB, p, 1, st);
      if (c == 3) return launch_cfg<tc::Cfg<256, 128, false, false, 64, 3, false, 256>>(ctx, tmA, tmB, p, 1, st);
      return launch_cfg<tc::Cfg<256, 128, false, false, 64, 2>>(ctx, tmA, tmB, p, 1, st);
    };
    if (const char* force = getenv("A3D_POOL4_FORCE")) return run(atoi(force));
    TuneKey key{};
    const int kv[16] = {5, d->N, d->H, d->W, d->C, d->K, d->R, d->S, d->stride_h, d->stride_w, d->pad_t, d->pad_l,
                        d->P, d->Q, d->ldy + 4096 * d->dil_w + 65536 * d->pix_pitch, pool_idx != nullptr};
    memcpy(key.v, kv, sizeof(kv));
    // candidates 0..3 one-CTA tiles, 6..7 CTA pairs
    int cands[8], nc = 0;
    for (int c = 0; c < 4; ++c) cands[nc++] = c;
    cands[nc++] = 6;
    cands[nc++] = 7;
    const int best = autotune(key, nc, [&](int i) { return run(cands[i]); }, st);
    if (best < 0) return A3D_EINVAL;
    return run(cands[best]);
  }
  if (!a3d_tc_conv_fwd_supported(d)) {
    a3d_set_error("tc conv fwd: unsupported shape (C=%d must be a multiple of 16)", d->C);
    return A3D_ENOTSUP;
  }
  // channels per TMA load: 64/32/16 -> swizzled rows of 128/64/32 B; 8 -> chunked mode (8 loads per stage)
  const int kc = d->C % 64 == 0 ? 64 : d->C % 32 == 0 ? 32 : d->C % 16 == 0 ? 16 : 8;
  const int kcb = kc * 2;
  const int cblocks = d->C / kc;
  const int num_kb = kc == 8 ? ceil_div(d->R * d->S * cblocks, 8) : d->R * d->S * cblocks;
  const long long M = (long long)d->N * d->P * d->Q;
  CUtensorMap tmA;
  int rc = make_tmap_im2col(ctx, &tmA, x, d->N, d->H, d->W, d->C, -d->pad_t, -d->pad_l, d->P, d->Q, d->stride_h,
                            d->stride_w, kc, 128);
  if (rc) return rc;
  tc::Params p{};
  p.M = (int)M; p.N = d->K; p.num_kb = num_kb;
  p.a_mode = tc::A_IM2COL; p.a_k0 = 0;
  p.PQ = d->P * d->Q; p.Q = d->Q; p.sh = d->stride_h; p.sw = d->stride_w; p.lower_h = -d->pad_t; p.lower_w = -d->pad_l;
  p.S = d->S; p.cblocks = cblocks;
  const bool can_split = ws && ws_bytes >= (size_t)M * d->K * sizeof(float);
  // whether an unsplit launch stores y through the TMA epilogue (maybe_tma_out): the CTA-pair kernel has no other one,
  // so its candidates exist only for such outputs, and the tuner key tells the two cases apart
  const bool out_tma = y_dtype == A3D_F32 ? epi_tma_ok(y, d->ldy)
                                          : (reinterpret_cast<uintptr_t>(y) & 15) == 0 && d->ldy % 8 == 0;

  auto launch = [&](int bn, int splits, int variant) -> int {
    CUtensorMap tmB;
    const int box_rows = bn / mcast_cl(variant);              // cluster kernel: every CTA loads a slice of the weight tile
    int r = kc == 8 ? make_tmap_chunked(ctx, &tmB, w, d->K, (uint64_t)d->R * d->S * d->C, bn)
                    : make_tmap_2d(ctx, &tmB, w, d->K, (uint64_t)d->R * d->S * d->C, (uint64_t)d->R * d->S * d->C, kc,
                                   box_rows);
    if (r) return r;
    tc::Params q = p;
    if (!can_split) splits = 1;
    q.kb_per_split = ceil_div(num_kb, splits);
    splits = ceil_div(num_kb, q.kb_per_split);
    if (splits == 1) {
      q.epi = y_dtype == A3D_F32 ? tc::EPI_ROW_F32 : tc::EPI_ROW_BF16;
      q.out = y; q.ldo = d->ldy; q.bias = bias; q.flags = flags; q.atomic = 0;
      return launch_kk(ctx, bn, kcb, tmA, tmB, q, 1, st, variant);
    }
    A3D_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)M * d->K * sizeof(float), st));
    q.epi = tc::EPI_ROW_F32; q.out = ws; q.ldo = d->K; q.bias = nullptr; q.flags = 0; q.atomic = 1;
    r = launch_kk(ctx, bn, kcb, tmA, tmB, q, splits, st, variant);
    if (r) return r;
    return finish(ctx, reinterpret_cast<const float*>(ws), bias, nullptr, 0.f, y, y_dtype == A3D_F32, (size_t)M, d->K,
                  d->ldy, flags, st);
  };
  auto tiles_of = [&](int bn) { return ceil_div(M, 128) * ceil_div(d->K, bn); };
  // candidate 0 = heuristic; then the tile widths that cover K with little padding, each with 1 and ~1-2 waves of split-K
  struct Cand { int bn, splits, variant; };
  Cand cand[64];
  int nc = 0;
  {
    int bn0 = pick_bn(d->K);
    if (kc == 8 && bn0 < 32) bn0 = 32;
    cand[nc++] = {bn0, pick_splits(ctx, tiles_of(bn0), num_kb, 8), V_BASE};
  }
  static const int widths[] = {64, 96, 128, 192, 256};
  for (int i = 0; i < 5; ++i) {
    const int bn = widths[i];
    if (kc == 8 && bn > 128) continue;                        // chunked kernels exist up to BN = 128
    if (kc == 16 && bn == 192) continue;                      // (no <192, 32> instantiation)
    const int padded = ceil_div(d->K, bn) * bn;
    if (padded > d->K + d->K / 3 + 15) continue;              // more than a third of the columns would be padding
    const int tiles = tiles_of(bn);
    const int sopts[3] = {1, ctx->sm_count / tiles, 2 * ctx->sm_count / tiles};
    for (int t = 0; t < 3; ++t) {
      int sp = sopts[t];
      const int max_s = num_kb / 8 > 0 ? num_kb / 8 : 1;
      if (sp > max_s) sp = max_s;
      if (sp < 1 || !can_split) sp = 1;
      for (int variant = 0; variant < V_COUNT; ++variant) {
        if (!variant_exists(bn, kcb, variant)) continue;
        // 256-row tiles only unsplit and when they still give every SM about one CTA
        if ((variant == V_BM256 || variant == V_BM256_DEEP) && (sp != 1 || tiles / 2 < ctx->sm_count * 3 / 4)) continue;
        // pair kernel: unsplit, at least one full pair of M tiles, TMA-stored output
        if ((variant == V_PAIR || variant == V_PAIR_DEEP) && (sp != 1 || ceil_div(M, 128) < 2 || !out_tma)) continue;
        // pair kernel with an f32 output: 32-column slabs, any BN; with a bf16 output BN % 64 (checked at launch)
        if ((variant == V_PAIR || variant == V_PAIR_DEEP) && y_dtype != A3D_F32 && bn % 64) continue;
        bool dup = false;
        for (int k = 0; k < nc; ++k) dup |= (cand[k].bn == bn && cand[k].splits == sp && cand[k].variant == variant);
        if (!dup && nc < 64) cand[nc++] = {bn, sp, variant};
      }
    }
  }
  if (const char* force = getenv("A3D_CONV_FORCE")) {            // "bn,splits,variant": tests and A/B runs
    int fbn = 0, fsp = 1, fv = 0;
    if (sscanf(force, "%d,%d,%d", &fbn, &fsp, &fv) >= 1 && fbn > 0) return launch(fbn, fsp, fv);
  }
  TuneKey key{};
  const int kv[16] = {2, d->N, d->H, d->W, d->C, d->K, d->R, d->S, d->stride_h, d->stride_w, d->pad_t, d->pad_l,
                      d->P, d->Q, d->ldy, y_dtype * 2 + (can_split ? 1 : 0) + (out_tma ? 0 : 4)};
  memcpy(key.v, kv, sizeof(kv));
  const int best = autotune(key, nc, [&](int c) { return launch(cand[c].bn, cand[c].splits, cand[c].variant); }, st);
  if (best < 0) return A3D_EINVAL;
  return launch(cand[best].bn, cand[best].splits, cand[best].variant);
}

// ------------------------------------------------------------------------------------------------
// dense forward: the weight matrix [N_out][K] is the 128-row operand (it is the one that has to be
// streamed from HBM exactly once); the activations [M_batch][K] are the UMMA N operand.
// acc_ws f32 [M_batch][N_out] receives the split-K partial sums; `finish` applies bias/act/dropout.
int a3d_tc_dense_fwd(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* w, const float* bias,
                     const uint8_t* mask, float drop_rate, void* y, int y_dtype, float* acc_ws, int M, int N, int K,
                     unsigned flags, cudaStream_t st) {
  if (K % 64 || ldx % 8 || M > 256 || !acc_ws) {
    a3d_set_error("tc dense fwd: needs K %% 64 == 0, batch <= 256 and an accumulation workspace (K=%d M=%d)", K, M);
    return A3D_ENOTSUP;
  }
  int bn = M <= 32 ? 32 : M <= 64 ? 64 : M <= 128 ? 128 : 256;
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, w, N, K, K, 64, 128);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, x, M, K, ldx, 64, bn);
  if (rc) return rc;
  tc::Params p{};
  p.M = N; p.N = M; p.num_kb = K / 64; p.a_mode = tc::A_TILED; p.a_k0 = 0;
  const int tiles = ceil_div(N, 128);
  int splits0 = pick_splits(ctx, tiles, p.num_kb, 4);
  // weight streaming is HBM-bound: two CTAs' worth of loads in flight per SM helps, so oversubscribe
  if (splits0 * tiles < 2 * ctx->sm_count && p.num_kb / (splits0 * 2) >= 4) splits0 *= 2;
  p.epi = tc::EPI_COL_F32; p.out = acc_ws; p.ldo = N; p.bias = nullptr; p.flags = 0; p.atomic = 1;
  auto launch = [&](int splits) -> int {          // splits >= 1000: interleaved k-blocks (Params::kb_interleave)
    tc::Params q = p;
    q.kb_interleave = splits >= 1000;
    splits %= 1000;
    q.kb_per_split = ceil_div(q.num_kb, splits);
    splits = ceil_div(q.num_kb, q.kb_per_split);
    A3D_CHECK_CUDA(cudaMemsetAsync(acc_ws, 0, (size_t)M * N * sizeof(float), st));
    int r = launch_kk(ctx, bn, 128, tmA, tmB, q, splits, st);
    if (r) return r;
    return finish(ctx, acc_ws, bias, mask, drop_rate, y, y_dtype == A3D_F32, (size_t)M, N, N, flags, st);
  };
  // batch <= 32: the weight-streaming mma.sync kernel (dense_stream.cu) competes with the tcgen05 tiles;
  // candidates >= 100 are stream launches with 1x / 2x / 3x the resident CTA slots
  const bool s_ok = a3d_stream_dense_fwd_ok(M, N, K, ldx);
  auto launch_stream = [&](int ctas) -> int {
    int r = a3d_stream_dense_fwd(ctx, x, ldx, w, acc_ws, M, N, K, ctas, st);
    if (r) return r;
    return finish(ctx, acc_ws, bias, mask, drop_rate, y, y_dtype == A3D_F32, (size_t)M, N, N, flags, st);
  };
  int cand[24];
  int nc = split_candidates(ctx, tiles, p.num_kb, splits0, cand);
  for (int i = 0, n0 = nc; i < n0; ++i)
    if (cand[i] > 1) cand[nc++] = 1000 + cand[i];
  if (s_ok)
    for (int m = 1; m <= 3; ++m) cand[nc++] = 100 + m;
  auto run = [&](int c) -> int {
    return c >= 100 && c < 1000 ? launch_stream((c - 100) * 2 * ctx->sm_count) : launch(c);
  };
  if (const char* force = getenv("A3D_DENSE_FORCE")) return run(atoi(force));   // tests: e.g. 1006 = 6 interleaved splits
  TuneKey key{};
  const int kv[16] = {3, M, N, K, ldx, y_dtype, (int)flags, mask != nullptr, s_ok};
  memcpy(key.v, kv, sizeof(kv));
  const int best = autotune(key, nc, [&](int c) { return run(cand[c]); }, st);
  if (best < 0) return A3D_EINVAL;
  return run(cand[best]);
}

// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// convolution weight gradient:  dW[co][(tap,ci)] = sum_m dY[m][co] * im2col(X)[m][(tap,ci)]
// Both operands are MN-major (the reduction index m = output pixel is the slow one in memory):
//   A = dY  [m][co]   tiled loads of 64 pixels x 64 channels
//   B = X in im2col mode, 64 pixels x BW channels per (tap, channel-block)
// split-K over the pixel range with fp32 atomics into the (zeroed) dW.
namespace {
template <int BW, int NBLK, int BM = 128>
int launch_wgrad(a3d_ctx* ctx, const CUtensorMap& tmA, const CUtensorMap& tmB, const tc::Params& p, int splits,
                 cudaStream_t st) {
  return launch_cfg<tc::Cfg<BW * NBLK, 128, true, true, BW, A3D_MIN_STAGES, false, BM>>(ctx, tmA, tmB, p, splits, st);
}
int pick_nblk(int bw, int total_blocks) {
  static const int c64[] = {4, 3, 2, 1, 0}, c32[] = {6, 5, 4, 3, 0}, c16[] = {16, 11, 8, 0};
  const int* cand = bw == 64 ? c64 : bw == 32 ? c32 : c16;
  int best = cand[0], best_pad = 1 << 30;
  for (int i = 0; cand[i]; ++i) {
    int padded = (total_blocks + cand[i] - 1) / cand[i] * cand[i];
    if (padded < best_pad) { best_pad = padded; best = cand[i]; }
  }
  return best;
}
}  // namespace

int a3d_tc_conv_wgrad_supported(const a3d_conv_desc* d) {
  return d->C % 16 == 0 && d->ldy % 8 == 0 && d->stride_h <= 8 && d->stride_w <= 8 && d->R <= 256 && d->S <= 256;
}

int a3d_tc_conv_wgrad(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* x, const uint16_t* dy, float* dw,
                      cudaStream_t st) {
  if (!a3d_tc_conv_wgrad_supported(d)) {
    a3d_set_error("tc conv wgrad: unsupported shape (C=%d ldy=%d)", d->C, d->ldy);
    return A3D_ENOTSUP;
  }
  const int bw = d->C % 64 == 0 ? 64 : d->C % 32 == 0 ? 32 : 16;
  const int cblocks = d->C / bw;
  const int RS = d->R * d->S;
  const int total_blocks = RS * cblocks;
  const long long Mpix = (long long)d->N * d->P * d->Q;
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, dy, Mpix, d->K, d->ldy, 64, 64);
  if (rc) return rc;
  rc = make_tmap_im2col(ctx, &tmB, x, d->N, d->H, d->W, d->C, -d->pad_t, -d->pad_l, d->P, d->Q, d->stride_h,
                        d->stride_w, bw, 64, 2, false, d->pix_pitch);
  if (rc) return rc;
  tc::Params p{};
  p.M = d->K; p.N = RS * d->C; p.num_kb = ceil_div(Mpix, 64);
  p.a_mode = tc::A_TILED; p.b_im2col = 1; p.RS = RS;
  p.PQ = d->P * d->Q; p.Q = d->Q; p.sh = d->stride_h; p.sw = d->stride_w; p.lower_h = -d->pad_t; p.lower_w = -d->pad_l;
  p.S = d->S; p.cblocks = cblocks; p.dil_w = d->dil_w > 1 ? d->dil_w : 1;
  p.epi = tc::EPI_ROW_F32; p.out = dw; p.ldo = (long long)RS * d->C;

  // bm = 256: 256 filters per CTA, i.e. two accumulators share every im2col stage of X (the expensive operand)
  auto launch = [&](int nblk, int splits, int bm = 128) -> int {
    tc::Params q = p;
    q.kb_per_split = ceil_div(q.num_kb, splits);
    splits = ceil_div(q.num_kb, q.kb_per_split);
    q.atomic = splits > 1;
    if (splits > 1) A3D_CHECK_CUDA(cudaMemsetAsync(dw, 0, (size_t)d->K * RS * d->C * sizeof(float), st));
    if (bm == 256) {
      if (bw == 64 && nblk == 4) return launch_wgrad<64, 4, 256>(ctx, tmA, tmB, q, splits, st);
      if (bw == 64 && nblk == 3) return launch_wgrad<64, 3, 256>(ctx, tmA, tmB, q, splits, st);
      if (bw == 64 && nblk == 2) return launch_wgrad<64, 2, 256>(ctx, tmA, tmB, q, splits, st);
      if (bw == 64 && nblk == 1) return launch_wgrad<64, 1, 256>(ctx, tmA, tmB, q, splits, st);
      a3d_set_error("tc conv wgrad: no 256-row kernel for BW=%d NBLK=%d", bw, nblk);
      return A3D_ENOTSUP;
    }
#define A3D_WG(BW, NB) if (bw == BW && nblk == NB) return launch_wgrad<BW, NB>(ctx, tmA, tmB, q, splits, st);
    A3D_WG(64, 4) A3D_WG(64, 3) A3D_WG(64, 2) A3D_WG(64, 1)
    A3D_WG(32, 6) A3D_WG(32, 5) A3D_WG(32, 4) A3D_WG(32, 3)
    A3D_WG(16, 16) A3D_WG(16, 11) A3D_WG(16, 8)
#undef A3D_WG
    a3d_set_error("tc conv wgrad: no kernel for BW=%d NBLK=%d", bw, nblk);
    return A3D_ENOTSUP;
  };
  auto tiles_of = [&](int nblk, int bm = 128) { return ceil_div(d->K, bm) * ceil_div(total_blocks, nblk); };
  if (const char* force = getenv("A3D_WGRAD_FORCE")) {           // "nblk,splits,bm": tests and A/B runs
    int fn = 0, fs = 1, fb = 128;
    if (sscanf(force, "%d,%d,%d", &fn, &fs, &fb) >= 1 && fn > 0) return launch(fn, fs, fb);
  }
  // candidates: candidate 0 is the heuristic; then every tile width x {1, 1.5, 2, 3} waves' worth of CTAs,
  // with 128 and (layers with > 128 filters, 64-channel blocks) 256 filters per CTA
  struct Cand { int nblk, splits, bm; };
  Cand cand[80];
  int nc = 0;
  {
    const int nb0 = pick_nblk(bw, total_blocks);
    cand[nc++] = {nb0, pick_splits(ctx, tiles_of(nb0), p.num_kb, 4), 128};
  }
  static const int w64[] = {1, 2, 3, 4, 0}, w32[] = {3, 4, 5, 6, 0}, w16[] = {8, 11, 16, 0};
  const int* widths = bw == 64 ? w64 : bw == 32 ? w32 : w16;
  for (int bm = 128; bm <= 256; bm += 128) {
    if (bm == 256 && (bw != 64 || d->K <= 128)) continue;
    for (int i = 0; widths[i]; ++i) {
      const int tiles = tiles_of(widths[i], bm);
      static const int target_x2[] = {2, 3, 4, 6};      // CTAs ~ target/2 x SM count
      for (int t = 0; t < 4; ++t) {
        int s = (ctx->sm_count * target_x2[t] / 2) / tiles;
        const int max_s = p.num_kb / 4 > 0 ? p.num_kb / 4 : 1;
        if (s > max_s) s = max_s;
        if (s < 1) s = 1;
        bool dup = false;
        for (int k = 0; k < nc; ++k) dup |= (cand[k].nblk == widths[i] && cand[k].splits == s && cand[k].bm == bm);
        if (!dup && nc < 80) cand[nc++] = {widths[i], s, bm};
      }
    }
  }
  TuneKey key{};
  const int kv[16] = {1, d->N, d->H, d->W, d->C, d->K, d->R, d->S, d->stride_h, d->stride_w, d->pad_t, d->pad_l,
                      d->P, d->Q, d->ldy, d->dil_w * 4096 + d->pix_pitch};
  memcpy(key.v, kv, sizeof(kv));
  const int best = autotune(key, nc, [&](int c) { return launch(cand[c].nblk, cand[c].splits, cand[c].bm); }, st);
  if (best < 0) return A3D_EINVAL;
  return launch(cand[best].nblk, cand[best].splits, cand[best].bm);
}

// ------------------------------------------------------------------------------------------------
// strided dgrad, GEMM half:  col[m][(tap,ci)] = sum_co dY[m][co] * W[co][(tap,ci)]   (f32, then col2im)
int a3d_tc_dgrad_cols(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* dy, const uint16_t* w, float* col,
                      cudaStream_t st) {
  const long long Mpix = (long long)d->N * d->P * d->Q;
  const int J = d->R * d->S * d->C;
  if (d->K % 64 || J % 64 || d->ldy % 8) {
    a3d_set_error("tc dgrad cols: needs K %% 64 == 0 and R*S*C %% 64 == 0");
    return A3D_ENOTSUP;
  }
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, dy, Mpix, d->K, d->ldy, 64, 128);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, w, d->K, J, J, 64, 64);
  if (rc) return rc;
  tc::Params p{};
  p.M = (int)Mpix; p.N = J; p.num_kb = d->K / 64; p.kb_per_split = p.num_kb; p.a_mode = tc::A_TILED;
  p.epi = tc::EPI_ROW_F32; p.out = col; p.ldo = J; p.atomic = 0;
  const int bn = J % 256 == 0 ? 256 : J % 192 == 0 ? 192 : J % 128 == 0 ? 128 : 64;
  if (bn == 256) return launch_cfg<tc::Cfg<256, 128, false, true, 64>>(ctx, tmA, tmB, p, 1, st);
  if (bn == 192) return launch_cfg<tc::Cfg<192, 128, false, true, 64>>(ctx, tmA, tmB, p, 1, st);
  if (bn == 128) return launch_cfg<tc::Cfg<128, 128, false, true, 64>>(ctx, tmA, tmB, p, 1, st);
  return launch_cfg<tc::Cfg<64, 128, false, true, 64>>(ctx, tmA, tmB, p, 1, st);
}

// dense dgrad of a LONG batch (DCNF: 768 patches x 128 -> 12544): the batch is the GEMM M dimension, A = dy K-major,
// B = w MN-major (as in a3d_tc_dgrad_cols), bf16 rows written straight from the epilogue -- one launch, no accumulation
// buffer.  The weight-streaming form below (batch <= 128 as the UMMA N dimension) is for the batch-32 MSDN layers.
int a3d_tc_dense_dgrad_rows(a3d_ctx* ctx, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx, int M, int N, int K,
                            cudaStream_t st) {
  if (N % 64 || K % 64 || lddy % 8) {
    a3d_set_error("tc dense dgrad (rows): needs N %% 64 == 0, K %% 64 == 0, lddy %% 8 == 0 (N=%d K=%d)", N, K);
    return A3D_ENOTSUP;
  }
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, dy, M, N, lddy, 64, 128);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, w, N, K, K, 64, 64);
  if (rc) return rc;
  tc::Params p{};
  p.M = M; p.N = K; p.num_kb = N / 64; p.kb_per_split = p.num_kb; p.a_mode = tc::A_TILED;
  p.epi = tc::EPI_ROW_BF16; p.out = dx; p.ldo = K; p.atomic = 0;
  const int bn = K % 256 == 0 ? 256 : K % 128 == 0 ? 128 : 64;
  if (bn == 256) return launch_cfg<tc::Cfg<256, 128, false, true, 64>>(ctx, tmA, tmB, p, 1, st);
  if (bn == 128) return launch_cfg<tc::Cfg<128, 128, false, true, 64>>(ctx, tmA, tmB, p, 1, st);
  return launch_cfg<tc::Cfg<64, 128, false, true, 64>>(ctx, tmA, tmB, p, 1, st);
}

// ------------------------------------------------------------------------------------------------
// dense backward.  dgrad: dx[b][k] = sum_n dy[b][n] w[n][k]  -> D^T[k][b], A = w MN-major, B = dy K-major.
struct a3d_actbwd_args { const uint16_t* y; const uint8_t* keep_mask; float drop_rate; unsigned flags; };
int a3d_tc_dense_dgrad(a3d_ctx* ctx, const uint16_t* dy, int lddy, const uint16_t* w, uint16_t* dx, float* acc_ws,
                       int M, int N, int K, cudaStream_t st, const a3d_actbwd_args* ab = nullptr) {
  if (K % 8 || lddy % 8 || M > 128 || !acc_ws) {
    a3d_set_error("tc dense dgrad: needs K %% 8 == 0, lddy %% 8 == 0, batch <= 128, workspace");
    return A3D_ENOTSUP;
  }
  const int bn = M <= 32 ? 32 : M <= 64 ? 64 : 128;
  auto finish_dx = [&]() -> int {
    if (!ab) return finish(ctx, acc_ws, nullptr, nullptr, 0.f, dx, 0, (size_t)M, K, K, 0, st);
    const size_t total = (size_t)M * K;
    size_t blocks = (total + 255) / 256;
    if (blocks > (size_t)ctx->sm_count * 16) blocks = (size_t)ctx->sm_count * 16;
    act_bwd_cast_kernel<<<(int)blocks, 256, 0, st>>>(acc_ws, ab->y, ab->keep_mask, 1.f / (1.f - ab->drop_rate), dx, total,
                                                    ab->flags);
    A3D_LAUNCH_OK(ctx);
    return 0;
  };
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, w, N, K, K, 64, 64);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, dy, M, N, lddy, 64, bn);
  if (rc) return rc;
  tc::Params p{};
  p.M = K; p.N = M; p.num_kb = ceil_div(N, 64); p.a_mode = tc::A_TILED;
  const int tiles = ceil_div(K, 128);
  int splits0 = pick_splits(ctx, tiles, p.num_kb, 4);
  if (splits0 * tiles < 2 * ctx->sm_count && p.num_kb / (splits0 * 2) >= 4) splits0 *= 2;
  p.epi = tc::EPI_COL_F32; p.out = acc_ws; p.ldo = K; p.atomic = 1;
  auto launch = [&](int splits) -> int {          // splits >= 1000: interleaved k-blocks
    tc::Params q = p;
    q.kb_interleave = splits >= 1000;
    splits %= 1000;
    q.kb_per_split = ceil_div(q.num_kb, splits);
    splits = ceil_div(q.num_kb, q.kb_per_split);
    A3D_CHECK_CUDA(cudaMemsetAsync(acc_ws, 0, (size_t)M * K * sizeof(float), st));
    int r;
    if (bn == 32) r = launch_cfg<tc::Cfg<32, 128, true, false>>(ctx, tmA, tmB, q, splits, st);
    else if (bn == 64) r = launch_cfg<tc::Cfg<64, 128, true, false>>(ctx, tmA, tmB, q, splits, st);
    else r = launch_cfg<tc::Cfg<128, 128, true, false>>(ctx, tmA, tmB, q, splits, st);
    if (r) return r;
    return finish_dx();
  };
  const bool s_ok = a3d_stream_dense_dgrad_ok(M, N, K, lddy);
  auto launch_stream = [&](int ctas) -> int {
    int r = a3d_stream_dense_dgrad(ctx, dy, lddy, w, acc_ws, M, N, K, ctas, st);
    if (r) return r;
    return finish_dx();
  };
  int cand[24];
  int nc = split_candidates(ctx, tiles, p.num_kb, splits0, cand);
  for (int i = 0, n0 = nc; i < n0; ++i)
    if (cand[i] > 1) cand[nc++] = 1000 + cand[i];
  if (s_ok)
    for (int m = 1; m <= 3; ++m) cand[nc++] = 100 + m;
  auto run = [&](int c) -> int {
    return c >= 100 && c < 1000 ? launch_stream((c - 100) * 2 * ctx->sm_count) : launch(c);
  };
  if (const char* force = getenv("A3D_DENSE_FORCE")) return run(atoi(force));
  TuneKey key{};
  const int kv[16] = {4, M, N, K, lddy, s_ok};
  memcpy(key.v, kv, sizeof(kv));
  const int best = autotune(key, nc, [&](int c) { return run(cand[c]); }, st);
  if (best < 0) return A3D_EINVAL;
  return run(cand[best]);
}

// wgrad: dw[n][k] = sum_b dy[b][n] x[b][k]; both operands MN-major with the batch as the reduction index.
int a3d_tc_dense_wgrad(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* dy, int lddy, float* dw, int M, int N,
                       int K, cudaStream_t st) {
  if (K % 64 || ldx % 8 || lddy % 8) {
    a3d_set_error("tc dense wgrad: needs K %% 64 == 0 and 16-byte aligned row pitches");
    return A3D_ENOTSUP;
  }
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, dy, M, N, lddy, 64, 64);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, x, M, K, ldx, 64, 64);
  if (rc) return rc;
  tc::Params p{};
  p.M = N; p.N = K; p.num_kb = ceil_div(M, 64); p.kb_per_split = p.num_kb; p.a_mode = tc::A_TILED;
  p.epi = tc::EPI_ROW_F32; p.out = dw; p.ldo = K; p.atomic = 0;
  // One k-block per CTA: the kernel is all prologue + epilogue.  N tiles of 128 keep the stage ring under
  // 104 KB so that two CTAs share an SM and one's epilogue hides the other's prologue.
  if (K % 128 == 0) return launch_cfg<tc::Cfg<128, 128, true, true, 64>>(ctx, tmA, tmB, p, 1, st);
  return launch_cfg<tc::Cfg<64, 128, true, true, 64>>(ctx, tmA, tmB, p, 1, st);
}

// Raw GEMM for unit tests of the engine: D[M][N] (f32, row-major) = A * B^T with every combination
// of operand majors.  K-major operand: [rows][K]; MN-major operand: [K][rows].
extern "C" int a3d_debug_tc_gemm_v(a3d_ctx* ctx, const uint16_t* A, const uint16_t* B, float* D, int M, int N, int K,
                                   int bn, int kcb, int a_mn, int b_mn, int splits, int variant, void* stream);
extern "C" int a3d_debug_tc_gemm(a3d_ctx* ctx, const uint16_t* A, const uint16_t* B, float* D, int M, int N, int K,
                                 int bn, int kcb, int a_mn, int b_mn, int splits, void* stream) {
  return a3d_debug_tc_gemm_v(ctx, A, B, D, M, N, K, bn, kcb, a_mn, b_mn, splits, 0, stream);
}
// variant: tile variant of launch_kk (K-major x K-major only): 1 deeper ring, 2 256-row tile, 3 both
extern "C" int a3d_debug_tc_gemm_v(a3d_ctx* ctx, const uint16_t* A, const uint16_t* B, float* D, int M, int N, int K,
                                   int bn, int kcb, int a_mn, int b_mn, int splits, int variant, void* stream) {
  A3D_REQUIRE(ctx && A && B && D, "debug gemm: null argument");
  cudaStream_t st = as_stream(stream);
  CUtensorMap tmA, tmB;
  int rc;
  const int kelems = (a_mn || b_mn) ? 64 : kcb / 2;
  A3D_REQUIRE(K % kelems == 0, "debug gemm: K must be a multiple of %d", kelems);
  if (a_mn) rc = make_tmap_2d(ctx, &tmA, A, K, M, M, 64, 64);
  else rc = make_tmap_2d(ctx, &tmA, A, M, K, K, kelems, 128);
  if (rc) return rc;
  if (b_mn) rc = make_tmap_2d(ctx, &tmB, B, K, N, N, 64, 64);
  else rc = make_tmap_2d(ctx, &tmB, B, N, K, K, kelems, bn / mcast_cl(variant));
  if (rc) return rc;
  tc::Params p{};
  p.M = M; p.N = N; p.num_kb = K / kelems; p.a_mode = tc::A_TILED;
  if (splits < 1) splits = 1;
  p.kb_per_split = ceil_div(p.num_kb, splits);
  splits = ceil_div(p.num_kb, p.kb_per_split);
  p.epi = tc::EPI_ROW_F32; p.out = D; p.ldo = N; p.atomic = splits > 1;
  if (splits > 1) A3D_CHECK_CUDA(cudaMemsetAsync(D, 0, (size_t)M * N * sizeof(float), st));
  if (!a_mn && !b_mn) return launch_kk(ctx, bn, kcb, tmA, tmB, p, splits, st, variant);
#define A3D_MN_CASE(BN, AM, BM_) \
  if (bn == BN && (bool)a_mn == AM && (bool)b_mn == BM_) \
    return launch_cfg<tc::Cfg<BN, 128, AM, BM_>>(ctx, tmA, tmB, p, splits, st);
  A3D_MN_CASE(64, true, true) A3D_MN_CASE(128, true, true) A3D_MN_CASE(256, true, true)
  A3D_MN_CASE(32, true, false) A3D_MN_CASE(64, true, false) A3D_MN_CASE(128, true, false)
  A3D_MN_CASE(64, false, true) A3D_MN_CASE(128, false, true) A3D_MN_CASE(256, false, true)
#undef A3D_MN_CASE
  a3d_set_error("debug gemm: no kernel for BN=%d a_mn=%d b_mn=%d", bn, a_mn, b_mn);
  return A3D_ENOTSUP;
}

// =====================================================================================================================
// TF32 precision mode: the same implicit-GEMM formulations with float32 tensors in HBM / shared memory and
// tcgen05.mma kind::tf32 (10-bit mantissa inputs, f32 accumulation) -- the reference's arithmetic is float32
// (src/models.py:211-251); BASELINE.json's north star asks for 1e-4 agreement in this mode.  One tile configuration per
// shape class and closed-form split-K (no autotuning: the mode is about precision; its step time is reported, not tuned).
// =====================================================================================================================
namespace {
template <int BN, bool AM, bool BM_, int MS = A3D_MIN_STAGES>
using CfgT = tc::Cfg<BN, 128, AM, BM_, 32, MS, false, 128, 4>;

__global__ void act_bwd_cast_f32_kernel(const float* __restrict__ acc, const float* __restrict__ y,
                                        const uint8_t* __restrict__ mask, float scale, float* __restrict__ dx, size_t n,
                                        unsigned flags) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    float g = acc[i];
    if (mask) g = mask[i] ? g * scale : 0.f;
    if (y) {
      const float yv = y[i];
      if (flags & A3D_EPI_RELU) g = yv > 0.f ? g : 0.f;
      if (flags & A3D_EPI_SIGMOID) g = g * yv * (1.f - yv);
    }
    dx[i] = g;
  }
}
}  // namespace

// acc_only: add the raw products into ws ([N*P*Q][K] f32, zeroed by the caller) and stop -- one term of a 3xTF32 sum
int a3d_tc_conv_fwd_tf32(a3d_ctx* ctx, const a3d_conv_desc* d, const float* x, const float* w, const float* bias, float* y,
                         unsigned flags, void* ws, size_t ws_bytes, cudaStream_t st, int acc_only) {
  if (d->C % 32 || d->stride_h > 8 || d->stride_w > 8 || d->R > 256 || d->S > 256) {
    a3d_set_error("tf32 conv fwd: needs C %% 32 == 0 (C=%d)", d->C);
    return A3D_ENOTSUP;
  }
  const int cblocks = d->C / 32;
  const int num_kb = d->R * d->S * cblocks;
  const long long M = (long long)d->N * d->P * d->Q;
  const long long J = (long long)d->R * d->S * d->C;
  const int bn = d->K <= 16 ? 16 : d->K <= 64 ? 64 : d->K <= 128 ? 128 : (d->K % 256 == 0 ? 256 : 128);
  CUtensorMap tmA, tmB;
  int rc = make_tmap_im2col(ctx, &tmA, x, d->N, d->H, d->W, d->C, -d->pad_t, -d->pad_l, d->P, d->Q, d->stride_h, d->stride_w,
                            32, 128, 4);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, w, d->K, J, J, 32, bn, 4);
  if (rc) return rc;
  tc::Params p{};
  p.M = (int)M; p.N = d->K; p.num_kb = num_kb; p.a_mode = tc::A_IM2COL;
  p.PQ = d->P * d->Q; p.Q = d->Q; p.sh = d->stride_h; p.sw = d->stride_w; p.lower_h = -d->pad_t; p.lower_w = -d->pad_l;
  p.S = d->S; p.cblocks = cblocks;
  const bool can_split = ws && ws_bytes >= (size_t)M * d->K * sizeof(float);
  int splits = can_split ? pick_splits(ctx, ceil_div(M, 128) * ceil_div(d->K, bn), num_kb, 8) : 1;
  p.kb_per_split = ceil_div(num_kb, splits);
  splits = ceil_div(num_kb, p.kb_per_split);
  if (acc_only && !can_split) {
    a3d_set_error("tf32 conv fwd: the accumulate-only form needs the [N*P*Q][K] f32 workspace");
    return A3D_EINVAL;
  }
  if (splits == 1 && !acc_only) {
    p.epi = tc::EPI_ROW_F32; p.out = y; p.ldo = d->ldy; p.bias = bias; p.flags = flags; p.atomic = 0;
  } else {
    if (!acc_only) A3D_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)M * d->K * sizeof(float), st));
    p.epi = tc::EPI_ROW_F32; p.out = ws; p.ldo = d->K; p.bias = nullptr; p.flags = 0; p.atomic = 1;
  }
  rc = bn == 16 ? launch_cfg<CfgT<16, false, false>>(ctx, tmA, tmB, p, splits, st)
       : bn == 64 ? launch_cfg<CfgT<64, false, false>>(ctx, tmA, tmB, p, splits, st)
       : bn == 128 ? launch_cfg<CfgT<128, false, false>>(ctx, tmA, tmB, p, splits, st)
                   : launch_cfg<CfgT<256, false, false>>(ctx, tmA, tmB, p, splits, st);
  if (rc || acc_only || splits == 1) return rc;
  return finish(ctx, reinterpret_cast<const float*>(ws), bias, nullptr, 0.f, y, 1, (size_t)M, d->K, d->ldy, flags, st);
}

int a3d_tc_conv_wgrad_tf32(a3d_ctx* ctx, const a3d_conv_desc* d, const float* x, const float* dy, float* dw,
                           cudaStream_t st) {
  if (d->C % 32 || d->ldy % 4 || d->stride_h > 8 || d->stride_w > 8) {
    a3d_set_error("tf32 conv wgrad: needs C %% 32 == 0 and a 16-byte aligned dY pitch (C=%d ldy=%d)", d->C, d->ldy);
    return A3D_ENOTSUP;
  }
  const int cblocks = d->C / 32, RS = d->R * d->S, total_blocks = RS * cblocks;
  const long long Mpix = (long long)d->N * d->P * d->Q;
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, dy, Mpix, d->K, d->ldy, 32, 32, 4, true);
  if (rc) return rc;
  rc = make_tmap_im2col(ctx, &tmB, x, d->N, d->H, d->W, d->C, -d->pad_t, -d->pad_l, d->P, d->Q, d->stride_h, d->stride_w,
                        32, 32, 4, true);
  if (rc) return rc;
  tc::Params p{};
  p.M = d->K; p.N = RS * d->C; p.num_kb = ceil_div(Mpix, 32);
  p.a_mode = tc::A_TILED; p.b_im2col = 1; p.RS = RS;
  p.PQ = d->P * d->Q; p.Q = d->Q; p.sh = d->stride_h; p.sw = d->stride_w; p.lower_h = -d->pad_t; p.lower_w = -d->pad_l;
  p.S = d->S; p.cblocks = cblocks;
  p.epi = tc::EPI_ROW_F32; p.out = dw; p.ldo = (long long)RS * d->C;
  int nblk = 8, best_pad = 1 << 30;
  for (int nb = 8; nb >= 1; nb /= 2) {                      // widest tile with the least padding
    const int padded = ceil_div(total_blocks, nb) * nb;
    if (padded < best_pad) { best_pad = padded; nblk = nb; }
  }
  const int tiles = ceil_div(d->K, 128) * ceil_div(total_blocks, nblk);
  int splits = pick_splits(ctx, tiles, p.num_kb, 8);
  p.kb_per_split = ceil_div(p.num_kb, splits);
  splits = ceil_div(p.num_kb, p.kb_per_split);
  p.atomic = splits > 1;
  if (splits > 1) A3D_CHECK_CUDA(cudaMemsetAsync(dw, 0, (size_t)d->K * RS * d->C * sizeof(float), st));
  if (nblk == 8) return launch_cfg<CfgT<256, true, true>>(ctx, tmA, tmB, p, splits, st);
  if (nblk == 4) return launch_cfg<CfgT<128, true, true>>(ctx, tmA, tmB, p, splits, st);
  if (nblk == 2) return launch_cfg<CfgT<64, true, true>>(ctx, tmA, tmB, p, splits, st);
  return launch_cfg<CfgT<32, true, true>>(ctx, tmA, tmB, p, splits, st);
}

// strided dgrad, GEMM half: col[m][(tap,ci)] = sum_co dY[m][co] * W[co][(tap,ci)]
int a3d_tc_dgrad_cols_tf32(a3d_ctx* ctx, const a3d_conv_desc* d, const float* dy, const float* w, float* col, cudaStream_t st) {
  const long long Mpix = (long long)d->N * d->P * d->Q;
  const int J = d->R * d->S * d->C;
  if (d->K % 32 || J % 64 || d->ldy % 4) {
    a3d_set_error("tf32 dgrad cols: needs K %% 32 == 0 and R*S*C %% 64 == 0");
    return A3D_ENOTSUP;
  }
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, dy, Mpix, d->K, d->ldy, 32, 128, 4);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, w, d->K, J, J, 32, 32, 4, true);
  if (rc) return rc;
  tc::Params p{};
  p.M = (int)Mpix; p.N = J; p.num_kb = d->K / 32; p.kb_per_split = p.num_kb; p.a_mode = tc::A_TILED;
  p.epi = tc::EPI_ROW_F32; p.out = col; p.ldo = J; p.atomic = 0;
  if (J % 256 == 0) return launch_cfg<CfgT<256, false, true>>(ctx, tmA, tmB, p, 1, st);
  if (J % 128 == 0) return launch_cfg<CfgT<128, false, true>>(ctx, tmA, tmB, p, 1, st);
  return launch_cfg<CfgT<64, false, true>>(ctx, tmA, tmB, p, 1, st);
}

// dense layers.  acc_ws f32 [M][N] (fwd) / [M][K] (dgrad) receives the split-K partial sums.
int a3d_tc_dense_fwd_tf32(a3d_ctx* ctx, const float* x, int ldx, const float* w, const float* bias, const uint8_t* mask,
                          float drop_rate, float* y, float* acc_ws, int M, int N, int K, unsigned flags, cudaStream_t st,
                          int acc_only) {
  if (K % 32 || ldx % 4 || M > 256 || !acc_ws) {
    a3d_set_error("tf32 dense fwd: needs K %% 32 == 0, batch <= 256 and an accumulation workspace (K=%d M=%d)", K, M);
    return A3D_ENOTSUP;
  }
  const int bn = M <= 32 ? 32 : M <= 64 ? 64 : M <= 128 ? 128 : 256;
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, w, N, K, K, 32, 128, 4);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, x, M, K, ldx, 32, bn, 4);
  if (rc) return rc;
  tc::Params p{};
  p.M = N; p.N = M; p.num_kb = K / 32; p.a_mode = tc::A_TILED;
  const int tiles = ceil_div(N, 128);
  int splits = pick_splits(ctx, tiles, p.num_kb, 8);
  if (splits * tiles < 2 * ctx->sm_count && p.num_kb / (splits * 2) >= 8) splits *= 2;
  p.kb_per_split = ceil_div(p.num_kb, splits);
  splits = ceil_div(p.num_kb, p.kb_per_split);
  p.epi = tc::EPI_COL_F32; p.out = acc_ws; p.ldo = N; p.atomic = 1;
  if (!acc_only) A3D_CHECK_CUDA(cudaMemsetAsync(acc_ws, 0, (size_t)M * N * sizeof(float), st));
  rc = bn == 32 ? launch_cfg<CfgT<32, false, false>>(ctx, tmA, tmB, p, splits, st)
       : bn == 64 ? launch_cfg<CfgT<64, false, false>>(ctx, tmA, tmB, p, splits, st)
       : bn == 128 ? launch_cfg<CfgT<128, false, false>>(ctx, tmA, tmB, p, splits, st)
                   : launch_cfg<CfgT<256, false, false>>(ctx, tmA, tmB, p, splits, st);
  if (rc || acc_only) return rc;
  return finish(ctx, acc_ws, bias, mask, drop_rate, y, 1, (size_t)M, N, N, flags, st);
}

// dx[b][k] = act'(y_act) * mask/(1-rate) * sum_n dy[b][n] w[n][k]   (y_act / keep_mask nullable)
int a3d_tc_dense_dgrad_tf32(a3d_ctx* ctx, const float* dy, int lddy, const float* w, float* dx, float* acc_ws, int M, int N,
                            int K, const float* y_act, const uint8_t* keep_mask, float drop_rate, unsigned flags,
                            cudaStream_t st) {
  if (K % 4 || lddy % 4 || M > 128 || !acc_ws) {
    a3d_set_error("tf32 dense dgrad: needs K %% 4 == 0, lddy %% 4 == 0, batch <= 128, workspace");
    return A3D_ENOTSUP;
  }
  const int bn = M <= 32 ? 32 : M <= 64 ? 64 : 128;
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, w, N, K, K, 32, 32, 4, true);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, dy, M, N, lddy, 32, bn, 4);
  if (rc) return rc;
  tc::Params p{};
  p.M = K; p.N = M; p.num_kb = ceil_div(N, 32); p.a_mode = tc::A_TILED;
  const int tiles = ceil_div(K, 128);
  int splits = pick_splits(ctx, tiles, p.num_kb, 8);
  if (splits * tiles < 2 * ctx->sm_count && p.num_kb / (splits * 2) >= 8) splits *= 2;
  p.kb_per_split = ceil_div(p.num_kb, splits);
  splits = ceil_div(p.num_kb, p.kb_per_split);
  p.epi = tc::EPI_COL_F32; p.out = acc_ws; p.ldo = K; p.atomic = 1;
  A3D_CHECK_CUDA(cudaMemsetAsync(acc_ws, 0, (size_t)M * K * sizeof(float), st));
  rc = bn == 32 ? launch_cfg<CfgT<32, true, false>>(ctx, tmA, tmB, p, splits, st)
       : bn == 64 ? launch_cfg<CfgT<64, true, false>>(ctx, tmA, tmB, p, splits, st)
                  : launch_cfg<CfgT<128, true, false>>(ctx, tmA, tmB, p, splits, st);
  if (rc) return rc;
  const size_t total = (size_t)M * K;
  size_t blocks = (total + 255) / 256;
  if (blocks > (size_t)ctx->sm_count * 16) blocks = (size_t)ctx->sm_count * 16;
  act_bwd_cast_f32_kernel<<<(int)blocks, 256, 0, st>>>(acc_ws, y_act, keep_mask, 1.f / (1.f - drop_rate), dx, total, flags);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

// dw[n][k] = sum_b dy[b][n] x[b][k]; both operands MN-major with the batch as the reduction index
int a3d_tc_dense_wgrad_tf32(a3d_ctx* ctx, const float* x, int ldx, const float* dy, int lddy, float* dw, int M, int N, int K,
                            cudaStream_t st) {
  if (K % 32 || ldx % 4 || lddy % 4) {
    a3d_set_error("tf32 dense wgrad: needs K %% 32 == 0 and 16-byte aligned row pitches");
    return A3D_ENOTSUP;
  }
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, dy, M, N, lddy, 32, 32, 4, true);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, x, M, K, ldx, 32, 32, 4, true);
  if (rc) return rc;
  tc::Params p{};
  p.M = N; p.N = K; p.num_kb = ceil_div(M, 32); p.kb_per_split = p.num_kb; p.a_mode = tc::A_TILED;
  p.epi = tc::EPI_ROW_F32; p.out = dw; p.ldo = K; p.atomic = 0;
  if (K % 128 == 0) return launch_cfg<CfgT<128, true, true>>(ctx, tmA, tmB, p, 1, st);
  return launch_cfg<CfgT<32, true, true>>(ctx, tmA, tmB, p, 1, st);
}

// ---- TF32 (kind::tf32) engine test hook: D[M][N] (f32) = A * B^T with f32 operands read as TF32, every combination of
// operand majors.  K-major operand: [rows][K]; MN-major operand: [K][rows].  kcb: bytes of K per row and stage (K-major).
extern "C" int a3d_debug_tc_gemm_tf32(a3d_ctx* ctx, const float* A, const float* B, float* D, int M, int N, int K, int bn,
                                      int kcb, int a_mn, int b_mn, int splits, void* stream) {
  A3D_REQUIRE(ctx && A && B && D, "debug gemm tf32: null argument");
  cudaStream_t st = as_stream(stream);
  CUtensorMap tmA, tmB;
  int rc;
  const int kelems = (a_mn || b_mn) ? 32 : kcb / 4;
  A3D_REQUIRE(K % kelems == 0, "debug gemm tf32: K must be a multiple of %d", kelems);
  if (a_mn) rc = make_tmap_2d(ctx, &tmA, A, K, M, M, 32, 32, 4, true);
  else rc = make_tmap_2d(ctx, &tmA, A, M, K, K, kelems, 128, 4);
  if (rc) return rc;
  if (b_mn) rc = make_tmap_2d(ctx, &tmB, B, K, N, N, 32, 32, 4, true);
  else rc = make_tmap_2d(ctx, &tmB, B, N, K, K, kelems, bn, 4);
  if (rc) return rc;
  tc::Params p{};
  p.M = M; p.N = N; p.num_kb = K / kelems; p.a_mode = tc::A_TILED;
  if (splits < 1) splits = 1;
  p.kb_per_split = ceil_div(p.num_kb, splits);
  splits = ceil_div(p.num_kb, p.kb_per_split);
  p.epi = tc::EPI_ROW_F32; p.out = D; p.ldo = N; p.atomic = splits > 1;
  if (splits > 1) A3D_CHECK_CUDA(cudaMemsetAsync(D, 0, (size_t)M * N * sizeof(float), st));
#define A3D_T32(BN, KCB, AM, BM_) \
  if (bn == BN && kcb == KCB && (bool)a_mn == AM && (bool)b_mn == BM_) \
    return launch_cfg<tc::Cfg<BN, KCB, AM, BM_, 32, A3D_MIN_STAGES, false, 128, 4>>(ctx, tmA, tmB, p, splits, st);
  A3D_T32(32, 128, false, false) A3D_T32(64, 128, false, false) A3D_T32(128, 128, false, false) A3D_T32(256, 128, false, false)
  A3D_T32(64, 64, false, false) A3D_T32(128, 64, false, false) A3D_T32(64, 32, false, false) A3D_T32(16, 128, false, false)
  A3D_T32(64, 128, true, true) A3D_T32(128, 128, true, true) A3D_T32(256, 128, true, true)
  A3D_T32(32, 128, true, false) A3D_T32(64, 128, true, false) A3D_T32(128, 128, true, false)
  A3D_T32(64, 128, false, true) A3D_T32(128, 128, false, true) A3D_T32(256, 128, false, true)
#undef A3D_T32
  a3d_set_error("debug gemm tf32: no kernel for BN=%d KCB=%d a_mn=%d b_mn=%d", bn, kcb, a_mn, b_mn);
  return A3D_ENOTSUP;
}

// =====================================================================================================================
// FP8 inference mode (fp8.cu): E4M3 operands, tcgen05.mma kind::f8f6f4, f32 accumulation.  Every operand is K-major with
// 128- or 64-byte rows per stage (SWIZZLE_128B / 64B); the epilogue multiplies each accumulator by its row and column
// scales (tc::Params::rs / cs) before bias and activation.  Split-K partial sums are scaled before they are added, which
// is the same linear map.  Own tuner kinds (6 conv, 7 pool-fused conv, 8 dense), so no bf16 choice is ever reused.
// =====================================================================================================================
namespace {
template <int BN, int KCB, int MS = A3D_MIN_STAGES>
using CfgF8 = tc::Cfg<BN, KCB, false, false, 64, MS, false, 128, 1>;

int launch_f8(a3d_ctx* ctx, int bn, int kcb, int deep, const CUtensorMap& tmA, const CUtensorMap& tmB, const tc::Params& p,
              int splits, cudaStream_t st) {
#define A3D_F8(BN, KCB) \
  if (bn == BN && kcb == KCB && !deep) return launch_cfg<CfgF8<BN, KCB>>(ctx, tmA, tmB, p, splits, st);
  A3D_F8(32, 128) A3D_F8(64, 128) A3D_F8(96, 128) A3D_F8(128, 128) A3D_F8(192, 128) A3D_F8(256, 128)
  A3D_F8(32, 64) A3D_F8(64, 64) A3D_F8(96, 64) A3D_F8(128, 64) A3D_F8(192, 64) A3D_F8(256, 64)
#undef A3D_F8
#define A3D_F8D(BN) \
  if (bn == BN && kcb == 128 && deep) return launch_cfg<CfgF8<BN, 128, 3>>(ctx, tmA, tmB, p, splits, st);
  A3D_F8D(64) A3D_F8D(96) A3D_F8D(128) A3D_F8D(192) A3D_F8D(256)
#undef A3D_F8D
  a3d_set_error("fp8 gemm: no kernel for BN=%d KCB=%d deep=%d", bn, kcb, deep);
  return A3D_ENOTSUP;
}
}  // namespace

// y = act(conv(x, w) * x_scale[image] * w_scale[filter] + bias); pool4: the fused 2x2 max-pool of a3d_tc_conv_fwd (K = 256
// = 4 window positions x 64 filters), the column scales applied before the max.  ws: [N*P*Q][K] f32 split-K accumulator.
int a3d_tc_conv_fwd_fp8(a3d_ctx* ctx, const a3d_conv_desc* d, const uint8_t* x, const float* x_scale, const uint8_t* w,
                        const float* w_scale, const float* bias, void* y, int y_dtype, unsigned flags, void* ws,
                        size_t ws_bytes, cudaStream_t st, int pool4) {
  if (d->C % 64 || d->stride_h > 8 || d->stride_w > 8 || d->R > 256 || d->S > 256 || d->dil_w > 1 ||
      (d->pix_pitch && d->pix_pitch != d->C)) {
    a3d_set_error("fp8 conv fwd: needs C %% 64 == 0 (64- or 128-byte pixels), no dil_w / pix_pitch views (C=%d)", d->C);
    return A3D_ENOTSUP;
  }
  const int kc = d->C % 128 == 0 ? 128 : 64;        // channels = bytes per TMA load
  const int cblocks = d->C / kc;
  const int num_kb = d->R * d->S * cblocks;
  const long long M = (long long)d->N * d->P * d->Q;
  const long long J = (long long)d->R * d->S * d->C;
  CUtensorMap tmA;
  int rc = make_tmap_im2col(ctx, &tmA, x, d->N, d->H, d->W, d->C, -d->pad_t, -d->pad_l, d->P, d->Q, d->stride_h,
                            d->stride_w, kc, 128, 1);
  if (rc) return rc;
  tc::Params p{};
  p.M = (int)M; p.N = d->K; p.num_kb = num_kb; p.kb_per_split = num_kb; p.a_mode = tc::A_IM2COL;
  p.PQ = d->P * d->Q; p.Q = d->Q; p.sh = d->stride_h; p.sw = d->stride_w; p.lower_h = -d->pad_t; p.lower_w = -d->pad_l;
  p.S = d->S; p.cblocks = cblocks;
  p.rs = x_scale; p.rs_div = p.PQ; p.cs = w_scale;
  if (pool4) {
    if (d->K != 256 || y_dtype != A3D_BF16 || d->ldy % 8 || (reinterpret_cast<uintptr_t>(y) & 15)) {
      a3d_set_error("fp8 conv pool4 fwd: needs K == 256 (4 x 64) and a bf16 output with 16-byte aligned rows");
      return A3D_ENOTSUP;
    }
    CUtensorMap tmB;
    rc = make_tmap_2d(ctx, &tmB, w, 256, J, J, kc, 256, 1);
    if (rc) return rc;
    p.epi = tc::EPI_POOL4_BF16; p.out = y; p.ldo = d->ldy; p.bias = bias; p.flags = flags;
    auto run = [&](int c) -> int {
      if (kc == 64) return c ? launch_cfg<CfgF8<256, 64, 3>>(ctx, tmA, tmB, p, 1, st) : launch_cfg<CfgF8<256, 64>>(ctx, tmA, tmB, p, 1, st);
      return c ? launch_cfg<CfgF8<256, 128, 3>>(ctx, tmA, tmB, p, 1, st) : launch_cfg<CfgF8<256, 128>>(ctx, tmA, tmB, p, 1, st);
    };
    TuneKey key{};
    const int kv[16] = {7, d->N, d->H, d->W, d->C, d->K, d->R, d->S, d->stride_h, d->stride_w, d->pad_t, d->pad_l,
                        d->P, d->Q, d->ldy};
    memcpy(key.v, kv, sizeof(kv));
    const int best = autotune(key, 2, run, st);
    if (best < 0) return A3D_EINVAL;
    return run(best);
  }
  const bool can_split = ws && ws_bytes >= (size_t)M * d->K * sizeof(float);
  auto launch = [&](int bn, int splits, int deep) -> int {
    CUtensorMap tmB;
    int r = make_tmap_2d(ctx, &tmB, w, d->K, J, J, kc, bn, 1);
    if (r) return r;
    tc::Params q = p;
    if (!can_split) splits = 1;
    q.kb_per_split = ceil_div(num_kb, splits);
    splits = ceil_div(num_kb, q.kb_per_split);
    if (splits == 1) {
      q.epi = y_dtype == A3D_F32 ? tc::EPI_ROW_F32 : tc::EPI_ROW_BF16;
      q.out = y; q.ldo = d->ldy; q.bias = bias; q.flags = flags; q.atomic = 0;
      return launch_f8(ctx, bn, kc, deep, tmA, tmB, q, 1, st);
    }
    A3D_CHECK_CUDA(cudaMemsetAsync(ws, 0, (size_t)M * d->K * sizeof(float), st));
    q.epi = tc::EPI_ROW_F32; q.out = ws; q.ldo = d->K; q.bias = nullptr; q.flags = 0; q.atomic = 1;
    r = launch_f8(ctx, bn, kc, deep, tmA, tmB, q, splits, st);
    if (r) return r;
    return finish(ctx, reinterpret_cast<const float*>(ws), bias, nullptr, 0.f, y, y_dtype == A3D_F32, (size_t)M, d->K,
                  d->ldy, flags, st);
  };
  // candidate 0 = the bf16 heuristic's tile; then every width that pads K by at most a third, unsplit and with ~1-2
  // waves of split-K, with the default and (128-byte rows) the deeper ring
  struct Cand { int bn, splits, deep; };
  Cand cand[48];
  int nc = 0;
  auto tiles_of = [&](int bn) { return (int)(ceil_div(M, 128) * ceil_div(d->K, bn)); };
  {
    const int bn0 = pick_bn(d->K) < 32 ? 32 : pick_bn(d->K);
    cand[nc++] = {bn0, can_split ? pick_splits(ctx, tiles_of(bn0), num_kb, 8) : 1, 0};
  }
  static const int widths[] = {32, 64, 96, 128, 192, 256};
  for (int i = 0; i < 6; ++i) {
    const int bn = widths[i];
    if (ceil_div(d->K, bn) * bn > d->K + d->K / 3 + 15) continue;
    const int tiles = tiles_of(bn);
    const int sopts[3] = {1, ctx->sm_count / tiles, 2 * ctx->sm_count / tiles};
    for (int t = 0; t < 3; ++t) {
      int sp = sopts[t];
      const int max_s = num_kb / 8 > 0 ? num_kb / 8 : 1;
      if (sp > max_s) sp = max_s;
      if (sp < 1 || !can_split) sp = 1;
      for (int deep = 0; deep < 2; ++deep) {
        if (deep && (kc != 128 || bn == 32)) continue;
        bool dup = false;
        for (int k = 0; k < nc; ++k) dup |= cand[k].bn == bn && cand[k].splits == sp && cand[k].deep == deep;
        if (!dup && nc < 48) cand[nc++] = {bn, sp, deep};
      }
    }
  }
  if (const char* force = getenv("A3D_FP8_CONV_FORCE")) {            // "bn,splits,deep": tests and A/B runs
    int fbn = 0, fsp = 1, fd = 0;
    if (sscanf(force, "%d,%d,%d", &fbn, &fsp, &fd) >= 1 && fbn > 0) return launch(fbn, fsp, fd);
  }
  TuneKey key{};
  const int kv[16] = {6, d->N, d->H, d->W, d->C, d->K, d->R, d->S, d->stride_h, d->stride_w, d->pad_t, d->pad_l,
                      d->P, d->Q, d->ldy, y_dtype * 2 + (can_split ? 1 : 0)};
  memcpy(key.v, kv, sizeof(kv));
  const int best = autotune(key, nc, [&](int c) { return launch(cand[c].bn, cand[c].splits, cand[c].deep); }, st);
  if (best < 0) return A3D_EINVAL;
  return launch(cand[best].bn, cand[best].splits, cand[best].deep);
}

// dense forward, batch M <= 256 as the UMMA N dimension (as a3d_tc_dense_fwd): the weights [N][K] stream once as the
// 128-row operand; acc_ws [M][N] f32 receives the scaled split-K sums, `finish` adds bias and activation.
int a3d_tc_dense_fwd_fp8(a3d_ctx* ctx, const uint8_t* x, int ldx, const float* x_scale, const uint8_t* w,
                         const float* w_scale, const float* bias, void* y, int y_dtype, float* acc_ws, int M, int N, int K,
                         unsigned flags, cudaStream_t st) {
  if (K % 128 || ldx % 16 || M > 256 || !acc_ws) {
    a3d_set_error("fp8 dense fwd: needs K %% 128 == 0, ldx %% 16 == 0, batch <= 256, a workspace (K=%d M=%d)", K, M);
    return A3D_ENOTSUP;
  }
  const int bn = M <= 32 ? 32 : M <= 64 ? 64 : M <= 128 ? 128 : 256;
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, w, N, K, K, 128, 128, 1);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, x, M, K, ldx, 128, bn, 1);
  if (rc) return rc;
  tc::Params p{};
  p.M = N; p.N = M; p.num_kb = K / 128; p.a_mode = tc::A_TILED;
  p.rs = w_scale; p.rs_div = 1; p.cs = x_scale;
  p.epi = tc::EPI_COL_F32; p.out = acc_ws; p.ldo = N; p.atomic = 1;
  const int tiles = ceil_div(N, 128);
  int splits0 = pick_splits(ctx, tiles, p.num_kb, 4);
  if (splits0 * tiles < 2 * ctx->sm_count && p.num_kb / (splits0 * 2) >= 4) splits0 *= 2;
  auto launch = [&](int splits) -> int {          // splits >= 1000: interleaved k-blocks (Params::kb_interleave)
    tc::Params q = p;
    q.kb_interleave = splits >= 1000;
    splits %= 1000;
    q.kb_per_split = ceil_div(q.num_kb, splits);
    splits = ceil_div(q.num_kb, q.kb_per_split);
    A3D_CHECK_CUDA(cudaMemsetAsync(acc_ws, 0, (size_t)M * N * sizeof(float), st));
    int r = launch_f8(ctx, bn, 128, 0, tmA, tmB, q, splits, st);
    if (r) return r;
    return finish(ctx, acc_ws, bias, nullptr, 0.f, y, y_dtype == A3D_F32, (size_t)M, N, N, flags, st);
  };
  int cand[24];
  int nc = split_candidates(ctx, tiles, p.num_kb, splits0, cand);
  for (int i = 0, n0 = nc; i < n0; ++i)
    if (cand[i] > 1) cand[nc++] = 1000 + cand[i];
  if (const char* force = getenv("A3D_FP8_DENSE_FORCE")) return launch(atoi(force));
  TuneKey key{};
  const int kv[16] = {8, M, N, K, ldx, y_dtype, (int)flags};
  memcpy(key.v, kv, sizeof(kv));
  const int best = autotune(key, nc, [&](int c) { return launch(cand[c]); }, st);
  if (best < 0) return A3D_EINVAL;
  return launch(cand[best]);
}

// ---- E4M3 (kind::f8f6f4) engine test hook: D[M][N] (f32) = A * B^T with A [M][K], B [N][K] E4M3 codes, K-major,
// kcb = 128 or 64 bytes of K per stage; row / column scales when rs / cs are given (rs_div rows share one row scale).
extern "C" int a3d_debug_tc_gemm_fp8(a3d_ctx* ctx, const uint8_t* A, const uint8_t* B, float* D, int M, int N, int K, int bn,
                                     int kcb, int splits, const float* rs, int rs_div, const float* cs, void* stream) {
  A3D_REQUIRE(ctx && A && B && D && (!rs == !cs) && rs_div >= 1, "debug gemm fp8: bad argument");
  A3D_REQUIRE((kcb == 128 || kcb == 64) && K % kcb == 0, "debug gemm fp8: kcb 128 or 64 and K %% kcb == 0");
  cudaStream_t st = as_stream(stream);
  CUtensorMap tmA, tmB;
  int rc = make_tmap_2d(ctx, &tmA, A, M, K, K, kcb, 128, 1);
  if (rc) return rc;
  rc = make_tmap_2d(ctx, &tmB, B, N, K, K, kcb, bn, 1);
  if (rc) return rc;
  tc::Params p{};
  p.M = M; p.N = N; p.num_kb = K / kcb; p.a_mode = tc::A_TILED;
  p.rs = rs; p.rs_div = rs_div; p.cs = cs;
  if (splits < 1) splits = 1;
  p.kb_per_split = ceil_div(p.num_kb, splits);
  splits = ceil_div(p.num_kb, p.kb_per_split);
  p.epi = tc::EPI_ROW_F32; p.out = D; p.ldo = N; p.atomic = splits > 1;
  if (splits > 1) A3D_CHECK_CUDA(cudaMemsetAsync(D, 0, (size_t)M * N * sizeof(float), st));
  return launch_f8(ctx, bn, kcb, 0, tmA, tmB, p, splits, st);
}

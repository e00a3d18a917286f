// metrics.cu -- depth-estimation metrics (Eigen et al. 2014) of a predicted depth map against full-resolution ground truth,
// beyond the reference (it has no evaluation).  See a3d_depth_metrics in include/a3d.h for the definitions.
//
// One thread-block cluster of S CTAs per image (S in {1,2,4,8}, chosen so that B*S fills the SMs: B = 1 still spreads over
// 8 SMs).  CTA rank r owns the r-th contiguous share of the image's ground-truth pixels; every pixel samples the
// prediction with the TF1 bilinear mapping of a3d_resize_bilinear_tf1 (tf1_coord / tf1_lerp, common.cuh -- the same
// instructions, so the same float), gathering the small prediction map through L1 / L2.  No upsampled map is written.
//
// Median scaling: an exact radix select of the rank-floor((n-1)/2) element of gt and of the clamped prediction p~ over the
// valid pixels, both in the same three passes over the float bit patterns (all values are > 0 after the validity test and
// the clamp, so the bit patterns order like the floats): digits of 11, 11 and 10 bits.  Each CTA histograms its share in
// shared memory; after a cluster barrier every CTA sums the S histograms through distributed shared memory
// (cluster.map_shared_rank), scans them and keeps the digit that holds the wanted rank.  Two histogram buffers alternate,
// so one barrier per pass separates the writers of pass p+1 from the readers of pass p.  A last pass applies the scale and
// reduces the sums: float32 per-thread partials, combined across threads and across the cluster in float64 in a fixed
// order (no float atomics), so a captured graph replays to identical sums.
//
// Affine (scale-and-shift) alignment: one pass of float64 per-thread moments (n, sum p~, sum g, sum p~^2, sum p~ g) and
// the float32 min / max of p~ (an exact test for a constant p~, which the moments cannot give after rounding), reduced
// in the same fixed order across warps and, after one cluster barrier, across the cluster: every CTA reads the S
// partials over DSMEM in rank order, so all CTAs derive the same (s, t) before the final pass.
#include "common.cuh"
#include <cooperative_groups.h>
#include <cmath>

namespace cg = cooperative_groups;

namespace {

constexpr int kThreads = 512;
constexpr int kBins = 2048;                 // largest digit: 11 bits
constexpr int kPasses = 3;
__constant__ int kShift[kPasses] = {21, 10, 0};
__constant__ int kWidth[kPasses] = {11, 11, 10};

struct Pixel {
  float g, p;        // ground truth, clamped prediction p~
  bool valid, nonfinite;
};

// Ground-truth pixel (row, col) of one image and the prediction sampled there.
__device__ __forceinline__ Pixel load_pixel(const float* __restrict__ pred, int ph, int pw, const float* __restrict__ gt,
                                            int row, int col, int gw, float sy, float sx, float lo, float hi) {
  Pixel px;
  px.g = __ldg(gt + (size_t)row * gw + col);
  px.valid = px.g > lo && px.g <= hi;
  int y0, y1, x0, x1;
  float ly, lx;
  tf1_coord(row, sy, ph, y0, y1, ly);
  tf1_coord(col, sx, pw, x0, x1, lx);
  const float* r0 = pred + (size_t)y0 * pw;
  const float* r1 = pred + (size_t)y1 * pw;
  float v = tf1_lerp(__ldg(r0 + x0), __ldg(r0 + x1), __ldg(r1 + x0), __ldg(r1 + x1), ly, lx);
  px.nonfinite = !isfinite(v);
  px.p = isnan(v) ? lo : fminf(fmaxf(v, lo), hi);
  return px;
}

// Visits the valid pixels of the CTA's share [begin, end) of an image's gh*gw pixels, kThreads apart, kUnroll pixels per
// thread at a time: their loads are issued together (one dependent HBM + L1 round trip per kUnroll pixels, not per pixel),
// and the row / column advance needs no division per pixel.
constexpr int kUnroll = 4;
template <class F>
__device__ __forceinline__ void for_pixels(int begin, int end, const float* __restrict__ pred, int ph, int pw,
                                           const float* __restrict__ gt, int gw, float sy, float sx, float lo, float hi,
                                           F&& f) {
  int i = begin + (int)threadIdx.x;
  if (i >= end) return;
  int row = i / gw, col = i - row * gw;
  for (; i < end; i += kUnroll * kThreads) {
    Pixel px[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      if (i + u * kThreads < end) {
        px[u] = load_pixel(pred, ph, pw, gt, row, col, gw, sy, sx, lo, hi);
      } else {
        px[u].valid = false;
      }
      col += kThreads;
      while (col >= gw) { col -= gw; ++row; }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; ++u)
      if (px[u].valid) f(px[u]);
  }
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ double warp_max_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Alignment statistics of the affine mode: sums n, sum p~, sum g, sum p~^2, sum p~ g, then maxima -min p~, max p~.
constexpr int kAlign = 7, kAlignSums = 5;

// Block-wide exclusive scan of one value per thread; returns the prefix, `total` = the block's sum.
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* warp_tot, uint32_t& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  uint32_t before = 0;
  total = 0;
  for (int w = 0; w < kThreads / 32; ++w) {
    uint32_t t = warp_tot[w];
    if (w < warp) before += t;
    total += t;
  }
  __syncthreads();                          // warp_tot is reused by the next scan
  return before + inc - v;
}

template <int MODE>
__global__ void __launch_bounds__(kThreads) depth_metrics_kernel(const float* __restrict__ pred, int ph, int pw,
                                                                 const float* __restrict__ gt, int gh, int gw, float lo,
                                                                 float hi, double* __restrict__ sums,
                                                                 float* __restrict__ scale_out) {
  cg::cluster_group cluster = cg::this_cluster();
  const int S = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
  const int b = blockIdx.x / S;
  const int npix = gh * gw;
  const int begin = (int)((long long)npix * rank / S), end = (int)((long long)npix * (rank + 1) / S);
  const float sy = (float)ph / (float)gh, sx = (float)pw / (float)gw;     // as a3d_resize_bilinear_tf1 forms them
  pred += (size_t)b * ph * pw;
  gt += (size_t)b * npix;

  __shared__ uint32_t warp_tot[kThreads / 32];
  __shared__ double part[A3D_DM_SLOTS];
  float s = 1.f, t = 0.f;
  if constexpr (MODE == A3D_DM_SCALE_MEDIAN) {
    __shared__ uint32_t hist[2][2][kBins];       // [buffer][gt, p~][bin]
    __shared__ uint32_t found[2][2];             // [gt, p~][selected prefix, residual rank]
    uint32_t prefix[2] = {0u, 0u}, want[2] = {0u, 0u};
    uint32_t n = 0;
    for (int pass = 0; pass < kPasses; ++pass) {
      const int shift = kShift[pass], nb = 1 << kWidth[pass], top = shift + kWidth[pass];
      uint32_t (*h)[kBins] = hist[pass & 1];
      for (int i = threadIdx.x; i < 2 * kBins; i += kThreads) (&h[0][0])[i] = 0u;
      __syncthreads();
      for_pixels(begin, end, pred, ph, pw, gt, gw, sy, sx, lo, hi, [&](const Pixel& px) {
        uint32_t bits[2] = {__float_as_uint(px.g), __float_as_uint(px.p)};
#pragma unroll
        for (int a = 0; a < 2; ++a)
          if (top == 32 || (bits[a] >> top) == (prefix[a] >> top)) atomicAdd(&h[a][(bits[a] >> shift) & (nb - 1)], 1u);
      });
      cluster.sync();                            // every CTA's histogram of this pass is complete
      // merge the S histograms (bins t*per .. t*per+per-1 per thread), then find the digit holding rank want[a]
      const int per = nb / kThreads;
#pragma unroll
      for (int a = 0; a < 2; ++a) {
        uint32_t c[kBins / kThreads];
        uint32_t mine = 0;
#pragma unroll
        for (int j = 0; j < kBins / kThreads; ++j) {
          uint32_t v = 0;
          if (j < per)
            for (int r = 0; r < S; ++r) v += cluster.map_shared_rank(&h[a][0], r)[threadIdx.x * per + j];
          c[j] = v;
          mine += v;
        }
        uint32_t total;
        uint32_t before = block_exclusive_scan(mine, warp_tot, total);
        if (pass == 0 && a == 0) n = total;
        if (pass == 0) want[a] = total ? (total - 1) / 2 : 0u;
#pragma unroll
        for (int j = 0; j < kBins / kThreads; ++j) {
          if (c[j] && before <= want[a] && want[a] < before + c[j]) {
            found[a][0] = prefix[a] | ((uint32_t)(threadIdx.x * per + j) << shift);
            found[a][1] = want[a] - before;
          }
          before += c[j];
        }
      }
      __syncthreads();
      if (n == 0) break;                         // no valid pixel: s = 1 (the same decision in every CTA)
#pragma unroll
      for (int a = 0; a < 2; ++a) { prefix[a] = found[a][0]; want[a] = found[a][1]; }
      __syncthreads();
    }
    if (n > 0) s = __uint_as_float(prefix[0]) / __uint_as_float(prefix[1]);
    // the next cluster.sync (before the partial sums are read) also keeps every CTA's histograms alive until the last
    // remote read of them has finished
  }
  if constexpr (MODE == A3D_DM_SCALE_AFFINE) {
    uint32_t c = 0;
    double sp = 0.0, sg = 0.0, spp = 0.0, spg = 0.0;
    float pmin = INFINITY, pmax = -INFINITY;
    for_pixels(begin, end, pred, ph, pw, gt, gw, sy, sx, lo, hi, [&](const Pixel& px) {
      const double p = px.p, g = px.g;
      c += 1;
      sp += p;
      sg += g;
      spp += p * p;
      spg += p * g;
      pmin = fminf(pmin, px.p);
      pmax = fmaxf(pmax, px.p);
    });
    const double vals[kAlign] = {(double)c, sp, sg, spp, spg, -(double)pmin, (double)pmax};
    __shared__ double awarp[kThreads / 32][kAlign];
    __shared__ double apart[kAlign], atot[kAlign];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < kAlign; ++k) {
      double v = k < kAlignSums ? warp_sum_f64(vals[k]) : warp_max_f64(vals[k]);
      if (lane == 0) awarp[warp][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < kAlign) {
      const int k = threadIdx.x;
      double v = awarp[0][k];
      for (int w = 1; w < kThreads / 32; ++w) v = k < kAlignSums ? v + awarp[w][k] : fmax(v, awarp[w][k]);
      apart[k] = v;
    }
    cluster.sync();                              // every CTA's partials are complete
    if (threadIdx.x < kAlign) {
      const int k = threadIdx.x;
      double v = cluster.map_shared_rank(apart, 0)[k];
      for (int r = 1; r < S; ++r) {
        double x = cluster.map_shared_rank(apart, r)[k];
        v = k < kAlignSums ? v + x : fmax(v, x);
      }
      atot[k] = v;
    }
    __syncthreads();
    // the same float64 arithmetic on the same totals in every thread of every CTA; the final pass's cluster.sync keeps
    // apart alive until the last remote read of it has finished
    const double n = atot[0];
    if (n > 0.0) {
      const double mp = atot[1] / n, mg = atot[2] / n;
      const double sxx = atot[3] - atot[1] * mp, sxy = atot[4] - atot[1] * mg;
      const double sd = (-atot[5] < atot[6] && sxx > 0.0) ? sxy / sxx : 1.0;
      s = (float)sd;
      t = (float)(mg - sd * mp);
    }
  }

  // final pass: per-thread float32 partials
  float f_abs = 0.f, f_sqrel = 0.f, f_sq = 0.f, f_d = 0.f, f_d2 = 0.f, f_l10 = 0.f;
  uint32_t c_n = 0, c_d1 = 0, c_d2 = 0, c_d3 = 0, c_nf = 0;
  for_pixels(begin, end, pred, ph, pw, gt, gw, sy, sx, lo, hi, [&](const Pixel& px) {
    float p = px.p, g = px.g;
    if constexpr (MODE == A3D_DM_SCALE_MEDIAN) p = fminf(fmaxf(s * p, lo), hi);
    if constexpr (MODE == A3D_DM_SCALE_AFFINE) p = fminf(fmaxf(__fadd_rn(__fmul_rn(s, p), t), lo), hi);
    float q = p / g, qi = g / p;
    float diff = p - g, rel = q - 1.f;
    float d = logf(q);
    f_abs += fabsf(rel);
    f_sqrel += diff * rel;                       // (p-g)^2 / g
    f_sq += diff * diff;
    f_d += d;
    f_d2 += d * d;
    f_l10 += fabsf(d);
    float m = fmaxf(q, qi);
    c_n += 1;
    c_d1 += m < 1.25f;
    c_d2 += m < 1.5625f;
    c_d3 += m < 1.953125f;
    c_nf += px.nonfinite;
  });
  // float64 across the block (fixed shuffle tree, warps in order), then across the cluster in rank order
  const double vals[A3D_DM_SLOTS] = {(double)c_n, f_abs, f_sqrel, f_sq, f_d, f_d2, f_l10 * 0.43429448190325182,
                                     (double)c_d1, (double)c_d2, (double)c_d3, (double)c_nf};
  __shared__ double wpart[kThreads / 32][A3D_DM_SLOTS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < A3D_DM_SLOTS; ++k) {
    double v = warp_sum_f64(vals[k]);
    if (lane == 0) wpart[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < A3D_DM_SLOTS) {
    double v = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) v += wpart[w][threadIdx.x];
    part[threadIdx.x] = v;
  }
  cluster.sync();
  if (rank == 0) {
    if (threadIdx.x < A3D_DM_SLOTS) {
      double v = 0.0;
      for (int r = 0; r < S; ++r) v += cluster.map_shared_rank(part, r)[threadIdx.x];
      sums[(size_t)b * A3D_DM_SLOTS + threadIdx.x] = v;
    }
    if (threadIdx.x == 0 && scale_out) {
      if constexpr (MODE == A3D_DM_SCALE_AFFINE) {
        scale_out[2 * b] = s;
        scale_out[2 * b + 1] = t;
      } else {
        scale_out[b] = s;
      }
    }
  }
  cluster.sync();                                // rank 0's remote reads are done before any CTA exits
}

}  // namespace

static int cluster_size_for(a3d_ctx* ctx, int B) {
  int S = 8;
  while (S > 1 && (long long)B * S > ctx->sm_count) S >>= 1;
  return S;
}

extern "C" int a3d_depth_metrics(a3d_ctx* ctx, const float* pred, int B, int ph, int pw, const float* gt, int gh, int gw,
                                 float min_depth, float max_depth, int scale_mode, double* sums, float* scale,
                                 void* stream) {
  A3D_REQUIRE(ctx && pred && gt && sums, "depth_metrics: null argument");
  A3D_REQUIRE(B > 0 && ph > 0 && pw > 0 && gh > 0 && gw > 0 && (long long)gh * gw < (1ll << 31),
              "depth_metrics: bad shape");
  A3D_REQUIRE(min_depth > 0.f && min_depth < max_depth && std::isfinite(max_depth),
              "depth_metrics: need 0 < min_depth < max_depth (finite)");
  A3D_REQUIRE(scale_mode == A3D_DM_SCALE_NONE || scale_mode == A3D_DM_SCALE_MEDIAN || scale_mode == A3D_DM_SCALE_AFFINE,
              "depth_metrics: bad scale_mode");
  const int S = cluster_size_for(ctx, B);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(B * S);
  cfg.blockDim = dim3(kThreads);
  cfg.stream = as_stream(stream);
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = S; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (scale_mode == A3D_DM_SCALE_MEDIAN)
    A3D_CHECK_CUDA(cudaLaunchKernelEx(&cfg, depth_metrics_kernel<A3D_DM_SCALE_MEDIAN>, pred, ph, pw, gt, gh, gw,
                                      min_depth, max_depth, sums, scale));
  else if (scale_mode == A3D_DM_SCALE_AFFINE)
    A3D_CHECK_CUDA(cudaLaunchKernelEx(&cfg, depth_metrics_kernel<A3D_DM_SCALE_AFFINE>, pred, ph, pw, gt, gh, gw,
                                      min_depth, max_depth, sums, scale));
  else
    A3D_CHECK_CUDA(cudaLaunchKernelEx(&cfg, depth_metrics_kernel<A3D_DM_SCALE_NONE>, pred, ph, pw, gt, gh, gw,
                                      min_depth, max_depth, sums, scale));
  A3D_LAUNCH_OK(ctx);
  return 0;
}

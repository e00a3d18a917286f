// dense_stream.cu -- weight-streaming kernels for the MSDN layers that are HBM-bound, not tensor-bound:
//
//   * dense forward / dgrad at batch <= 32 (coarse/dense_0 12288 -> 4096, dense_1 4096 -> 4070,
//     src/models.py:228-232): 2 FLOP per weight byte, so the only thing that matters is streaming the bf16
//     weight matrix from HBM once, with enough bytes in flight.  A 128-row tcgen05 tile at batch 32 spends its
//     time in CTA prologues/epilogues (measured 28/15/12/25 us for 100/33/33/100 MB = 3.6/2.2/2.8/4.0 TB/s);
//     here every thread streams its own 16-byte pieces of the matrix through a private cp.async ring
//     (no block-wide synchronisation in the main loop) and feeds warp-level mma.sync m16n8k16 directly.
//   * fine/third (5x5x64 -> 1, src/models.py:250-251): per-pixel tap products on mma.sync, then a 25-point
//     stencil sum from shared memory; the 64-channel input is read once instead of 25 times.
//
// mma.sync fragment conventions (PTX ISA, m16n8k16 .bf16, g = lane >> 2, c = lane & 3):
//   A (16x16, row): a0 = (row g, k 2c..2c+1)  a1 = (row g+8, k 2c..2c+1)  a2 = (row g, k 2c+8..)  a3 = (row g+8, k 2c+8..)
//   B (16x8,  col): b0 = (k 2c..2c+1, col g)  b1 = (k 2c+8..2c+9, col g)
//   C (16x8)      : c0 = (row g, col 2c)  c1 = (row g, col 2c+1)  c2 = (row g+8, col 2c)  c3 = (row g+8, col 2c+1)
// The reduction index may be permuted freely as long as A and B use the same permutation, and so may the
// output columns; both freedoms are used so that every global access is a 16-byte load of consecutive elements.
#include "common.cuh"
#include <stdlib.h>

namespace {

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
  return v;
}
__device__ __forceinline__ uint32_t lds32(uint32_t saddr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(saddr));
  return v;
}
__device__ __forceinline__ void mma16816(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

constexpr int DS_THREADS = 256;
constexpr int DS_DEPTH = 4;          // cp.async ring depth (steps); DS_DEPTH - 1 steps are in flight per thread

// ------------------------------------------------------------------------------------------------ forward
// acc[b][n] += sum_{k in this CTA's range} x[b][k] * w[n][k]       (acc f32 [M][N], zeroed by the caller)
// CTA = 8 warps x 32 weight rows, all warps share one K range whose activations sit in shared memory.
// One step = 32 rows x 32 k per warp: thread (g, c) copies w[row][k0 + c*8 .. +7] for its 4 rows
// (row = 16*rg + 8*h + g).  The 8 k of a 16-byte piece are two MMA k-slots each: logical k {2c,2c+1} and
// {2c+8,2c+9} of MMA #1 are actual k c*8+{0,1} and c*8+{2,3}; MMA #2 takes c*8+{4..7}.
__global__ void __launch_bounds__(DS_THREADS, 2)
dense_fwd_stream_kernel(const uint16_t* __restrict__ w, const uint16_t* __restrict__ x, int ldx, float* __restrict__ acc,
                        int M, int N, int K, int kb_per) {
  extern __shared__ __align__(16) uint8_t ds_smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, c = lane & 3;
  const int kb0 = blockIdx.y * kb_per;
  int nkb = K / 64 - kb0;
  if (nkb > kb_per) nkb = kb_per;
  const int k_begin = kb0 * 64;
  const int xpitch = kb_per * 128 + 64;                       // bytes; +64: rows g, g+1 fall into different bank halves
  uint8_t* xs = ds_smem;                                      // [32][xpitch]
  const uint32_t stg = smem_addr(ds_smem + 32 * xpitch);      // [DS_DEPTH][4][256] x 16 B (slot, j, thread)

  const int n_base = blockIdx.x * 256 + warp * 32;
  const uint16_t* wrow[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int r = n_base + (j >> 1) * 16 + (j & 1) * 8 + g;
    if (r > N - 1) r = N - 1;                                 // clamped rows are computed and never stored
    wrow[j] = w + (size_t)r * K + k_begin + c * 8;
  }
  const int nsteps = nkb * 2;
  auto issue = [&](int step) {
    const uint32_t dst = stg + (uint32_t)(((step % DS_DEPTH) * 4) * DS_THREADS + tid) * 16u;
#pragma unroll
    for (int j = 0; j < 4; ++j) cp_async16(dst + (uint32_t)(j * DS_THREADS * 16), wrow[j] + step * 32);
  };
#pragma unroll
  for (int s = 0; s < DS_DEPTH - 1; ++s) {
    if (s < nsteps) issue(s);
    cp_async_commit();
  }
  // activations of this K range -> shared memory (rows >= M are zero)
  {
    const int cpr = nkb * 8;                                  // 16-byte chunks per row
    for (int i = tid; i < 32 * cpr; i += DS_THREADS) {
      const int r = i / cpr, ch = i - r * cpr;
      uint4 v = make_uint4(0, 0, 0, 0);
      if (r < M) v = __ldg(reinterpret_cast<const uint4*>(x + (size_t)r * ldx + k_begin + ch * 8));
      *reinterpret_cast<uint4*>(xs + r * xpitch + ch * 16) = v;
    }
  }
  __syncthreads();

  float d[2][4][4];
#pragma unroll
  for (int rg = 0; rg < 2; ++rg)
#pragma unroll
    for (int bb = 0; bb < 4; ++bb)
#pragma unroll
      for (int e = 0; e < 4; ++e) d[rg][bb][e] = 0.f;

  const uint32_t xs_thread = smem_addr(xs) + (uint32_t)(g * xpitch + c * 16);
  for (int step = 0; step < nsteps; ++step) {
    cp_async_wait<DS_DEPTH - 2>();                            // this thread's copies of `step` have landed
    const uint32_t src = stg + (uint32_t)(((step % DS_DEPTH) * 4) * DS_THREADS + tid) * 16u;
    uint4 wv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) wv[j] = lds128(src + (uint32_t)(j * DS_THREADS * 16));
#pragma unroll
    for (int bb = 0; bb < 4; ++bb) {
      const uint4 xv = lds128(xs_thread + (uint32_t)(bb * 8 * xpitch + step * 64));
#pragma unroll
      for (int rg = 0; rg < 2; ++rg) {
        mma16816(d[rg][bb], wv[rg * 2].x, wv[rg * 2 + 1].x, wv[rg * 2].y, wv[rg * 2 + 1].y, xv.x, xv.y);
        mma16816(d[rg][bb], wv[rg * 2].z, wv[rg * 2 + 1].z, wv[rg * 2].w, wv[rg * 2 + 1].w, xv.z, xv.w);
      }
    }
    // the slot of step - 1 is free (its values went through the MMAs above in program order): refill it
    const int nxt = step + DS_DEPTH - 1;
    if (nxt < nsteps) issue(nxt);
    cp_async_commit();
  }
#pragma unroll
  for (int rg = 0; rg < 2; ++rg)
#pragma unroll
    for (int bb = 0; bb < 4; ++bb)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int n = n_base + rg * 16 + g + (e >> 1) * 8;
        const int b = bb * 8 + 2 * c + (e & 1);
        if (n < N && b < M) atomicAdd(acc + (size_t)b * N + n, d[rg][bb][e]);
      }
}

// ------------------------------------------------------------------------------------------------ dgrad
// acc[b][k] += sum_{n in this CTA's range} dy[b][n] * w[n][k]       (acc f32 [M][K], zeroed by the caller)
// The reduction runs over weight ROWS while memory is contiguous along k, so the B fragment (pairs of
// consecutive reduction indices for one output column) is assembled from two rows with byte permutes:
// thread (g, c) copies w[n0 + {2c, 2c+1, 2c+8, 2c+9}][col0 + g*8 .. +7]; MMA j (0..7) has column g <-> col0 + g*8 + j.
// A = dy (batch x n) from shared memory.  Afterwards a thread owns, per batch row, 16 consecutive columns
// col0 + 16c .. +15 -> four 16-byte vector atomics.
// CTA = 8 warps x 64 columns, all warps share one range of weight rows.  One step = 16 rows.
__global__ void __launch_bounds__(DS_THREADS, 2)
dense_dgrad_stream_kernel(const uint16_t* __restrict__ w, const uint16_t* __restrict__ dy, int lddy,
                          float* __restrict__ acc, int M, int N, int K, int steps_per) {
  extern __shared__ __align__(16) uint8_t ds_smem[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, c = lane & 3;
  const int total_steps = (N + 15) / 16;
  const int step0 = blockIdx.y * steps_per;
  int nsteps = total_steps - step0;
  if (nsteps > steps_per) nsteps = steps_per;
  const int n_begin = step0 * 16;
  const int ypitch = ((steps_per * 32 + 127) / 128) * 128 + 16;    // bytes; +16: the 8 batch rows of a fragment load hit 32 banks
  uint8_t* ys = ds_smem;                                           // [32][ypitch]
  const uint32_t stg = smem_addr(ds_smem + 32 * ypitch);           // [DS_DEPTH][4][256] x 16 B

  const int col0 = blockIdx.x * 512 + warp * 64;
  const bool active = col0 < K;                                    // K % 64 == 0 (host)
  const uint16_t* wcol = w + col0 + g * 8;
  auto issue = [&](int step) {
    const uint32_t dst = stg + (uint32_t)(((step % DS_DEPTH) * 4) * DS_THREADS + tid) * 16u;
    const int nb = n_begin + step * 16 + 2 * c;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int r = nb + (j & 1) + (j >> 1) * 8;
      if (r > N - 1) r = N - 1;                                    // dy is zero there
      cp_async16(dst + (uint32_t)(j * DS_THREADS * 16), wcol + (size_t)r * K);
    }
  };
  if (active) {
#pragma unroll
    for (int s = 0; s < DS_DEPTH - 1; ++s) {
      if (s < nsteps) issue(s);
      cp_async_commit();
    }
  }
  // dy of this row range -> shared memory, zero beyond M / N
  {
    const int cpr = nsteps * 2;                                    // 16-byte chunks (8 elements) per row
    const bool vec_ok = (lddy % 8 == 0) && ((reinterpret_cast<uintptr_t>(dy) & 15) == 0);
    for (int i = tid; i < 32 * cpr; i += DS_THREADS) {
      const int r = i / cpr, ch = i - r * cpr;
      const int n = n_begin + ch * 8;
      uint4 v = make_uint4(0, 0, 0, 0);
      if (r < M && n < N) {
        const uint16_t* src = dy + (size_t)r * lddy + n;
        if (vec_ok && n + 8 <= N) {
          v = __ldg(reinterpret_cast<const uint4*>(src));
        } else {
          uint32_t t[4] = {0, 0, 0, 0};
          for (int e = 0; e < 8; ++e)
            if (n + e < N) t[e >> 1] |= (uint32_t)src[e] << ((e & 1) * 16);
          v = make_uint4(t[0], t[1], t[2], t[3]);
        }
      }
      *reinterpret_cast<uint4*>(ys + r * ypitch + ch * 16) = v;
    }
  }
  __syncthreads();
  if (!active) return;

  float d[2][8][4];
#pragma unroll
  for (int t = 0; t < 2; ++t)
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
      for (int e = 0; e < 4; ++e) d[t][j][e] = 0.f;

  const uint32_t ys_thread = smem_addr(ys) + (uint32_t)(g * ypitch + c * 4);
  for (int step = 0; step < nsteps; ++step) {
    cp_async_wait<DS_DEPTH - 2>();
    const uint32_t src = stg + (uint32_t)(((step % DS_DEPTH) * 4) * DS_THREADS + tid) * 16u;
    uint4 r0 = lds128(src), r1 = lds128(src + DS_THREADS * 16), r2 = lds128(src + 2 * DS_THREADS * 16),
          r3 = lds128(src + 3 * DS_THREADS * 16);
    uint32_t bp[8], bq[8];
    bp[0] = __byte_perm(r0.x, r1.x, 0x5410); bp[1] = __byte_perm(r0.x, r1.x, 0x7632);
    bp[2] = __byte_perm(r0.y, r1.y, 0x5410); bp[3] = __byte_perm(r0.y, r1.y, 0x7632);
    bp[4] = __byte_perm(r0.z, r1.z, 0x5410); bp[5] = __byte_perm(r0.z, r1.z, 0x7632);
    bp[6] = __byte_perm(r0.w, r1.w, 0x5410); bp[7] = __byte_perm(r0.w, r1.w, 0x7632);
    bq[0] = __byte_perm(r2.x, r3.x, 0x5410); bq[1] = __byte_perm(r2.x, r3.x, 0x7632);
    bq[2] = __byte_perm(r2.y, r3.y, 0x5410); bq[3] = __byte_perm(r2.y, r3.y, 0x7632);
    bq[4] = __byte_perm(r2.z, r3.z, 0x5410); bq[5] = __byte_perm(r2.z, r3.z, 0x7632);
    bq[6] = __byte_perm(r2.w, r3.w, 0x5410); bq[7] = __byte_perm(r2.w, r3.w, 0x7632);
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const uint32_t ya = ys_thread + (uint32_t)(t * 16 * ypitch + step * 32);
      const uint32_t a0 = lds32(ya), a1 = lds32(ya + 8 * ypitch), a2 = lds32(ya + 16), a3 = lds32(ya + 8 * ypitch + 16);
#pragma unroll
      for (int j = 0; j < 8; ++j) mma16816(d[t][j], a0, a1, a2, a3, bp[j], bq[j]);
    }
    const int nxt = step + DS_DEPTH - 1;
    if (nxt < nsteps) issue(nxt);
    cp_async_commit();
  }
#pragma unroll
  for (int t = 0; t < 2; ++t)
#pragma unroll
    for (int hi = 0; hi < 2; ++hi) {                               // batch row g (c0/c1) or g + 8 (c2/c3)
      const int b = t * 16 + g + hi * 8;
      if (b >= M) continue;
      float* dst = acc + (size_t)b * K + col0 + 16 * c;
#pragma unroll
      for (int half = 0; half < 2; ++half) {                       // columns 16c + half*8 + j  <->  fragment element half
        const int e = hi * 2 + half;
        atomicAdd(reinterpret_cast<float4*>(dst + half * 8),
                  make_float4(d[t][0][e], d[t][1][e], d[t][2][e], d[t][3][e]));
        atomicAdd(reinterpret_cast<float4*>(dst + half * 8 + 4),
                  make_float4(d[t][4][e], d[t][5][e], d[t][6][e], d[t][7][e]));
      }
    }
}

// ------------------------------------------------------------------------------------------------ K = 1 conv
// y[n,p,q] = bias + sum_{r,s,ch} x[n, p - pt + r, q - pl + s, ch] * w[r][s][ch]     (stride 1, C = 64, R*S <= 32)
// Stage 1: for every input pixel of the CTA's row band, all tap products t[tap][pixel] = <x[pixel], w[tap]> as one
//          [pixels x 64] x [64 x 32] mma.sync product (A = pixels straight from global memory, B = the filter
//          in registers), stored tap-major in shared memory.
// Stage 2: y[p][q] = sum_taps t[tap][(p + r, q - pl + s)], conflict-free (consecutive q).
// The input is read (band + halo)/band times instead of R*S times.
constexpr int K1_THREADS = 256;
__global__ void __launch_bounds__(K1_THREADS, 2)
conv_k1_tiled_kernel(const uint16_t* __restrict__ x, const uint16_t* __restrict__ w, const float* __restrict__ bias,
                     void* __restrict__ y, int y_f32, int H, int W, int R, int S, int pt, int pl, int P, int Q, int ldy,
                     unsigned flags, int band, int pixp) {
  extern __shared__ __align__(16) float k1_t[];                    // [R*S][pixp]
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, c = lane & 3;
  const int n = blockIdx.y;
  const int p0 = blockIdx.x * band;
  int rows_out = P - p0;
  if (rows_out > band) rows_out = band;
  const int rows_in = rows_out + R - 1;
  const int npix = rows_in * W;
  const int RS = R * S;
  const int h0 = p0 - pt;                                          // input row of tile row 0

  // filter fragments: B (k = channel, col = tap): tap nb*8 + g, channels h*32 + c*8 + m*4 + {0,1} / {2,3}
  uint32_t bf[4][2][2][2];
#pragma unroll
  for (int nb = 0; nb < 4; ++nb) {
    const int tap = nb * 8 + g;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (tap < RS) v = __ldg(reinterpret_cast<const uint4*>(w + (size_t)tap * 64 + h * 32 + c * 8));
      bf[nb][h][0][0] = v.x; bf[nb][h][0][1] = v.y; bf[nb][h][1][0] = v.z; bf[nb][h][1][1] = v.w;
    }
  }
  const int nblk = (npix + 15) / 16;
  const uint16_t* img = x + (size_t)n * H * W * 64;
  auto load_blk = [&](int mb, uint4 (&v)[4]) {
#pragma unroll
    for (int hi = 0; hi < 2; ++hi) {
      const int i = mb * 16 + g + hi * 8;
      const int row = i / W;
      const int ih = h0 + row;
      const bool ok = i < npix && ih >= 0 && ih < H;
      const uint16_t* px = img + ((size_t)ih * W + (i - row * W)) * 64 + c * 8;
#pragma unroll
      for (int h = 0; h < 2; ++h)
        v[hi * 2 + h] = ok ? __ldg(reinterpret_cast<const uint4*>(px + h * 32)) : make_uint4(0, 0, 0, 0);
    }
  };
  uint4 cur[4], nxt[4];
  if (warp < nblk) load_blk(warp, cur);
  for (int mb = warp; mb < nblk; mb += K1_THREADS / 32) {
    const bool more = mb + K1_THREADS / 32 < nblk;
    if (more) load_blk(mb + K1_THREADS / 32, nxt);
    float d[4][4];
#pragma unroll
    for (int nb = 0; nb < 4; ++nb)
#pragma unroll
      for (int e = 0; e < 4; ++e) d[nb][e] = 0.f;
#pragma unroll
    for (int nb = 0; nb < 4; ++nb)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        // cur[0 + h] = pixel g, cur[2 + h] = pixel g + 8
        mma16816(d[nb], cur[h].x, cur[2 + h].x, cur[h].y, cur[2 + h].y, bf[nb][h][0][0], bf[nb][h][0][1]);
        mma16816(d[nb], cur[h].z, cur[2 + h].z, cur[h].w, cur[2 + h].w, bf[nb][h][1][0], bf[nb][h][1][1]);
      }
#pragma unroll
    for (int nb = 0; nb < 4; ++nb)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int tap = nb * 8 + 2 * c + (e & 1);
        const int i = mb * 16 + g + (e >> 1) * 8;
        if (tap < RS) k1_t[tap * pixp + i] = d[nb][e];             // i < nblk * 16 <= pixp
      }
    if (more) {
#pragma unroll
      for (int q = 0; q < 4; ++q) cur[q] = nxt[q];
    }
  }
  __syncthreads();
  const float b0 = bias ? __ldg(bias) : 0.f;
  for (int o = tid; o < rows_out * Q; o += K1_THREADS) {
    const int pr = o / Q, q = o - pr * Q;
    float a = b0;
    for (int r = 0; r < R; ++r) {
      const float* trow = k1_t + (size_t)(r * S) * pixp + (pr + r) * W + (q - pl);
      for (int s = 0; s < S; ++s)
        if ((unsigned)(q - pl + s) < (unsigned)W) a += trow[s * pixp + s];
    }
    if (flags & A3D_EPI_RELU) a = fmaxf(a, 0.f);
    const size_t m = ((size_t)n * P + p0 + pr) * Q + q;
    if (y_f32) reinterpret_cast<float*>(y)[m * ldy] = a;
    else reinterpret_cast<uint16_t*>(y)[m * ldy] = f32_to_bf16_bits(a);
  }
}

}  // namespace

bool a3d_stream_dense_fwd_ok(int M, int N, int K, int ldx) { return M <= 32 && K % 64 == 0 && ldx % 8 == 0 && N >= 1; }
bool a3d_stream_dense_dgrad_ok(int M, int N, int K, int lddy) { return M <= 32 && K % 64 == 0 && N >= 1 && lddy >= N; }

// ctas: wanted number of CTAs (the tuner passes ~1x / 2x / 3x the resident slots); acc is zeroed here
int a3d_stream_dense_fwd(a3d_ctx* ctx, const uint16_t* x, int ldx, const uint16_t* w, float* acc, int M, int N, int K,
                         int ctas, cudaStream_t st) {
  const int groups = ceil_div(N, 256), num_kb = K / 64;
  int splits = ctas / groups;
  if (splits < 1) splits = 1;
  if (splits > num_kb) splits = num_kb;
  int kb_per = ceil_div(num_kb, splits);
  if (kb_per > 11) kb_per = 11;                                    // 46 KB of activations + 64 KB ring: two CTAs per SM
  splits = ceil_div(num_kb, kb_per);
  const size_t smem = 32 * (size_t)(kb_per * 128 + 64) + (size_t)DS_DEPTH * 4 * DS_THREADS * 16;
  static bool attr = false;
  if (!attr) {
    A3D_CHECK_CUDA(cudaFuncSetAttribute(dense_fwd_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 116 * 1024));
    attr = true;
  }
  A3D_CHECK_CUDA(cudaMemsetAsync(acc, 0, (size_t)M * N * sizeof(float), st));
  dense_fwd_stream_kernel<<<dim3(groups, splits), DS_THREADS, smem, st>>>(w, x, ldx, acc, M, N, K, kb_per);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

int a3d_stream_dense_dgrad(a3d_ctx* ctx, const uint16_t* dy, int lddy, const uint16_t* w, float* acc, int M, int N, int K,
                           int ctas, cudaStream_t st) {
  const int groups = ceil_div(K, 512), total_steps = ceil_div(N, 16);
  int splits = ctas / groups;
  if (splits < 1) splits = 1;
  if (splits > total_steps) splits = total_steps;
  int steps_per = ceil_div(total_steps, splits);
  if (steps_per > 44) steps_per = 44;                              // 45 KB of dy + 64 KB ring: two CTAs per SM
  splits = ceil_div(total_steps, steps_per);
  const size_t smem = 32 * (size_t)(((steps_per * 32 + 127) / 128) * 128 + 16) + (size_t)DS_DEPTH * 4 * DS_THREADS * 16;
  static bool attr = false;
  if (!attr) {
    A3D_CHECK_CUDA(cudaFuncSetAttribute(dense_dgrad_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 116 * 1024));
    attr = true;
  }
  A3D_CHECK_CUDA(cudaMemsetAsync(acc, 0, (size_t)M * K * sizeof(float), st));
  dense_dgrad_stream_kernel<<<dim3(groups, splits), DS_THREADS, smem, st>>>(w, dy, lddy, acc, M, N, K, steps_per);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

bool a3d_conv_k1_tiled_ok(const a3d_conv_desc* d) {
  return d->K == 1 && d->C == 64 && d->stride_h == 1 && d->stride_w == 1 && d->R * d->S <= 32 &&
         (size_t)d->R * d->S * (((d->R) * d->W + 15) / 16 * 16 / 32 * 32 + 36) * 4 <= 100 * 1024;
}

int a3d_conv_k1_tiled(a3d_ctx* ctx, const a3d_conv_desc* d, const uint16_t* x, const uint16_t* w, const float* bias,
                      void* y, int y_dtype, unsigned flags, cudaStream_t st) {
  // the tallest row band whose tap products fit ~100 KB (two CTAs per SM), at most 8 output rows
  int band = 8;
  auto pixp_of = [&](int b) { return ((b + d->R - 1) * d->W + 15) / 16 * 16 / 32 * 32 + 36; };   // >= npix16, == 4 mod 32 (conflict-free tap-major stores)
  while (band > 1 && (size_t)d->R * d->S * pixp_of(band) * 4 > 100 * 1024) --band;
  const int pixp = pixp_of(band);
  const size_t smem = (size_t)d->R * d->S * pixp * 4;
  static bool attr = false;
  if (!attr) {
    A3D_CHECK_CUDA(cudaFuncSetAttribute(conv_k1_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
    attr = true;
  }
  conv_k1_tiled_kernel<<<dim3(ceil_div(d->P, band), d->N), K1_THREADS, smem, st>>>(
      x, w, bias, y, y_dtype == A3D_F32, d->H, d->W, d->R, d->S, d->pad_t, d->pad_l, d->P, d->Q, d->ldy, flags, band, pixp);
  A3D_LAUNCH_OK(ctx);
  return 0;
}

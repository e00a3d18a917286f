// tc_gemm.cuh -- the tcgen05 / TMEM / TMA GEMM engine of liba3d (sm_100a only).
//
// One CTA computes one 128 x BN tile of  D[m][n] = sum_k A[m][k] * B[n][k]  with bf16 operands and
// fp32 accumulation in tensor memory:
//   warp 0     : TMA producer (one elected lane) -- tiled 2-D loads, or im2col-mode loads of an NHWC
//                activation tensor so that the convolution never materialises its im2col matrix
//   warp 1     : TMEM allocator + single-thread tcgen05.mma issuer
//   warps 2..5 : epilogue -- tcgen05.ld the accumulator (32 lanes per warp), bias / ReLU / cast, store
// Producer and issuer are decoupled by a STAGES-deep ring of shared-memory stages guarded by
// full/empty mbarriers; the issuer hands a stage back with tcgen05.commit.
//
// Operand layouts in shared memory are the canonical UMMA layouts that TMA produces directly:
//   K-major  : tile rows = M (or N) index, each row KCB bytes of K (128/64/32 -> SWIZZLE_128B/64B/32B)
//   MN-major : tile rows = K index (64 per stage), each row 128 B = 64 consecutive M (or N) elements,
//              one 8 KB block per 64 columns (SWIZZLE_128B)
//   K-major, KCB = 16 ("chunked", no swizzle): for tensors with only 8 channels per (virtual) pixel.
//              A stage holds 8 chunks of 8 K-elements; chunk j = rows x 16 B, i.e. contiguous 128-byte
//              core matrices (8 rows x 16 B).  Two adjacent chunks form one UMMA K = 16 step (LBO = chunk).
#pragma once
#include "common.cuh"
#include "ptx.cuh"

// Stage-ring budget per CTA and the minimum pipeline depth.  Measured on the MSDN step (tools/gpu/run_r.sh):
// 104 KB / >= 3 stages (two CTAs per SM) 1.128 ms; 72 KB / >= 2 stages (128x128 tiles: 64 KB, THREE CTAs per SM)
// 1.072 ms; 64 KB / >= 2 stages 1.123 ms.  The MSDN tiles have 9..100 k-blocks, so a CTA's life is dominated by
// its prologue (barrier init, TMEM alloc, first TMA round trip) and epilogue; a third resident CTA hides more of
// that than a deeper ring does.
#ifndef A3D_RING_KB
#define A3D_RING_KB 72
#endif
#ifndef A3D_MIN_STAGES
#define A3D_MIN_STAGES 2
#endif

namespace tc {

enum AMode : int { A_TILED = 0, A_IM2COL = 1 };
enum Epi : int {
  EPI_ROW_BF16 = 0,       // out_bf16[row*ldo + col] = act(acc + bias[col])
  EPI_ROW_F32 = 1,        // out_f32 [row*ldo + col] = act(acc + bias[col])   (atomicAdd when split-K)
  EPI_COL_F32 = 2,        // out_f32 [col*ldo + row] (+)= acc                  (transposed; dense layers)
  // (3: removed -- a TF-Adam epilogue that consumed dense weight-gradient tiles from TMEM lost 535 us vs 277 us to the
  //  optimizer-shaped mma.sync kernel of elementwise.cu)
  EPI_TMA_F32 = 4,        // out_f32[row*ldo + col] = act(acc + bias[col]) staged through shared memory and written
                          // with TMA (tmC): whole 128-byte lines per row instead of one 64-byte piece per thread;
                          // split-K accumulates with cp.reduce.async.bulk (.add.f32, performed in L2)
  EPI_TMA_BF16 = 5,       // out_bf16[row*ldo + col] = act(acc + bias[col]), 64-column slabs written with TMA
  EPI_POOL4_BF16 = 6,     // fused 2x2 max-pool of a convolution whose 4 window positions are 4 groups of 64 GEMM
                          // columns (BN = N = 256): out_bf16[row*ldo + c] = act(max_g acc[g*64 + c] + bias[c]),
                          // pool_idx[row*64 + c] (nullable) = first arg-max group
};

struct Params {
  int M, N;                 // valid rows of A / rows of B (GEMM M, N)
  int num_kb;               // k-blocks in total
  int kb_per_split;         // k-blocks handled by one blockIdx.z
  int kb_interleave;        // split z takes k-blocks z, z + gridDim.z, ... instead of a contiguous range: the CTAs of
                            // one row tile then read ADJACENT 128-byte pieces of the same rows at the same time
                            // (DRAM page locality when a weight matrix is streamed once: dense fwd / dgrad)
  // A operand addressing
  int a_mode;
  int a_k0;                 // tiled: first K coordinate
  int PQ, Q, sh, sw, lower_h, lower_w, S, cblocks;   // im2col
  int dil_w = 1;            // im2col: horizontal tap spacing in pixels (a3d_conv_desc::dil_w)
  // B operand addressing: coords (kb*KC, n0) for K-major, (n0, kb*64) for MN-major.
  // b_im2col (wgrad): B is the im2col view of an NHWC tensor, MN-major: K rows = 64 consecutive output
  // pixels, N blocks of BW channels; block jb <-> (tap = jb / cblocks, channel block jb % cblocks).
  int b_im2col;
  int RS;                   // number of filter taps (b_im2col)
  // epilogue
  int epi;
  void* out;
  long long ldo;
  const float* bias;
  unsigned flags;
  int atomic;               // accumulate with atomicAdd (split-K)
  uint8_t* pool_idx;        // EPI_POOL4_BF16: routing record (nullable)
  // E4M3 operands (ELT = 1): acc[row][col] * rs[row / rs_div] * cs[col] before bias / activation (rs == nullptr: none).
  // Convolutions: rs = per-image activation scales (rs_div = P*Q rows per image), cs = per-filter weight scales; dense
  // layers (weights are the row operand): rs = weight scales (rs_div = 1), cs = per-image activation scales.
  const float* rs = nullptr;
  int rs_div = 1;
  const float* cs = nullptr;
};

// ELT_ = operand element size in bytes: 2 = bf16 (kind::f16), 4 = f32 consumed as TF32 (kind::tf32), 1 = E4M3
// (kind::f8f6f4; K-major swizzled operands and 128-row tiles only, 32 elements per UMMA K step).  All shared-memory
// geometry below is in BYTES, so the two differ only in elements per row: a UMMA K step is always 32 bytes (16 bf16 /
// 8 tf32), an MN-major row always 128 bytes (64 bf16 / 32 tf32 elements), and an MN-major stage holds 128 / ELT K-rows.
template <int BN_, int KCB_, bool A_MN_, bool B_MN_, int B_BW_ = 64, int MIN_STAGES_ = A3D_MIN_STAGES, bool ADAM_ = false,
          int BM_ = 128, int ELT_ = 2>
struct Cfg {
  static constexpr int ELT = ELT_;
  static constexpr int KROWS = 128 / ELT_;                // MN-major: K rows per stage (64 bf16, 32 tf32)
  static constexpr int A_MN_BLOCKS = ELT_;                // MN-major A: 128-byte-wide blocks per 128 rows (2 / 4)
  static constexpr int A_MN_BLK_BYTES = KROWS * 128;      // one block: KROWS rows x 128 bytes (8 KB / 4 KB)
  static constexpr int A_MN_BLK_ELEMS = 128 / ELT_;       // M elements per block (64 / 32)
  static_assert(ELT_ == 2 || ((ELT_ == 4 || ELT_ == 1) && KCB_ != 16 && !ADAM_ && BM_ == 128),
                "tf32 / e4m3: swizzled operands, plain epilogues");
  static_assert(ELT_ != 1 || (!A_MN_ && !B_MN_), "e4m3: K-major operands only");
  static_assert(ELT_ == 2 || !B_MN_ || B_BW_ == 32, "tf32 MN-major B: 128-byte rows only (32-byte-atom swizzle)");
  // BM = 256: the CTA owns TWO 128-row accumulators (TMEM columns [0,BN) and [BN,2BN)) that share every B stage:
  // operand traffic per FLOP drops from (128+BN) to (256+BN)/2 rows per k-block -- the 5x5 layers are bound by
  // L2->SM operand bandwidth (conv2d_1: 819 MB per launch at ~13 TB/s), not by the tensor pipe.  K-major A only.
  static constexpr int MT = BM_ / 128;
  static_assert(BM_ == 128 || (BM_ == 256 && KCB_ != 16), "BM = 256: swizzled A");
  static_assert(!ADAM_, "the TF-Adam epilogue was removed (template slot kept so that Cfg<...> argument lists stay valid)");
  static constexpr int B_BW = B_BW_;                     // MN-major B: elements per block (row = B_BW * ELT = 128/64/32 bytes)
  static constexpr int B_BLK_BYTES = KROWS * B_BW_ * ELT_;   // KROWS K-rows x BW elements
  static constexpr int B_NBLK = BN_ / B_BW_;
  static constexpr int BM = BM_;
  static constexpr int BN = BN_;
  static constexpr int KCB = KCB_;                       // K-major: bytes of K per row per stage
  static constexpr bool A_MN = A_MN_, B_MN = B_MN_;
  static constexpr bool CHUNKED = (KCB_ == 16);           // 8 chunks of 16 B per stage, no swizzle
  static constexpr int KELEMS = (A_MN_ || B_MN_) ? KROWS : CHUNKED ? 64 : KCB_ / ELT_;   // K elements per stage
  static constexpr int A_SUB_BYTES = A_MN_ ? A_MN_BLOCKS * A_MN_BLK_BYTES : 128 * KCB_;  // one 128-row sub-tile (16 KB)
  static constexpr int A_BYTES = A_MN_ ? MT * A_SUB_BYTES : CHUNKED ? 8 * BM * 16 : BM * KCB_;
  static constexpr int B_BYTES = B_MN_ ? B_NBLK * B_BLK_BYTES : CHUNKED ? 8 * BN_ * 16 : BN_ * KCB_;
  static_assert(!CHUNKED || (!A_MN_ && !B_MN_), "chunked mode is K-major only");
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // A3D_RING_KB of stages per CTA: two or three CTAs (of this or of a concurrently running kernel on another
  // stream) fit on one SM, so one CTA's epilogue / prologue hides under the others' main loops.
  static constexpr int STAGES_RAW = (A3D_RING_KB * 1024) / STAGE_BYTES;
  static constexpr int STAGES = STAGES_RAW > 8 ? 8 : (STAGES_RAW < MIN_STAGES_ ? MIN_STAGES_ : STAGES_RAW);
  static constexpr int ACC_COLS = MT * BN_;
  static constexpr int TMEM_COLS = ACC_COLS <= 32 ? 32 : ACC_COLS <= 64 ? 64 : ACC_COLS <= 128 ? 128 : ACC_COLS <= 256 ? 256 : 512;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
  static_assert(!(A_MN_ || B_MN_) || KCB_ == 128, "MN-major operands use 128-byte rows");
  static_assert(!B_MN_ || BN_ % B_BW_ == 0, "MN-major B needs BN % BW == 0");
  static_assert(B_BW_ * ELT_ == 128 || B_BW_ * ELT_ == 64 || B_BW_ * ELT_ == 32, "MN-major block width: 128/64/32-byte rows");
  static_assert(BN_ % 16 == 0 && BN_ >= 16 && BN_ <= 256, "UMMA N");
};

// E4M3 tiles: v[j] (row `row`, columns col0 + j) *= row scale x column scale (Params::rs / cs)
template <class C, int NV>
__device__ __forceinline__ void scale_acc(const Params& p, int row, int col0, float* v) {
  if constexpr (C::ELT == 1) {
    if (p.rs) {
      const float r = row < p.M ? __ldg(p.rs + row / p.rs_div) : 0.f;
#pragma unroll
      for (int j = 0; j < NV; ++j) v[j] *= r * (col0 + j < p.N ? __ldg(p.cs + col0 + j) : 0.f);
    }
  }
}

template <class C>
__global__ void __launch_bounds__(192, 2)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmC, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment: required by the 128-byte swizzle atoms
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + C::STAGES * C::STAGE_BYTES);
  uint64_t* empty_bar = full_bar + C::STAGES;
  uint64_t* tmem_full_bar = empty_bar + C::STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * C::BM;
  const int n0 = blockIdx.y * C::BN;
  int kb_begin = blockIdx.z * p.kb_per_split, kb_step = 1;
  int kb_end = kb_begin + p.kb_per_split;
  if (kb_end > p.num_kb) kb_end = p.num_kb;
  int nkb = kb_end - kb_begin;            // host guarantees nkb >= 1
  if (p.kb_interleave) {
    kb_begin = blockIdx.z;
    kb_step = gridDim.z;
    nkb = (p.num_kb - kb_begin + kb_step - 1) / kb_step;
  }

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tmap(&tmA);
    ptx::prefetch_tmap(&tmB);
    for (int s = 0; s < C::STAGES; ++s) {
      ptx::mbar_init(&full_bar[s], 1);
      ptx::mbar_init(&empty_bar[s], 1);
    }
    ptx::mbar_init(tmem_full_bar, 1);
    ptx::fence_mbar_init();
  }
  if (warp == 1) ptx::tmem_alloc<C::TMEM_COLS>(tmem_slot);
  ptx::tc_fence_before_sync();
  __syncthreads();
  ptx::tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int n_img = 0, h0 = 0, w0 = 0;
      int n_img1 = 0, h01 = 0, w01 = 0;          // second 128-row sub-tile (BM = 256)
      // a second sub-tile that starts beyond M is not loaded at all (its accumulator rows are never stored)
      const bool sub1 = C::MT == 2 && m0 + 128 < p.M;
      const uint32_t stage_tx = C::STAGE_BYTES - ((C::MT == 2 && !sub1) ? C::A_SUB_BYTES : 0);
      if (p.a_mode == A_IM2COL) {
        // first output pixel of this tile -> base coordinates in input space
        n_img = m0 / p.PQ;
        int rem = m0 - n_img * p.PQ;
        int p0 = rem / p.Q, q0 = rem - p0 * p.Q;
        h0 = p.lower_h + p0 * p.sh;
        w0 = p.lower_w + q0 * p.sw;
        if (sub1) {
          n_img1 = (m0 + 128) / p.PQ;
          rem = m0 + 128 - n_img1 * p.PQ;
          p0 = rem / p.Q; q0 = rem - p0 * p.Q;
          h01 = p.lower_h + p0 * p.sh;
          w01 = p.lower_w + q0 * p.sw;
        }
      }
      for (int i = 0; i < nkb; ++i) {
        const int kb = kb_begin + i * kb_step;
        const int stage = i % C::STAGES;
        const uint32_t phase = (i / C::STAGES) & 1;
        ptx::mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sA = smem + stage * C::STAGE_BYTES;
        uint8_t* sB = sA + C::A_BYTES;
        ptx::mbar_expect_tx(&full_bar[stage], stage_tx);
        // ---- A
        if constexpr (C::CHUNKED) {
          // 8 im2col loads of 128 pixels x 8 channels (one per tap / channel-chunk), one 3-D load of B
#pragma unroll 1
          for (int j = 0; j < 8; ++j) {
            int ch = kb * 8 + j;
            int tap = ch / p.cblocks, cb = ch - tap * p.cblocks;
            int r = tap / p.S, sx = tap - r * p.S;      // taps beyond the filter meet zero-filled weights
            ptx::tma_load_im2col_4d(sA + j * (C::BM * 16), &tmA, &full_bar[stage], cb * 8, w0, h0, n_img,
                                    (uint16_t)(sx * p.dil_w), (uint16_t)r);
          }
          ptx::tma_load_3d(sB, &tmB, &full_bar[stage], 0, n0, kb * 8);
        } else if constexpr (!C::A_MN) {
          if (p.a_mode == A_TILED) {
            ptx::tma_load_2d(sA, &tmA, &full_bar[stage], p.a_k0 + kb * C::KELEMS, m0);
            if (sub1) ptx::tma_load_2d(sA + C::A_SUB_BYTES, &tmA, &full_bar[stage], p.a_k0 + kb * C::KELEMS, m0 + 128);
          } else {
            int tap = kb / p.cblocks, cb = kb - tap * p.cblocks;
            int r = tap / p.S, s = tap - r * p.S;
            ptx::tma_load_im2col_4d(sA, &tmA, &full_bar[stage], cb * C::KELEMS, w0, h0, n_img, (uint16_t)(s * p.dil_w),
                                    (uint16_t)r);
            if (sub1)
              ptx::tma_load_im2col_4d(sA + C::A_SUB_BYTES, &tmA, &full_bar[stage], cb * C::KELEMS, w01, h01, n_img1,
                                      (uint16_t)(s * p.dil_w), (uint16_t)r);
          }
        } else {
          // MN-major A: global [K rows][M cols]; 128-byte-wide boxes of KROWS K-rows (2 per 128 rows for bf16, 4 for tf32)
#pragma unroll
          for (int b = 0; b < C::A_MN_BLOCKS; ++b)
            ptx::tma_load_2d(sA + b * C::A_MN_BLK_BYTES, &tmA, &full_bar[stage], m0 + b * C::A_MN_BLK_ELEMS, kb * C::KROWS);
          if (sub1) {
#pragma unroll
            for (int b = 0; b < C::A_MN_BLOCKS; ++b)
              ptx::tma_load_2d(sA + C::A_SUB_BYTES + b * C::A_MN_BLK_BYTES, &tmA, &full_bar[stage],
                               m0 + 128 + b * C::A_MN_BLK_ELEMS, kb * C::KROWS);
          }
        }
        // ---- B
        if constexpr (C::CHUNKED) {
          // loaded above
        } else if constexpr (!C::B_MN) {
          ptx::tma_load_2d(sB, &tmB, &full_bar[stage], kb * C::KELEMS, n0);
        } else if (!p.b_im2col) {
#pragma unroll
          for (int j = 0; j < C::B_NBLK; ++j)
            ptx::tma_load_2d(sB + j * C::B_BLK_BYTES, &tmB, &full_bar[stage], n0 + j * C::B_BW, kb * C::KROWS);
        } else {
          // KROWS consecutive output pixels starting at kb*KROWS -> base coordinates in input space
          const int mk = kb * C::KROWS;
          const int ni = mk / p.PQ;
          const int rem = mk - ni * p.PQ;
          const int pp = rem / p.Q, qq = rem - pp * p.Q;
          const int hh = p.lower_h + pp * p.sh, ww = p.lower_w + qq * p.sw;
#pragma unroll 1
          for (int j = 0; j < C::B_NBLK; ++j) {
            int jb = blockIdx.y * C::B_NBLK + j;
            int tap = jb / p.cblocks, cb = jb - tap * p.cblocks;
            if (tap >= p.RS) tap = p.RS - 1;              // columns beyond N: loaded but never stored
            int r = tap / p.S, sx = tap - r * p.S;
            ptx::tma_load_im2col_4d(sB + j * C::B_BLK_BYTES, &tmB, &full_bar[stage], cb * C::B_BW, ww, hh, ni,
                                    (uint16_t)(sx * p.dil_w), (uint16_t)r);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    if (lane == 0) {
      constexpr uint32_t idesc = C::ELT == 4   ? ptx::make_idesc_tf32(128, C::BN, C::A_MN ? 1 : 0, C::B_MN ? 1 : 0)
                                 : C::ELT == 1 ? ptx::make_idesc_f8f6f4(128, C::BN, 0, 0)
                                               : ptx::make_idesc_bf16(128, C::BN, C::A_MN ? 1 : 0, C::B_MN ? 1 : 0);
      constexpr uint32_t k_layout =
          C::KCB == 128 ? ptx::LAYOUT_SW128 : C::KCB == 64 ? ptx::LAYOUT_SW64 : ptx::LAYOUT_SW32;
      for (int i = 0; i < nkb; ++i) {
        const int stage = i % C::STAGES;
        const uint32_t phase = (i / C::STAGES) & 1;
        ptx::mbar_wait(&full_bar[stage], phase);
        ptx::tc_fence_after_sync();
        const uint32_t sA = ptx::smem_u32(smem + stage * C::STAGE_BYTES);
        const uint32_t sB = sA + C::A_BYTES;
        // K-major : SBO = 8 rows * KCB bytes, LBO unused (1) ; K step = 32 B inside the swizzled row
        // MN-major: SBO = 1024 (next 8 K-rows), LBO = 8192 (next 64 MN elements) ; K step = 16 rows = 2048 B
        // MN-major tf32: the hardware transposes 32-byte units, so the canonical layout is the 128-byte swizzle with
        // 32-byte atomicity (TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B; descriptor layout 1): swizzle atoms of 4 K-rows
        // (SBO = 512 bytes) instead of 8 (SBO = 1024)
        constexpr uint32_t mn_layout = C::ELT == 4 ? ptx::LAYOUT_SW128_B32 : ptx::LAYOUT_SW128;
        constexpr uint32_t mn_sbo = C::ELT == 4 ? 512 : 1024;
        const uint64_t a_desc = C::A_MN      ? ptx::make_smem_desc(sA, C::A_MN_BLK_BYTES, mn_sbo, mn_layout)
                                : C::CHUNKED ? ptx::make_smem_desc(sA, C::BM * 16, 128, ptx::LAYOUT_NONE)
                                             : ptx::make_smem_desc(sA, 16, 8 * C::KCB, k_layout);
        // MN-major B with block width BW: row pitch BW*2 bytes, 8-row atom = 16*BW bytes (SBO),
        // next block of BW columns at 64 rows * BW*2 bytes (LBO), swizzle = row pitch
        constexpr uint32_t b_mn_layout = C::ELT == 4 ? ptx::LAYOUT_SW128_B32
                                         : C::B_BW * C::ELT == 128 ? ptx::LAYOUT_SW128
                                         : C::B_BW * C::ELT == 64 ? ptx::LAYOUT_SW64 : ptx::LAYOUT_SW32;
        constexpr uint32_t b_mn_sbo = C::ELT == 4 ? 512 : 8 * C::B_BW * C::ELT;
        const uint64_t b_desc = C::B_MN      ? ptx::make_smem_desc(sB, C::B_BLK_BYTES, b_mn_sbo, b_mn_layout)
                                : C::CHUNKED ? ptx::make_smem_desc(sB, C::BN * 16, 128, ptx::LAYOUT_NONE)
                                             : ptx::make_smem_desc(sB, 16, 8 * C::KCB, k_layout);
        // one UMMA covers 32 bytes of K: 16 bf16 / 8 tf32 / 32 e4m3 elements.  K-major: 32 bytes along the swizzled row;
        // MN-major: 32 / ELT K-rows of 128 (A) or B_BW * ELT (B) bytes
        constexpr int KSTEP = 32 / C::ELT;
        constexpr uint32_t a_step = C::A_MN ? ((KSTEP * 128) >> 4) : C::CHUNKED ? ((2 * C::BM * 16) >> 4) : (32 >> 4);
        constexpr uint32_t b_step =
            C::B_MN ? ((KSTEP * C::B_BW * C::ELT) >> 4) : C::CHUNKED ? ((2 * C::BN * 16) >> 4) : (32 >> 4);
#pragma unroll
        for (int k = 0; k < C::KELEMS / KSTEP; ++k) {
          if constexpr (C::ELT == 4) {
            ptx::umma_tf32(tmem_base, a_desc + (uint64_t)(k * a_step), b_desc + (uint64_t)(k * b_step), idesc,
                           (uint32_t)((i | k) != 0));
          } else if constexpr (C::ELT == 1) {
            ptx::umma_f8(tmem_base, a_desc + (uint64_t)(k * a_step), b_desc + (uint64_t)(k * b_step), idesc,
                         (uint32_t)((i | k) != 0));
          } else {
            ptx::umma_bf16(tmem_base, a_desc + (uint64_t)(k * a_step), b_desc + (uint64_t)(k * b_step), idesc,
                           (uint32_t)((i | k) != 0));
            if constexpr (C::MT == 2)            // second accumulator: next 128 rows of A, same B stage
              ptx::umma_bf16(tmem_base + (uint32_t)C::BN, a_desc + (uint64_t)((C::A_SUB_BYTES >> 4) + k * a_step),
                             b_desc + (uint64_t)(k * b_step), idesc, (uint32_t)((i | k) != 0));
          }
        }
        ptx::umma_commit(&empty_bar[stage]);       // frees the smem stage when these MMAs retire
      }
      ptx::umma_commit(tmem_full_bar);             // accumulator complete
    }
  } else {
    // ------------------------------------------------------------------ epilogue (warps 2..5)
    const int quarter = warp & 3;                  // TMEM lane quarter this warp may access
    ptx::mbar_wait(tmem_full_bar, 0);
    ptx::tc_fence_after_sync();
    const int m0_cta = m0;
    const uint32_t tmem_cta = tmem_base;
#pragma unroll 1
    for (int mt = 0; mt < C::MT; ++mt) {           // one pass per 128-row accumulator
    const int m0 = m0_cta + mt * 128;
    if (m0 >= p.M) break;                          // warp-uniform
    const uint32_t tmem_base = tmem_cta + (uint32_t)(mt * C::BN);
    const int row = m0 + quarter * 32 + lane;
    const bool row_ok = row < p.M;
    int c_begin = 0;
    if (p.epi == EPI_TMA_F32) {
      // The accumulator is complete, hence every TMA load has landed and every UMMA has read its stage: the
      // stage ring is free and serves as staging.  Per warp two 4 KB slabs (32 rows x 32 f32, SWIZZLE_128B:
      // 16-byte chunk j of row r lives at chunk j ^ (r & 7), which also makes the st.shared conflict-free).
      // Rows >= M and columns >= N are clipped by TMA.  A trailing 16-column piece (BN % 32) takes the
      // register path below.
      uint8_t* slab0 = smem + quarter * 8192;
      const int row0 = m0 + quarter * 32;
      constexpr int NCH = C::BN / 32;
      if (row0 < p.M) {                            // warp-uniform
#pragma unroll 1
        for (int ch = 0; ch < NCH; ++ch) {
          const int col0 = n0 + ch * 32;
          if (col0 >= p.N) break;                  // warp-uniform
          uint8_t* slab = slab0 + (ch & 1) * 4096;
          if (ch >= 2) {                           // the store issued two chunks ago has finished reading this slab
            if (lane == 0) ptx::bulk_wait_read<1>();
          }
          __syncwarp();
          uint32_t ra[16], rb[16];
          const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ch * 32);
          ptx::tmem_ld_x16(taddr, ra);
          ptx::tmem_ld_x16(taddr + 16, rb);
          ptx::tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int j = 0; j < 16; ++j) { v[j] = __uint_as_float(ra[j]); v[16 + j] = __uint_as_float(rb[j]); }
          scale_acc<C, 32>(p, row, col0, v);
          if (p.bias) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (col0 + j < p.N) v[j] += __ldg(p.bias + col0 + j);
          }
          if (p.flags & A3D_EPI_RELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
          }
          const uint32_t srow = ptx::smem_u32(slab) + (uint32_t)lane * 128u;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            ptx::st_shared_v4(srow + (uint32_t)((j ^ (lane & 7)) << 4), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          ptx::fence_proxy_async_smem();           // generic-proxy writes -> visible to the TMA (async proxy)
          __syncwarp();
          if (lane == 0) {
            if (p.atomic) ptx::tma_reduce_add_2d(&tmC, slab, col0, row0);
            else ptx::tma_store_2d(&tmC, slab, col0, row0);
            ptx::bulk_commit();
          }
        }
        if (lane == 0) ptx::bulk_wait_all();
        __syncwarp();
      }
      c_begin = NCH * 32;
    }
    if (p.epi == EPI_TMA_BF16) {
      // as above with 64 bf16 columns (= 128 bytes) per slab row; a tail of BN % 64 columns takes the register path
      uint8_t* slab0 = smem + quarter * 8192;
      const int row0 = m0 + quarter * 32;
      constexpr int NCH = C::BN / 64;
      if (row0 < p.M) {
#pragma unroll 1
        for (int ch = 0; ch < NCH; ++ch) {
          const int col0 = n0 + ch * 64;
          if (col0 >= p.N) break;
          uint8_t* slab = slab0 + (ch & 1) * 4096;
          if (ch >= 2) {
            if (lane == 0) ptx::bulk_wait_read<1>();
          }
          __syncwarp();
          const uint32_t srow = ptx::smem_u32(slab) + (uint32_t)lane * 128u;
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            uint32_t ra[16], rb[16];
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ch * 64 + half * 32);
            ptx::tmem_ld_x16(taddr, ra);
            ptx::tmem_ld_x16(taddr + 16, rb);
            ptx::tmem_ld_wait();
            float v[32];
#pragma unroll
            for (int j = 0; j < 16; ++j) { v[j] = __uint_as_float(ra[j]); v[16 + j] = __uint_as_float(rb[j]); }
            const int cbase = col0 + half * 32;
            scale_acc<C, 32>(p, row, cbase, v);
            if (p.bias) {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (cbase + j < p.N) v[j] += __ldg(p.bias + cbase + j);
            }
            if (p.flags & A3D_EPI_RELU) {
#pragma unroll
              for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
            }
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const int j = half * 4 + jj;
              ptx::st_shared_v4_b32(srow + (uint32_t)((j ^ (lane & 7)) << 4), pack_bf16x2(v[8 * jj], v[8 * jj + 1]),
                                    pack_bf16x2(v[8 * jj + 2], v[8 * jj + 3]), pack_bf16x2(v[8 * jj + 4], v[8 * jj + 5]),
                                    pack_bf16x2(v[8 * jj + 6], v[8 * jj + 7]));
            }
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            ptx::tma_store_2d(&tmC, slab, col0, row0);
            ptx::bulk_commit();
          }
        }
        if (lane == 0) ptx::bulk_wait_all();
        __syncwarp();
      }
      c_begin = NCH * 64;
    }
    if constexpr (C::BN == 256) {
      if (p.epi == EPI_POOL4_BF16) {
        uint8_t* slab = smem + quarter * 8192;
        const int row0 = m0 + quarter * 32;
        if (row0 < p.M) {
          const uint32_t srow = ptx::smem_u32(slab) + (uint32_t)lane * 128u;
          float rsc = 1.f;                         // E4M3: row scale; the column scales apply before the max
          if constexpr (C::ELT == 1) {
            if (p.rs) rsc = row_ok ? __ldg(p.rs + row / p.rs_div) : 0.f;
          }
#pragma unroll 1
          for (int cc = 0; cc < 4; ++cc) {
            uint32_t r0[16], r1[16], r2[16], r3[16];
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(cc * 16);
            __syncwarp();
            ptx::tmem_ld_x16(taddr, r0);
            ptx::tmem_ld_x16(taddr + 64, r1);
            ptx::tmem_ld_x16(taddr + 128, r2);
            ptx::tmem_ld_x16(taddr + 192, r3);
            ptx::tmem_ld_wait();
            float v[16];
            uint32_t gi[4] = {0, 0, 0, 0};
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float m = __uint_as_float(r0[j]);
              uint32_t g = 0;
              float a1 = __uint_as_float(r1[j]), a2 = __uint_as_float(r2[j]), a3 = __uint_as_float(r3[j]);
              if constexpr (C::ELT == 1) {
                if (p.rs) {
                  const int c = cc * 16 + j;
                  m *= rsc * __ldg(p.cs + c);
                  a1 *= rsc * __ldg(p.cs + 64 + c);
                  a2 *= rsc * __ldg(p.cs + 128 + c);
                  a3 *= rsc * __ldg(p.cs + 192 + c);
                }
              }
              if (a1 > m) { m = a1; g = 1; }       // strict '>' keeps the FIRST arg-max (TF MaxPoolGrad)
              if (a2 > m) { m = a2; g = 2; }
              if (a3 > m) { m = a3; g = 3; }
              if (p.bias) m += __ldg(p.bias + cc * 16 + j);
              if (p.flags & A3D_EPI_RELU) m = fmaxf(m, 0.f);
              v[j] = m;
              gi[j >> 2] |= g << ((j & 3) * 8);
            }
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
              const int j = cc * 2 + jj;
              ptx::st_shared_v4_b32(srow + (uint32_t)((j ^ (lane & 7)) << 4), pack_bf16x2(v[8 * jj], v[8 * jj + 1]),
                                    pack_bf16x2(v[8 * jj + 2], v[8 * jj + 3]), pack_bf16x2(v[8 * jj + 4], v[8 * jj + 5]),
                                    pack_bf16x2(v[8 * jj + 6], v[8 * jj + 7]));
            }
            if (p.pool_idx && row_ok)
              *reinterpret_cast<uint4*>(p.pool_idx + (size_t)row * 64 + cc * 16) = make_uint4(gi[0], gi[1], gi[2], gi[3]);
          }
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            ptx::tma_store_2d(&tmC, slab, 0, row0);
            ptx::bulk_commit();
            ptx::bulk_wait_all();
          }
          __syncwarp();
        }
        c_begin = C::BN;
      }
    }
#pragma unroll 1
    for (int c0 = c_begin; c0 < C::BN; c0 += 16) {
      const int col0 = n0 + c0;
      if (col0 >= p.N) break;                      // warp-uniform
      __syncwarp();                                // tcgen05.ld is .sync.aligned: reconverge first
      uint32_t r[16];
      ptx::tmem_ld_x16(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c0, r);
      ptx::tmem_ld_wait();
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
      scale_acc<C, 16>(p, row, col0, v);
      if (p.epi == EPI_COL_F32) {
        float* o = reinterpret_cast<float*>(p.out);
        if (row_ok) {
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            if (col0 + j < p.N) {
              float* dst = o + (long long)(col0 + j) * p.ldo + row;
              if (p.atomic) atomicAdd(dst, v[j]); else *dst = v[j];
            }
          }
        }
      } else {
        if (p.bias) {
#pragma unroll
          for (int j = 0; j < 16; ++j)
            if (col0 + j < p.N) v[j] += __ldg(p.bias + col0 + j);
        }
        if (p.flags & A3D_EPI_RELU) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (row_ok && (p.epi == EPI_ROW_BF16 || p.epi == EPI_TMA_BF16)) {
          uint16_t* o = reinterpret_cast<uint16_t*>(p.out) + (long long)row * p.ldo + col0;
          const bool vec = (col0 + 16 <= p.N) && ((reinterpret_cast<uintptr_t>(o) & 15) == 0);
          if (vec) {
            uint4 q0 = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]),
                                  pack_bf16x2(v[6], v[7]));
            uint4 q1 = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]),
                                  pack_bf16x2(v[14], v[15]));
            reinterpret_cast<uint4*>(o)[0] = q0;
            reinterpret_cast<uint4*>(o)[1] = q1;
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (col0 + j < p.N) o[j] = f32_to_bf16_bits(v[j]);
          }
        } else if (row_ok) {  // EPI_ROW_F32 (and the 16-column tail of EPI_TMA_F32)
          float* o = reinterpret_cast<float*>(p.out) + (long long)row * p.ldo + col0;
          if (p.atomic) {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (col0 + j < p.N) atomicAdd(o + j, v[j]);
          } else {
            const bool vec = (col0 + 16 <= p.N) && ((reinterpret_cast<uintptr_t>(o) & 15) == 0);
            if (vec) {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                reinterpret_cast<float4*>(o)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (col0 + j < p.N) o[j] = v[j];
            }
          }
        }
      }
    }
    }  // mt
  }

  ptx::tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after_sync();
    ptx::tmem_dealloc<C::TMEM_COLS>(tmem_base);
  }
}

}  // namespace tc

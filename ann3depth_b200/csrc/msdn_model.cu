// msdn_model.cu -- model-level entry points: the whole MSDN step / inference behind the C-ABI, so that a host in ANY
// language (no Python) can drive the reference's `session.run(model_op)` (src/ann3depth.py:126-127) for
// `models.msdn` (src/models.py:203-367): a3d_msdn_create / a3d_msdn_step / a3d_msdn_infer.
//
// The library still allocates nothing: the caller queries a3d_msdn_workspace_bytes(), hands ONE device buffer to
// a3d_msdn_create, and the net carves its parameter arena (f32 master, gradients, Adam slots, bf16 mirror -- same
// segment table and packed layouts as ann3depth_b200/params.py, so a packed arena is interchangeable between the two
// hosts), activations, routing records and scratch out of it.  Every launch goes to the caller's stream; a step has no
// host synchronisation and no allocation, i.e. it is CUDA-graph capturable once the first (autotuning) call is done.
// Schedule: the sequential single-stream form of ann3depth_b200/msdn.py (forward of both stacks + both losses; backward
// of the active tf.case branch with the dense weight gradients fused into TF-Adam up to batch A3D_DENSE_WGRAD_ADAM_MAX_M
// (separate wgrad + TF-Adam above it); TF-Adam of the branch's groups;
// global_step += 1).  BF16 storage, tcgen05 kernels.  The Python host adds the multi-stream overlap (stream placement as
// annotations on the same launch sequence: msdn.py's _Lanes), data parallelism and the TF32 mode on top of the same kernels.
#include "common.cuh"
#include <math.h>
#include <string.h>

namespace {
constexpr int IN_H = 228, IN_W = 304, OUT_H = 55, OUT_W = 74, N_PIX = OUT_H * OUT_W;     // src/models.py:282-283,269
constexpr float LAMBDA_OVER_N = 0.5f / (74 * 55);
enum Group { G_DENSE = 0, G_CONV = 1, G_FINEA = 2, G_FINEB = 3 };
const float GROUP_LR[4] = {0.1f, 0.001f, 0.001f, 0.01f};                                  // src/models.py:318-345
constexpr float BETA1 = 0.9f, EPS = 1e-8f;

struct Seg { const char* name; int shape[4]; int ndim; int group; size_t numel, offset, size; };
// arena order = ann3depth_b200/params.py msdn_specs(): backward order inside each optimizer group
Seg kSegs[] = {
    {"coarse/dense/dense_1/kernel", {4096, 4096, 0, 0}, 2, G_DENSE},   {"coarse/dense/dense_1/bias", {4070, 0, 0, 0}, 1, G_DENSE},
    {"coarse/dense/dense_0/kernel", {4096, 12288, 0, 0}, 2, G_DENSE},  {"coarse/dense/dense_0/bias", {4096, 0, 0, 0}, 1, G_DENSE},
    {"coarse/conv/conv2d_4/kernel", {256, 3, 3, 384}, 4, G_CONV},      {"coarse/conv/conv2d_4/bias", {256, 0, 0, 0}, 1, G_CONV},
    {"coarse/conv/conv2d_3/kernel", {384, 3, 3, 384}, 4, G_CONV},      {"coarse/conv/conv2d_3/bias", {384, 0, 0, 0}, 1, G_CONV},
    {"coarse/conv/conv2d_2/kernel", {384, 3, 3, 256}, 4, G_CONV},      {"coarse/conv/conv2d_2/bias", {384, 0, 0, 0}, 1, G_CONV},
    {"coarse/conv/conv2d_1/kernel", {256, 5, 5, 128}, 4, G_CONV},      {"coarse/conv/conv2d_1/bias", {256, 0, 0, 0}, 1, G_CONV},
    {"coarse/conv/conv2d_0/kernel", {96, 3, 3, 64}, 4, G_CONV},        {"coarse/conv/conv2d_0/bias", {96, 0, 0, 0}, 1, G_CONV},
    {"fine/third/kernel", {1, 5, 5, 64}, 4, G_FINEA},                  {"fine/third/bias", {1, 0, 0, 0}, 1, G_FINEA},
    {"fine/first/conv2d/kernel", {64, 5, 5, 16}, 4, G_FINEA},          {"fine/first/conv2d/bias", {64, 0, 0, 0}, 1, G_FINEA},
    {"fine/second/conv2d/kernel", {64, 5, 5, 64}, 4, G_FINEB},         {"fine/second/conv2d/bias", {64, 0, 0, 0}, 1, G_FINEB},
};
constexpr int NSEG = sizeof(kSegs) / sizeof(kSegs[0]);

size_t al256(size_t x) { return (x + 255) & ~(size_t)255; }

a3d_conv_desc make_desc(int N, int H, int W, int C, int K, int R, int S, int stride, bool same, int ldy = 0) {
  a3d_conv_desc d;
  memset(&d, 0, sizeof(d));
  d.N = N; d.H = H; d.W = W; d.C = C; d.K = K; d.R = R; d.S = S; d.stride_h = d.stride_w = stride;
  if (same) {                                   // TF SAME: out = ceil(in/s), extra padding goes bottom/right
    d.P = (H + stride - 1) / stride; d.Q = (W + stride - 1) / stride;
    int ph = (d.P - 1) * stride + R - H, pw = (d.Q - 1) * stride + S - W;
    d.pad_t = (ph > 0 ? ph : 0) / 2; d.pad_l = (pw > 0 ? pw : 0) / 2;
  } else {
    d.P = (H - R) / stride + 1; d.Q = (W - S) / stride + 1;
  }
  d.ldy = ldy ? ldy : K;
  d.impl = A3D_IMPL_AUTO;
  return d;
}

__global__ void set_f32_kernel(float* p, float v) { *p = v; }
__global__ void set_i64_kernel(int64_t* p, long long v) { *p = v; }
}  // namespace

struct a3d_msdn {
  a3d_ctx* ctx;
  int B, inH, inW, dH, dW, train;
  float beta2;
  uint64_t seed;
  long long global_step;
  int adam_t[4];
  Seg seg[NSEG];
  size_t total, group_lo[4], group_hi[4];
  // carved from the caller's workspace
  float *w, *g, *m, *v; uint16_t* wb;
  uint16_t *img4, *p0, *p1, *c2, *c3, *c4, *d0, *cat, *f2, *wbig;
  float *tar, *c0, *c1, *coarse, *fine, *losses, *lps, *lr_dev, *g_wbig, *dense_acc;
  uint8_t *i0, *i1, *if1, *keep, *mask_c0;
  int *emb_k, *emb_b;
  int64_t* step_dev;
  uint16_t *g_coarse, *g_fine, *g_d0, *g_c4, *g_c3, *g_c2, *g_p1, *g_c1, *g_p0, *g_c0, *g_f2, *g_cat, *g_f1big;
  void* scratch; size_t scratch_bytes;
  a3d_conv_desc d_c0, d_c1, d_c2, d_c3, d_c4, d_f1, d_f1w, d_f2, d_f3;
};

namespace {
// one pass over the layout: with base == nullptr only the size is computed
size_t carve(a3d_msdn* n, uint8_t* base) {
  size_t off = 0;
  auto take = [&](size_t bytes) -> void* {
    void* p = base ? base + off : nullptr;
    off += al256(bytes);
    return p;
  };
  const size_t B = n->B, T = n->total;
  n->w = (float*)take(T * 4); n->g = (float*)take(T * 4); n->m = (float*)take(T * 4); n->v = (float*)take(T * 4);
  n->wb = (uint16_t*)take(T * 2);
  n->img4 = (uint16_t*)take(B * 57 * 76 * 64 * 2);
  n->tar = (float*)take(B * N_PIX * 4);
  n->c0 = (float*)take(B * 55 * 74 * 96 * 4);
  n->p0 = (uint16_t*)take(B * 27 * 37 * 128 * 2);
  n->i0 = (uint8_t*)take(B * 27 * 37 * 96);
  n->c1 = (float*)take(B * 27 * 37 * 256 * 4);
  n->p1 = (uint16_t*)take(B * 13 * 18 * 256 * 2);
  n->i1 = (uint8_t*)take(B * 13 * 18 * 256);
  n->c2 = (uint16_t*)take(B * 13 * 18 * 384 * 2);
  n->c3 = (uint16_t*)take(B * 13 * 18 * 384 * 2);
  n->c4 = (uint16_t*)take(B * 6 * 8 * 256 * 2);
  n->keep = (uint8_t*)take(B * 4096);
  n->d0 = (uint16_t*)take(B * 4096 * 2);
  n->coarse = (float*)take(B * N_PIX * 4);
  n->if1 = (uint8_t*)take(B * N_PIX * 64);
  n->cat = (uint16_t*)take(B * N_PIX * 64 * 2);
  n->wbig = (uint16_t*)take((size_t)256 * 576 * 2);
  n->emb_k = (int*)take((size_t)4 * 25600 * 4);
  n->emb_b = (int*)take((size_t)4 * 64 * 4);
  n->mask_c0 = (uint8_t*)take((size_t)96 * 576);
  n->f2 = (uint16_t*)take(B * N_PIX * 64 * 2);
  n->fine = (float*)take(B * N_PIX * 4);
  n->losses = (float*)take(2 * 4);
  n->lps = (float*)take(2 * B * 4);
  n->lr_dev = (float*)take(4 * 4);
  n->step_dev = (int64_t*)take(8);
  n->dense_acc = (float*)take(B * 12288 * 4);
  if (n->train) {
    n->g_coarse = (uint16_t*)take(B * 4096 * 2);
    n->g_fine = (uint16_t*)take(B * N_PIX * 2);
    n->g_d0 = (uint16_t*)take(B * 4096 * 2);
    n->g_c4 = (uint16_t*)take(B * 6 * 8 * 256 * 2);
    n->g_c3 = (uint16_t*)take(B * 13 * 18 * 384 * 2);
    n->g_c2 = (uint16_t*)take(B * 13 * 18 * 384 * 2);
    n->g_p1 = (uint16_t*)take(B * 13 * 18 * 256 * 2);
    n->g_c1 = (uint16_t*)take(B * 27 * 37 * 256 * 2);
    n->g_p0 = (uint16_t*)take(B * 27 * 37 * 128 * 2);
    n->g_c0 = (uint16_t*)take(B * 55 * 74 * 96 * 2);
    n->g_f2 = (uint16_t*)take(B * N_PIX * 64 * 2);
    n->g_cat = (uint16_t*)take(B * N_PIX * 64 * 2);
    n->g_f1big = (uint16_t*)take(B * N_PIX * 256 * 2);
    n->g_wbig = (float*)take(((size_t)256 * 576 + 256) * 4);
  }
  // one scratch region for every convolution of the (sequential) step
  size_t sc = 0;
  const a3d_conv_desc* ds[] = {&n->d_c0, &n->d_c1, &n->d_c2, &n->d_c3, &n->d_c4, &n->d_f1, &n->d_f1w, &n->d_f2, &n->d_f3};
  for (const a3d_conv_desc* d : ds)
    for (int op = A3D_OP_FWD; op <= A3D_OP_WGRAD; ++op) {
      size_t b = a3d_conv2d_ws_bytes(n->ctx, d, op);
      if (b > sc) sc = b;
    }
  n->scratch_bytes = al256(sc ? sc : 256);
  n->scratch = take(n->scratch_bytes);
  return off;
}

void init_layout(a3d_msdn* n, a3d_ctx* ctx, int batch, int in_h, int in_w, int dh, int dw, int train) {
  memset(n, 0, sizeof(*n));
  n->ctx = ctx; n->B = batch; n->inH = in_h; n->inW = in_w; n->dH = dh; n->dW = dw; n->train = train;
  n->beta2 = 1.0f;                                     // the reference's third AdamOptimizer argument (src/models.py:309)
  n->seed = 2;
  size_t off = 0;
  for (int g = 0; g < 4; ++g) { n->group_lo[g] = (size_t)-1; n->group_hi[g] = 0; }
  for (int i = 0; i < NSEG; ++i) {
    Seg s = kSegs[i];
    s.numel = 1;
    for (int k = 0; k < s.ndim; ++k) s.numel *= (size_t)s.shape[k];
    s.offset = off;
    s.size = (s.numel + 63) / 64 * 64;
    off += s.size;
    n->seg[i] = s;
    if (s.offset < n->group_lo[s.group]) n->group_lo[s.group] = s.offset;
    if (s.offset + s.size > n->group_hi[s.group]) n->group_hi[s.group] = s.offset + s.size;
  }
  n->total = off;
  const int B = batch;
  n->d_c0 = make_desc(B, IN_H / 4, IN_W / 4, 64, 96, 3, 3, 1, false);        // 11x11x3 s4 as 3x3x64 s1 (s2d(4) image)
  n->d_c1 = make_desc(B, 27, 37, 128, 256, 5, 5, 1, true);
  n->d_c2 = make_desc(B, 13, 18, 256, 384, 3, 3, 1, true);
  n->d_c3 = make_desc(B, 13, 18, 384, 384, 3, 3, 1, true);
  n->d_c4 = make_desc(B, 13, 18, 384, 256, 3, 3, 2, false);
  n->d_f1 = make_desc(B, IN_H / 4, IN_W / 4, 64, 256, 3, 3, 1, false, 64);   // 9x9x3 s2 + pool as 3x3x64 -> 4 x 64
  n->d_f1w = make_desc(B, IN_H / 4, IN_W / 4, 64, 256, 3, 3, 1, false);
  n->d_f2 = make_desc(B, 55, 74, 64, 64, 5, 5, 1, true);
  n->d_f3 = make_desc(B, 55, 74, 64, 1, 5, 5, 1, true);
}

const Seg* find_seg(const a3d_msdn* n, const char* name) {
  for (int i = 0; i < NSEG; ++i)
    if (!strcmp(n->seg[i].name, name)) return &n->seg[i];
  return nullptr;
}
size_t seg_off(const a3d_msdn* n, const char* name) { return find_seg(n, name)->offset; }

// src/models.py:301-305,347-364 (batchsize = the per-replica batch)
int phase_of(long long step, int batch) {
  const long long sc = 2000000 / batch, sf = 1500000 / batch;
  return step < sc ? 1 : step < sc + sf ? 2 : 3;
}
float adam_lr_t(float lr, float b1, float b2, int t) {
  return (float)(lr * sqrt(1.0 - pow((double)b2, t)) / (1.0 - pow((double)b1, t)));
}

#define CK(call) do { int rc_ = (call); if (rc_) return rc_; } while (0)

int refresh_derived(a3d_msdn* n, void* st) {
  // re-embed the canonical fine/first filter into the pool-fused filter the kernels read
  return a3d_scatter_cast_bf16(n->ctx, n->w + seg_off(n, "fine/first/conv2d/kernel"), n->emb_k, 4, 25600, n->wbig, st);
}

int forward(a3d_msdn* n, const float* images, const float* depths, const uint8_t* keep_mask, void* st) {
  a3d_ctx* c = n->ctx;
  const int B = n->B;
  auto W = [&](const char* nm) { return n->wb + seg_off(n, nm); };
  auto Bi = [&](const char* nm) { return n->w + seg_off(n, nm); };
  CK(a3d_resize_bilinear_tf1_s2d(c, images, B, n->inH, n->inW, 3, n->img4, IN_H, IN_W, 4, 64, st));
  if (depths) CK(a3d_resize_bilinear_tf1(c, depths, B, n->dH, n->dW, 1, n->tar, OUT_H, OUT_W, 1, A3D_F32, st));
  // coarse (src/models.py:208-236)
  CK(a3d_conv2d_fwd(c, &n->d_c0, n->img4, W("coarse/conv/conv2d_0/kernel"), Bi("coarse/conv/conv2d_0/bias"), n->c0, A3D_F32,
                    A3D_EPI_RELU, n->scratch, n->scratch_bytes, st));
  CK(a3d_maxpool2x2_fwd_f32(c, n->c0, B, 55, 74, 96, n->p0, 128, n->i0, st));
  CK(a3d_conv2d_fwd(c, &n->d_c1, n->p0, W("coarse/conv/conv2d_1/kernel"), Bi("coarse/conv/conv2d_1/bias"), n->c1, A3D_F32,
                    A3D_EPI_RELU, n->scratch, n->scratch_bytes, st));
  CK(a3d_maxpool2x2_fwd_f32(c, n->c1, B, 27, 37, 256, n->p1, 256, n->i1, st));
  CK(a3d_conv2d_fwd(c, &n->d_c2, n->p1, W("coarse/conv/conv2d_2/kernel"), Bi("coarse/conv/conv2d_2/bias"), n->c2, A3D_BF16,
                    A3D_EPI_RELU, n->scratch, n->scratch_bytes, st));
  CK(a3d_conv2d_fwd(c, &n->d_c3, n->c2, W("coarse/conv/conv2d_3/kernel"), Bi("coarse/conv/conv2d_3/bias"), n->c3, A3D_BF16,
                    A3D_EPI_RELU, n->scratch, n->scratch_bytes, st));
  CK(a3d_conv2d_fwd(c, &n->d_c4, n->c3, W("coarse/conv/conv2d_4/kernel"), Bi("coarse/conv/conv2d_4/bias"), n->c4, A3D_BF16,
                    A3D_EPI_RELU, n->scratch, n->scratch_bytes, st));
  const uint8_t* mask = nullptr;
  if (n->train) {                                      // dropout is active iff train (src/models.py:230)
    if (keep_mask) {
      A3D_CHECK_CUDA(cudaMemcpyAsync(n->keep, keep_mask, (size_t)B * 4096, cudaMemcpyDeviceToDevice, as_stream(st)));
    } else {
      CK(a3d_bernoulli_mask(c, n->keep, (size_t)B * 4096, 0.5f, n->seed, n->step_dev, st));
    }
    mask = n->keep;
  }
  CK(a3d_dense_fwd(c, n->c4, 12288, W("coarse/dense/dense_0/kernel"), Bi("coarse/dense/dense_0/bias"), mask, 0.5f, n->d0,
                   A3D_BF16, n->dense_acc, B, 4096, 12288, A3D_EPI_RELU, A3D_IMPL_AUTO, st));
  CK(a3d_dense_fwd(c, n->d0, 4096, W("coarse/dense/dense_1/kernel"), Bi("coarse/dense/dense_1/bias"), nullptr, 0.f, n->coarse,
                   A3D_F32, n->dense_acc, B, N_PIX, 4096, 0, A3D_IMPL_AUTO, st));
  // fine (src/models.py:238-253)
  CK(a3d_conv2d_pool4_fwd(c, &n->d_f1, n->img4, n->wbig, Bi("fine/first/conv2d/bias"), n->cat, n->train ? n->if1 : nullptr,
                          A3D_EPI_RELU, n->scratch, n->scratch_bytes, st));
  CK(a3d_scatter_channel_bf16(c, n->coarse, n->cat, (size_t)B * N_PIX, 64, 63, st));
  CK(a3d_conv2d_fwd(c, &n->d_f2, n->cat, W("fine/second/conv2d/kernel"), Bi("fine/second/conv2d/bias"), n->f2, A3D_BF16,
                    A3D_EPI_RELU, n->scratch, n->scratch_bytes, st));
  CK(a3d_conv2d_fwd(c, &n->d_f3, n->f2, W("fine/third/kernel"), Bi("fine/third/bias"), n->fine, A3D_F32, 0, n->scratch,
                    n->scratch_bytes, st));
  if (!depths) return 0;                               // inference: no target, no losses
  // both losses (src/models.py:288-290); the gradient of the prediction comes out of the same pass
  CK(a3d_silog_loss(c, n->coarse, n->tar, B, N_PIX, LAMBDA_OVER_N, n->lps, n->losses, nullptr, n->train ? n->g_coarse : nullptr,
                    4096, st));
  CK(a3d_silog_loss(c, n->fine, n->tar, B, N_PIX, LAMBDA_OVER_N, n->lps + B, n->losses + 1, nullptr,
                    n->train ? n->g_fine : nullptr, N_PIX, st));
  return 0;
}

int adam_range(a3d_msdn* n, int group, size_t lo, size_t hi, void* st) {
  const int t = n->adam_t[group] > 0 ? n->adam_t[group] : 1;
  return a3d_adam_tf(n->ctx, n->w + lo, n->g + lo, n->m + lo, n->v + lo, n->wb + lo, hi - lo,
                     adam_lr_t(GROUP_LR[group], BETA1, n->beta2, t), BETA1, n->beta2, EPS, 1.0f, n->lr_dev + group, st);
}

int dense_wgrad_adam(a3d_msdn* n, const char* layer_kernel, const char* layer_bias, const uint16_t* x, int K, const uint16_t* dy,
                     int N, void* st) {
  const size_t ko = seg_off(n, layer_kernel), bo = seg_off(n, layer_bias);
  const int t = n->adam_t[G_DENSE] > 0 ? n->adam_t[G_DENSE] : 1;
  const float lr_t = adam_lr_t(GROUP_LR[G_DENSE], BETA1, n->beta2, t);
  CK(a3d_dense_wgrad_adam(n->ctx, x, K, dy, 4096, n->g + bo, n->w + ko, n->m + ko, n->v + ko, n->wb + ko, n->B, N, K, lr_t, BETA1,
                          n->beta2, EPS, 1.0f, n->lr_dev + G_DENSE, st));
  const size_t bs = find_seg(n, layer_bias)->size;
  return a3d_adam_tf(n->ctx, n->w + bo, n->g + bo, n->m + bo, n->v + bo, n->wb + bo, bs, lr_t, BETA1, n->beta2, EPS, 1.0f,
                     n->lr_dev + G_DENSE, st);
}

int backward_coarse(a3d_msdn* n, void* st) {
  a3d_ctx* c = n->ctx;
  const int B = n->B;
  auto W = [&](const char* nm) { return n->wb + seg_off(n, nm); };
  auto G = [&](const char* nm) { return n->g + seg_off(n, nm); };
  // dense_1: dgrad (+ DropoutGrad + ReluGrad of dense_0), then its fused wgrad + TF-Adam (after the last reader of w).
  // The fused kernel takes batches up to A3D_DENSE_WGRAD_ADAM_MAX_M; a larger batch writes both weight gradients and
  // updates the CoarseDense group once both dgrads have read the weights.
  const bool fused = B <= A3D_DENSE_WGRAD_ADAM_MAX_M;
  if (!fused)
    CK(a3d_dense_wgrad(c, n->d0, 4096, n->g_coarse, 4096, G("coarse/dense/dense_1/kernel"), G("coarse/dense/dense_1/bias"), B,
                       N_PIX, 4096, A3D_IMPL_AUTO, st));
  CK(a3d_dense_dgrad_act(c, n->g_coarse, 4096, W("coarse/dense/dense_1/kernel"), n->g_d0, n->dense_acc, B, N_PIX, 4096,
                         A3D_IMPL_AUTO, n->d0, n->keep, 0.5f, A3D_EPI_RELU, st));
  if (fused)
    CK(dense_wgrad_adam(n, "coarse/dense/dense_1/kernel", "coarse/dense/dense_1/bias", n->d0, 4096, n->g_coarse, N_PIX, st));
  else
    CK(a3d_dense_wgrad(c, n->c4, 12288, n->g_d0, 4096, G("coarse/dense/dense_0/kernel"), G("coarse/dense/dense_0/bias"), B, 4096,
                       12288, A3D_IMPL_AUTO, st));
  CK(a3d_dense_dgrad_act(c, n->g_d0, 4096, W("coarse/dense/dense_0/kernel"), n->g_c4, n->dense_acc, B, 4096, 12288, A3D_IMPL_AUTO,
                         n->c4, nullptr, 0.f, A3D_EPI_RELU, st));
  if (fused)
    CK(dense_wgrad_adam(n, "coarse/dense/dense_0/kernel", "coarse/dense/dense_0/bias", n->c4, 12288, n->g_d0, 4096, st));
  else
    CK(adam_range(n, G_DENSE, n->group_lo[G_DENSE], n->group_hi[G_DENSE], st));
  // conv stack, top down
  CK(a3d_conv2d_wgrad(c, &n->d_c4, n->c3, n->g_c4, G("coarse/conv/conv2d_4/kernel"), G("coarse/conv/conv2d_4/bias"), n->scratch,
                      n->scratch_bytes, st));
  CK(a3d_conv2d_dgrad(c, &n->d_c4, n->g_c4, W("coarse/conv/conv2d_4/kernel"), n->g_c3, n->c3, n->scratch, n->scratch_bytes, st));
  CK(a3d_conv2d_wgrad(c, &n->d_c3, n->c2, n->g_c3, G("coarse/conv/conv2d_3/kernel"), G("coarse/conv/conv2d_3/bias"), n->scratch,
                      n->scratch_bytes, st));
  CK(a3d_conv2d_dgrad(c, &n->d_c3, n->g_c3, W("coarse/conv/conv2d_3/kernel"), n->g_c2, n->c2, n->scratch, n->scratch_bytes, st));
  CK(a3d_conv2d_wgrad(c, &n->d_c2, n->p1, n->g_c2, G("coarse/conv/conv2d_2/kernel"), G("coarse/conv/conv2d_2/bias"), n->scratch,
                      n->scratch_bytes, st));
  CK(a3d_conv2d_dgrad(c, &n->d_c2, n->g_c2, W("coarse/conv/conv2d_2/kernel"), n->g_p1, nullptr, n->scratch, n->scratch_bytes, st));
  CK(a3d_maxpool2x2_idx_bwd(c, n->i1, n->g_p1, 256, B, 27, 37, 256, n->g_c1, st));
  CK(a3d_conv2d_wgrad(c, &n->d_c1, n->p0, n->g_c1, G("coarse/conv/conv2d_1/kernel"), G("coarse/conv/conv2d_1/bias"), n->scratch,
                      n->scratch_bytes, st));
  CK(a3d_conv2d_dgrad(c, &n->d_c1, n->g_c1, W("coarse/conv/conv2d_1/kernel"), n->g_p0, nullptr, n->scratch, n->scratch_bytes, st));
  CK(a3d_maxpool2x2_idx_bwd(c, n->i0, n->g_p0, 128, B, 55, 74, 96, n->g_c0, st));
  CK(a3d_conv2d_wgrad(c, &n->d_c0, n->img4, n->g_c0, G("coarse/conv/conv2d_0/kernel"), G("coarse/conv/conv2d_0/bias"), n->scratch,
                      n->scratch_bytes, st));
  CK(a3d_apply_mask_f32(c, G("coarse/conv/conv2d_0/kernel"), n->mask_c0, (size_t)96 * 576, st));   // padding entries of the s2d(4) packing
  return adam_range(n, G_CONV, n->group_lo[G_CONV], n->group_hi[G_CONV], st);
}

int backward_fine(a3d_msdn* n, void* st) {
  a3d_ctx* c = n->ctx;
  const int B = n->B;
  auto W = [&](const char* nm) { return n->wb + seg_off(n, nm); };
  auto G = [&](const char* nm) { return n->g + seg_off(n, nm); };
  CK(a3d_conv2d_wgrad(c, &n->d_f3, n->f2, n->g_fine, G("fine/third/kernel"), G("fine/third/bias"), n->scratch, n->scratch_bytes, st));
  CK(a3d_conv2d_dgrad(c, &n->d_f3, n->g_fine, W("fine/third/kernel"), n->g_f2, n->f2, n->scratch, n->scratch_bytes, st));
  CK(a3d_conv2d_wgrad(c, &n->d_f2, n->cat, n->g_f2, G("fine/second/conv2d/kernel"), G("fine/second/conv2d/bias"), n->scratch,
                      n->scratch_bytes, st));
  CK(a3d_conv2d_dgrad(c, &n->d_f2, n->g_f2, W("fine/second/conv2d/kernel"), n->g_cat, nullptr, n->scratch, n->scratch_bytes, st));
  // fine/first: MaxPoolGrad + ReluGrad on the 4 x 64 GEMM columns, wgrad of the embedded filter, fold its four copies
  CK(a3d_pool4_bwd(c, n->g_cat, 64, n->cat, 64, n->if1, n->g_f1big, (size_t)B * N_PIX, st));
  const size_t nk = (size_t)256 * 576;
  CK(a3d_conv2d_wgrad(c, &n->d_f1w, n->img4, n->g_f1big, n->g_wbig, n->g_wbig + nk, n->scratch, n->scratch_bytes, st));
  CK(a3d_gather_sum_f32(c, n->g_wbig, n->emb_k, 4, 25600, G("fine/first/conv2d/kernel"), st));
  CK(a3d_gather_sum_f32(c, n->g_wbig + nk, n->emb_b, 4, 64, G("fine/first/conv2d/bias"), st));
  CK(adam_range(n, G_FINEA, n->group_lo[G_FINEA], n->group_hi[G_FINEA], st));
  CK(adam_range(n, G_FINEB, n->group_lo[G_FINEB], n->group_hi[G_FINEB], st));
  return refresh_derived(n, st);
}
}  // namespace

extern "C" size_t a3d_msdn_workspace_bytes(a3d_ctx* ctx, int batch, int in_h, int in_w, int depth_h, int depth_w, int train) {
  if (!ctx || batch <= 0) return 0;
  a3d_msdn n;
  init_layout(&n, ctx, batch, in_h, in_w, depth_h, depth_w, train);
  return carve(&n, nullptr) + 256;
}

extern "C" int a3d_msdn_create(a3d_ctx* ctx, int batch, int in_h, int in_w, int depth_h, int depth_w, int train, void* workspace,
                               size_t workspace_bytes, void* stream, a3d_msdn** out) {
  A3D_REQUIRE(ctx && workspace && out && batch > 0 && batch <= 256 && in_h > 0 && in_w > 0 && depth_h > 0 && depth_w > 0,
              "msdn_create: bad argument (batch 1..256)");
  a3d_msdn* n = new a3d_msdn();
  init_layout(n, ctx, batch, in_h, in_w, depth_h, depth_w, train);
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 255) & ~uintptr_t(255));
  const size_t need = carve(n, base);
  if (base + need > reinterpret_cast<uint8_t*>(workspace) + workspace_bytes) {
    delete n;
    a3d_set_error("msdn_create: workspace of %zu bytes is too small (a3d_msdn_workspace_bytes)", workspace_bytes);
    return A3D_EINVAL;
  }
  cudaStream_t st = as_stream(stream);
  A3D_CHECK_CUDA(cudaMemsetAsync(base, 0, need, st));        // zero weights / slots / padding channels / routing records
  // index maps of the pool-embedded fine/first filter (params.py fine_first_index_maps) and conv2d_0's padding mask
  {
    int* ek = new int[4 * 25600];
    int* eb = new int[4 * 64];
    uint8_t* mk = new uint8_t[96 * 576];
    for (int i = 0; i < 4 * 25600; ++i) ek[i] = -1;
    for (int i = 0; i < 4 * 64; ++i) eb[i] = -1;
    // canonical element (co, r', s', q = (di*2+dj)*4 + c) <-> TF (i = 2r'+di, j = 2s'+dj, c, co) of the 9x9x3x63 filter
    for (int co = 0; co < 63; ++co)
      for (int r2 = 0; r2 < 5; ++r2)
        for (int s2 = 0; s2 < 5; ++s2)
          for (int q = 0; q < 16; ++q) {
            const int di = (q >> 2) >> 1, dj = (q >> 2) & 1, ch = q & 3;
            const int i = 2 * r2 + di, j = 2 * s2 + dj;
            if (i >= 9 || j >= 9 || ch >= 3) continue;
            const int e = ((co * 5 + r2) * 5 + s2) * 16 + q;
            for (int a = 0; a < 2; ++a)
              for (int b = 0; b < 2; ++b) {
                // copy g = 2a+b: the filter shifted by (2a, 2b) inside the 11x11 field, s2d(4)-packed [256][3][3][64]
                const int gq = 2 * a + b, y = 2 * a + i, x = 2 * b + j;
                const int K = gq * 64 + co, R = y >> 2, dy = y & 3, S = x >> 2, dx = x & 3;
                ek[gq * 25600 + e] = ((K * 3 + R) * 3 + S) * 64 + (dy * 4 + dx) * 3 + ch;
              }
          }
    for (int gq = 0; gq < 4; ++gq)
      for (int co = 0; co < 63; ++co) eb[gq * 64 + co] = gq * 64 + co;
    for (int co = 0; co < 96; ++co)
      for (int R = 0; R < 3; ++R)
        for (int S = 0; S < 3; ++S)
          for (int q = 0; q < 64; ++q) {
            bool ok = false;
            if (q < 48) {
              const int dy = q / 12, dx = (q % 12) / 3;
              ok = 4 * R + dy < 11 && 4 * S + dx < 11;
            }
            mk[((co * 3 + R) * 3 + S) * 64 + q] = ok ? 1 : 0;
          }
    cudaError_t e1 = cudaMemcpyAsync(n->emb_k, ek, sizeof(int) * 4 * 25600, cudaMemcpyHostToDevice, st);
    cudaError_t e2 = cudaMemcpyAsync(n->emb_b, eb, sizeof(int) * 4 * 64, cudaMemcpyHostToDevice, st);
    cudaError_t e3 = cudaMemcpyAsync(n->mask_c0, mk, 96 * 576, cudaMemcpyHostToDevice, st);
    cudaStreamSynchronize(st);                               // the pageable staging arrays die below (creation only)
    delete[] ek; delete[] eb; delete[] mk;
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess) {
      delete n;
      a3d_set_error("msdn_create: uploading the index maps failed");
      return A3D_EINVAL;
    }
  }
  *out = n;
  return 0;
}

extern "C" int a3d_msdn_destroy(a3d_msdn* n) {
  delete n;
  return 0;
}

// Hyper-parameters that are constructor arguments in the reference: beta2 of the four AdamOptimizers (src/models.py:309
// passes 1) and the dropout seed (unseeded there).
extern "C" int a3d_msdn_configure(a3d_msdn* n, float adam_beta2, uint64_t dropout_seed) {
  A3D_REQUIRE(n, "msdn_configure: null net");
  n->beta2 = adam_beta2;
  n->seed = dropout_seed;
  return 0;
}

// Segment table of the parameter arena: name -> element offset / element count / packed shape (ndim <= 4).
// Returns the number of segments when name == nullptr.
extern "C" int a3d_msdn_segment(const a3d_msdn* n, int index, const char** name, size_t* offset, size_t* numel, int shape[4]) {
  if (!n) return 0;
  if (index < 0 || index >= NSEG) return NSEG;
  const Seg& s = n->seg[index];
  if (name) *name = s.name;
  if (offset) *offset = s.offset;
  if (numel) *numel = s.numel;
  if (shape) for (int k = 0; k < 4; ++k) shape[k] = k < s.ndim ? s.shape[k] : 0;
  return NSEG;
}

// Device pointers of the arena (each `total` elements): f32 master weights, Adam slots m / v, f32 gradients, bf16 mirror.
// After writing weights into `w` call a3d_msdn_sync_weights (refreshes the mirror and the derived fine/first filter).
extern "C" int a3d_msdn_arena(a3d_msdn* n, float** w, float** m, float** v, float** g, uint16_t** w_bf16, size_t* total) {
  A3D_REQUIRE(n, "msdn_arena: null net");
  if (w) *w = n->w;
  if (m) *m = n->m;
  if (v) *v = n->v;
  if (g) *g = n->g;
  if (w_bf16) *w_bf16 = n->wb;
  if (total) *total = n->total;
  return 0;
}

extern "C" int a3d_msdn_sync_weights(a3d_msdn* n, void* stream) {
  A3D_REQUIRE(n, "msdn_sync_weights: null net");
  CK(a3d_cast_f32_bf16(n->ctx, n->w, n->wb, n->total, stream));
  return refresh_derived(n, stream);
}

// global_step and the per-optimizer step counts (checkpoint / resume: src/ann3depth.py:113-125)
extern "C" int a3d_msdn_set_step(a3d_msdn* n, long long global_step, const int adam_t[4], void* stream) {
  A3D_REQUIRE(n && global_step >= 0, "msdn_set_step: bad argument");
  n->global_step = global_step;
  if (adam_t) for (int g = 0; g < 4; ++g) n->adam_t[g] = adam_t[g];
  set_i64_kernel<<<1, 1, 0, as_stream(stream)>>>(n->step_dev, global_step);
  A3D_CHECK_CUDA(cudaGetLastError());
  return 0;
}
extern "C" long long a3d_msdn_global_step(const a3d_msdn* n) { return n ? n->global_step : -1; }

// Host half of a step (NOT capturable): advances global_step and the beta-power state of the active branch's Adam
// instances and writes their bias-corrected step sizes lr_t to device scalars the (captured) kernels read.
// Returns the phase (1 coarse, 2 fine, 3 idle) of the step about to run, < 0 on error.
extern "C" int a3d_msdn_step_begin(a3d_msdn* n, void* stream) {
  if (!n || !n->train) { a3d_set_error("msdn_step_begin: needs a net created with train = 1"); return A3D_EINVAL; }
  const int phase = phase_of(n->global_step, n->B);
  const int g0 = phase == 1 ? G_DENSE : G_FINEA;
  if (phase != 3)
    for (int g = g0; g < g0 + 2; ++g) {
      n->adam_t[g] += 1;
      set_f32_kernel<<<1, 1, 0, as_stream(stream)>>>(n->lr_dev + g, adam_lr_t(GROUP_LR[g], BETA1, n->beta2, n->adam_t[g]));
    }
  if (cudaGetLastError() != cudaSuccess) { a3d_set_error("msdn_step_begin: launch failed"); return A3D_EINVAL; }
  n->global_step += 1;
  return phase;
}

// Device half of a step for `phase` (the value a3d_msdn_step_begin returned): pure kernel launches on `stream`,
// capturable in a CUDA graph (one graph per phase; replay it after each a3d_msdn_step_begin).
// images f32 [B,in_h,in_w,3], depths f32 [B,depth_h,depth_w,1] (device); keep_mask u8 [B,4096] or null (device RNG).
extern "C" int a3d_msdn_step_enqueue(a3d_msdn* n, int phase, const float* images, const float* depths, const uint8_t* keep_mask,
                                     void* stream) {
  A3D_REQUIRE(n && n->train && images && depths && phase >= 1 && phase <= 3, "msdn_step_enqueue: bad argument");
  CK(forward(n, images, depths, keep_mask, stream));
  if (phase == 1) CK(backward_coarse(n, stream));
  if (phase == 2) CK(backward_fine(n, stream));
  return a3d_increment_i64(n->ctx, n->step_dev, stream);     // global_step += 1 (src/models.py:329,343,356)
}

// One `session.run(model_op)`: a3d_msdn_step_begin + a3d_msdn_step_enqueue.  Returns the phase that ran (>= 1) or an
// error (< 0).  losses (nullable, device, 2 floats) receives loss/coarse_loss and loss/fine_loss.
extern "C" int a3d_msdn_step(a3d_msdn* n, const float* images, const float* depths, const uint8_t* keep_mask, float* losses,
                             void* stream) {
  const int phase = a3d_msdn_step_begin(n, stream);
  if (phase < 0) return phase;
  int rc = a3d_msdn_step_enqueue(n, phase, images, depths, keep_mask, stream);
  if (rc) return rc < 0 ? rc : -rc;
  if (losses) A3D_CHECK_CUDA(cudaMemcpyAsync(losses, n->losses, 2 * sizeof(float), cudaMemcpyDeviceToDevice, as_stream(stream)));
  return phase;
}

// Inference (train = False: dropout off, src/models.py:230,278,286): fine / coarse depth maps f32 [B,55,74] (device,
// nullable).  Works on a net created with train = 0 or 1.  Capturable.
extern "C" int a3d_msdn_infer(a3d_msdn* n, const float* images, float* fine, float* coarse, void* stream) {
  A3D_REQUIRE(n && images, "msdn_infer: bad argument");
  const int was = n->train;
  n->train = 0;
  const int rc = forward(n, images, nullptr, nullptr, stream);
  n->train = was;
  if (rc) return rc;
  const size_t bytes = (size_t)n->B * N_PIX * sizeof(float);
  if (fine) A3D_CHECK_CUDA(cudaMemcpyAsync(fine, n->fine, bytes, cudaMemcpyDeviceToDevice, as_stream(stream)));
  if (coarse) A3D_CHECK_CUDA(cudaMemcpyAsync(coarse, n->coarse, bytes, cudaMemcpyDeviceToDevice, as_stream(stream)));
  return 0;
}

// Losses of the last step / forward: device pointer to {coarse, fine}
extern "C" const float* a3d_msdn_losses(const a3d_msdn* n) { return n ? n->losses : nullptr; }

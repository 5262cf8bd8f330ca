// C ABI of libtld_b200.so (include/tld_b200.h): handle, weight packing, Denoiser.forward, CFG sampler.
#include <math.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/tld_b200.h"
#include <map>
#include <mutex>
#include <utility>

#include "common.h"
#include "gemm_tcgen05.cuh"  // EpiMode
#include "launch.h"

namespace tld {

static thread_local std::string g_err;
int fail(const std::string& msg) {
  g_err = msg;
  return 1;
}
const char* last_error() { return g_err.c_str(); }

bool ln_fold_requested();   // tld_set_option("ln_fold", 1) is in effect (defined with the option below)
static int g_pdl = 0;  // measured on B200: no gain (the step is power-capped, not launch-gap bound); kept as an option
void set_pdl(int v) { g_pdl = v; }
// Bumped by every tld_set_option call: a captured sampler graph bakes in the kernel selection (attention implementation,
// GEMM tile mode, PDL attribute), so a graph recorded under an older epoch is re-captured.
static int g_option_epoch = 0;
bool pdl_enabled() { return g_pdl != 0; }

float* device_scratch(ScratchSlot slot, size_t n_floats) {
  struct Buf { float* p = nullptr; size_t cap = 0; };
  static std::mutex mu;
  static std::map<std::pair<int, int>, Buf> bufs;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) { fail("device_scratch: cudaGetDevice failed"); return nullptr; }
  std::lock_guard<std::mutex> lock(mu);
  Buf& b = bufs[{dev, (int)slot}];
  if (n_floats > b.cap) {
    if (b.p) cudaFree(b.p);   // synchronises with any kernel still reading the old buffer
    b.p = nullptr;
    b.cap = 0;
    const size_t want = n_floats + n_floats / 4;   // some head room: batch sizes creep up during warm-up
    if (cudaMalloc(&b.p, want * sizeof(float)) != cudaSuccess) { fail("device_scratch: cudaMalloc failed"); return nullptr; }
    b.cap = want;
  }
  return b.p;
}

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

// ------------------------------------------------------------------------------------------ packing
__global__ void f32_to_bf16_kernel(const float* __restrict__ s, bf16* __restrict__ d, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] = __float2bfloat16(s[i]);
}
__global__ void transpose_f32_kernel(const float* __restrict__ s, float* __restrict__ d, int rows, int cols) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // d[c][r] = s[r][c]
  if (i < (long long)rows * cols) {
    const int r = int(i / cols), c = int(i % cols);
    d[(size_t)c * rows + r] = s[i];
  }
}

// all parameter slots of one refresh in a few launches: blockIdx.y = entry, blockIdx.x strides over its elements
struct RefreshEntry {
  const float* src;
  void* dst;
  long long numel;
  int kind, rows, cols, pad;   // kind: 0 copy fp32, 1 fp32 -> bf16, 2 fp32 [rows, cols] -> fp32 [cols, rows]
};
constexpr int REFRESH_BATCH = 96;   // 96 x 40 B = 3840 B of kernel arguments
struct RefreshBatch {
  RefreshEntry e[REFRESH_BATCH];
};
__global__ void __launch_bounds__(256) refresh_params_kernel(const __grid_constant__ RefreshBatch batch) {
  const RefreshEntry& e = batch.e[blockIdx.y];
  const long long stride = (long long)gridDim.x * 256;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < e.numel; i += stride) {
    const float v = e.src[i];
    if (e.kind == 0) {
      reinterpret_cast<float*>(e.dst)[i] = v;
    } else if (e.kind == 1) {
      reinterpret_cast<bf16*>(e.dst)[i] = __float2bfloat16(v);
    } else {
      const int r = int(i / e.cols), c = int(i % e.cols);
      reinterpret_cast<float*>(e.dst)[(size_t)c * e.rows + r] = v;
    }
  }
}

}  // namespace tld

#include "handle.h"
using namespace tld;

namespace tld {

template <typename T>
static int dev_alloc(tld_denoiser* h, T** p, long long n, bool track = true) {
  void* q = nullptr;
  TLD_CUDA_OK(cudaMalloc(&q, (size_t)(n > 0 ? n : 1) * sizeof(T)));
  *p = reinterpret_cast<T*>(q);
  if (track) h->allocs.push_back(q);
  return 0;
}

static int add_slot(tld_denoiser* h, const std::string& key, PackKind kind, void* dst, long long numel, int rows = 0,
                    int cols = 0) {
  Slot s{};
  s.kind = kind; s.dst = dst; s.numel = numel; s.rows = rows; s.cols = cols; s.filled = false;
  h->slots[key] = s;
  return 0;
}

template <typename T>
static int alloc_slot(tld_denoiser* h, const std::string& key, PackKind kind, T** dst, long long numel, int rows = 0,
                      int cols = 0) {
  if (dev_alloc(h, dst, numel)) return 1;
  return add_slot(h, key, kind, *dst, numel, rows, cols);
}

static int build_params(tld_denoiser* h) {
  const int D = h->D, L = h->L, N = h->N, pd = h->pd, H4 = h->H4, E = h->E, Te = h->Te;
  const std::string tb = "denoiser_trans_block.";
  float* f = nullptr;
#define F32(key, field, n)                                   \
  if (alloc_slot(h, key, P_F32, &f, (n))) return 1;          \
  field = f;
  F32("fourier_feats.0.angular_speeds", h->cond.speeds, E / 2)
  F32("fourier_feats.1.weight", h->cond.w1, (long long)D * E)
  F32("fourier_feats.1.bias", h->cond.b1, D)
  F32("fourier_feats.3.weight", h->cond.w2, (long long)D * D)
  F32("fourier_feats.3.bias", h->cond.b2, D)
  F32("label_proj.weight", h->cond.wl, (long long)D * Te)
  F32("label_proj.bias", h->cond.bl, D)
  F32("norm.weight", h->cond.ln_w, D)
  F32("norm.bias", h->cond.ln_b, D)
  F32(tb + "patchify_and_embed.0.weight", h->emb.conv_w, (long long)pd * pd)
  F32(tb + "patchify_and_embed.0.bias", h->emb.conv_b, pd)
  F32(tb + "patchify_and_embed.2.weight", h->emb.ln1_w, pd)
  F32(tb + "patchify_and_embed.2.bias", h->emb.ln1_b, pd)
  F32(tb + "patchify_and_embed.3.bias", h->emb.lin_b, D)
  F32(tb + "patchify_and_embed.4.weight", h->emb.ln2_w, D)
  F32(tb + "patchify_and_embed.4.bias", h->emb.ln2_b, D)
  F32(tb + "pos_embed.weight", h->emb.pos, (long long)N * D)
  F32(tb + "out_proj.0.weight", h->out_w, (long long)pd * D)
  F32(tb + "out_proj.0.bias", h->out_b, pd)
  {
    float* t = nullptr;
    if (alloc_slot(h, tb + "patchify_and_embed.3.weight", P_TRANSPOSE_F32, &t, (long long)D * pd, D, pd)) return 1;
    h->emb.lin_wT = t;
  }
  if (dev_alloc(h, &h->wkv_all, (long long)L * 2 * D * D)) return 1;
  h->layers.resize(L);
  h->fold.resize(L);
  for (int l = 0; l < L; ++l) {
    auto& ly = h->layers[l];
    const std::string b = tb + "decoder_blocks." + std::to_string(l) + ".";
    if (alloc_slot(h, b + "self_attention.qkv_linear.weight", P_BF16, &ly.wqkv, 3LL * D * D)) return 1;
    {
      auto& fl = h->fold[l];
      if (dev_alloc(h, &fl.wqkv32, 3LL * D * D) || dev_alloc(h, &fl.wup32, (long long)H4 * D) || dev_alloc(h, &fl.wqkv_f, 3LL * D * D) ||
          dev_alloc(h, &fl.wup_f, (long long)H4 * D) || dev_alloc(h, &fl.s_qkv, 3LL * D) || dev_alloc(h, &fl.c_qkv, 3LL * D) ||
          dev_alloc(h, &fl.s_up, H4) || dev_alloc(h, &fl.c_up, H4))
        return 1;
      h->slots[b + "self_attention.qkv_linear.weight"].shadow = fl.wqkv32;
    }
    if (alloc_slot(h, b + "cross_attention.q_linear.weight", P_BF16, &ly.wq, (long long)D * D)) return 1;
    add_slot(h, b + "cross_attention.kv_linear.weight", P_BF16, h->wkv_all + (size_t)l * 2 * D * D, 2LL * D * D);
    if (alloc_slot(h, b + "mlp.mlp.0.weight", P_BF16, &ly.wup, (long long)H4 * D)) return 1;
    h->slots[b + "mlp.mlp.0.weight"].shadow = h->fold[l].wup32;
    if (alloc_slot(h, b + "mlp.mlp.3.weight", P_BF16, &ly.wdown, (long long)D * H4)) return 1;
    F32(b + "mlp.mlp.0.bias", ly.bup, H4)
    F32(b + "mlp.mlp.1.bias", ly.dwb, H4)
    F32(b + "mlp.mlp.3.bias", ly.bdown, D)
    F32(b + "norm1.weight", ly.ln1w, D)
    F32(b + "norm1.bias", ly.ln1b, D)
    F32(b + "norm2.weight", ly.ln2w, D)
    F32(b + "norm2.bias", ly.ln2b, D)
    F32(b + "norm3.weight", ly.ln3w, D)
    F32(b + "norm3.bias", ly.ln3b, D)
    float* t = nullptr;  // depthwise weight [4D,1,3,3] -> tap-major [9, 4D]
    if (alloc_slot(h, b + "mlp.mlp.1.weight", P_TRANSPOSE_F32, &t, 9LL * H4, H4, 9)) return 1;
    ly.dww9 = t;
  }
#undef F32
  h->staging_elems = 0;
  for (auto& kv : h->slots) h->staging_elems = kv.second.numel > h->staging_elems ? kv.second.numel : h->staging_elems;
  return dev_alloc(h, &h->staging, h->staging_elems);
}

// Both captured sampler step graphs bake in the workspace, conditioning and sampler buffer addresses: every reallocation
// of any of them drops both.
static void drop_step_graphs(tld_denoiser* h) {
  if (h->graph_exec) { cudaGraphExecDestroy(h->graph_exec); h->graph_exec = nullptr; h->graph_batch = -1; }
  if (h->graph_exec_masked) { cudaGraphExecDestroy(h->graph_exec_masked); h->graph_exec_masked = nullptr; h->graph_batch_masked = -1; }
}

static void free_workspace(tld_denoiser* h) {
  void* ptrs[] = {h->x_res, h->xn, h->qkv, h->hid, h->hid2, h->model_out, h->xb[0], h->xb[1], h->part[0], h->part[1]};
  for (void* p : ptrs)
    if (p) cudaFree(p);
  h->x_res = nullptr; h->xn = nullptr; h->qkv = nullptr; h->hid = nullptr; h->hid2 = nullptr; h->model_out = nullptr;
  h->xb[0] = h->xb[1] = nullptr; h->part[0] = h->part[1] = nullptr;
  h->ws_batch = 0;
  drop_step_graphs(h);
}

static int ensure_workspace(tld_denoiser* h, int batch) {
  if (batch <= h->ws_batch) return 0;
  TLD_CUDA_OK(cudaDeviceSynchronize());
  free_workspace(h);
  const long long T = (long long)batch * h->N;
  if (dev_alloc(h, &h->x_res, T * h->D, false)) return 1;
  if (dev_alloc(h, &h->xn, T * h->D, false)) return 1;
  if (dev_alloc(h, &h->qkv, T * 3 * h->D, false)) return 1;
  if (dev_alloc(h, &h->hid, T * h->H4, false)) return 1;
  if (dev_alloc(h, &h->hid2, T * h->H4, false)) return 1;
  if (dev_alloc(h, &h->model_out, (long long)batch * h->C * h->img * h->img, false)) return 1;
  for (int i = 0; i < 2; ++i) {
    if (dev_alloc(h, &h->xb[i], T * h->D, false)) return 1;
    if (dev_alloc(h, &h->part[i], T * (h->D / 32), false)) return 1;
  }
  h->ws_batch = batch;
  return 0;
}

static int ensure_cond(tld_denoiser* h, int rows) {
  if (rows <= h->ws_cond_rows) return 0;
  TLD_CUDA_OK(cudaDeviceSynchronize());
  if (h->ycond) cudaFree(h->ycond);
  if (h->kv) cudaFree(h->kv);
  if (h->uk) cudaFree(h->uk);
  h->uk = nullptr;
  if (h->tlevels) cudaFree(h->tlevels);
  if (h->cond_scratch) cudaFree(h->cond_scratch);
  h->ycond = nullptr; h->kv = nullptr; h->tlevels = nullptr; h->cond_scratch = nullptr;
  drop_step_graphs(h);
  const int r = ((rows + 127) / 128) * 128;
  if (dev_alloc(h, &h->ycond, (long long)r * h->D, false)) return 1;
  if (dev_alloc(h, &h->kv, (long long)r * h->L * 2 * h->D, false)) return 1;
  // folded cross-attention keys: (D / 64) D floats per row and layer; past 1 GiB the q-GEMM path is used instead
  const long long uk_elems = (long long)r * h->L * (h->D / 64) * h->D;
  if (uk_elems * 4 <= (1ll << 30) && dev_alloc(h, &h->uk, uk_elems, false)) return 1;
  if (dev_alloc(h, &h->tlevels, r, false)) return 1;
  if (dev_alloc(h, &h->cond_scratch, (long long)r * (h->E + 2 * h->D), false)) return 1;
  h->ws_cond_rows = r;
  return 0;
}

}  // namespace tld
int tld_internal_ensure(tld_denoiser* h, int batch, int cond_rows) {
  return tld::ensure_workspace(h, batch) || tld::ensure_cond(h, cond_rows);
}
namespace tld {

static int g_attention_impl = 0;  // tld_set_option("attention_impl", ...)
static int g_fused_mlp = 1;       // tld_set_option("fused_mlp", ...): up-projection + depthwise conv + GELU in one kernel
// tld_set_option("ln_fold", ...): norm1 / norm3 folded into the neighbouring GEMMs.  OFF by default: measured on B200 the
// explicit read-modify-write epilogues cost more than the two LayerNorm kernels they remove (per layer: mlp.3 105.7 -> 129 us,
// cross-attention 42.5 -> 66 us, qkv 81 -> 90 us against 2 x 23.7 us saved; 256-px step 7.31 -> 7.49 ms).  The TMA reduce-add
// residual is a read-modify-write AT L2 with deep queues; doing it in the SM needs x_old in shared memory several chunks
// ahead, and the 6-stage operand pipeline leaves no room for that.  Kept selectable and parity-tested.
static int g_ln_fold = 0;

bool ln_fold_requested() { return g_ln_fold != 0; }
static bool use_ln_fold(const tld_denoiser* h) { return g_ln_fold && h->D % 128 == 0; }

// W' = bf16(gamma (.) W), s, c of every layer from the fp32 shadows, once after each parameter refresh
static int ensure_fold(tld_denoiser* h, cudaStream_t st) {
  if (!h->fold_dirty) return 0;
  const int D = h->D, H4 = h->H4;
  for (int l = 0; l < h->L; ++l) {
    const auto& ly = h->layers[l];
    const auto& fl = h->fold[l];
    if (launch_ln_fold_weights(fl.wqkv32, ly.ln1w, ly.ln1b, nullptr, fl.wqkv_f, fl.s_qkv, fl.c_qkv, 3 * D, D, st)) return 1;
    if (launch_ln_fold_weights(fl.wup32, ly.ln3w, ly.ln3b, ly.bup, fl.wup_f, fl.s_up, fl.c_up, H4, D, st)) return 1;
  }
  h->fold_dirty = false;
  return 0;
}

// the fused MLP front half needs one CTA-pair tile per sample (16x16 token grid) and whole 256-channel tiles
static bool use_fused_mlp(const tld_denoiser* h) { return g_fused_mlp && h->G == 16 && h->H4 % 256 == 0; }
static int g_share_cfg_prefix = 1;   // tld_set_option("share_cfg_prefix", ...): block 0's self-attention once per CFG pair (sampler)
static int g_fused_xattn = 1;     // tld_set_option("fused_xattn", ...): norm2 + cross-attention + residual + norm3 in one row-wise kernel
static bool use_fused_xattn(const tld_denoiser* h) {
  return g_fused_xattn && h->uk && ln_xattn_ln_supported(h->D, h->N) && !use_ln_fold(h);
}
// u = Wq_h^T k_h for every row of the K/V table and every layer (once per forward, once per generation in the sampler)
static int fold_xattn_keys(tld_denoiser* h, int rows, cudaStream_t st) {
  if (!use_fused_xattn(h)) return 0;
  const long long kvs = (long long)h->L * 2 * h->D, uks = (long long)h->L * (h->D / 64) * h->D;
  for (int l = 0; l < h->L; ++l)
    if (launch_xattn_fold_keys(h->kv + (size_t)l * 2 * h->D, kvs, rows, h->layers[l].wq, h->uk + (size_t)l * (h->D / 64) * h->D, uks,
                               h->D, st))
      return 1;
  return 0;
}
static int g_fused_qkv = 1;       // tld_set_option("fused_qkv", ...): qkv projection + attention in one kernel (256 tokens)
static bool use_fused_qkv(const tld_denoiser* h) { return g_fused_qkv && h->N == 256 && !use_ln_fold(h); }

// The L decoder blocks + output projection on the tokens already in h->x_res (transformer_blocks.py:135-139).
// `distinct`: the residual rows of samples [distinct, batch) are copies of samples [0, distinct) on entry (the CFG pair embeds
// the same x_t twice and differs only in the label token, i.e. from the first cross-attention on): block 0's norm1 +
// self-attention then run on the distinct samples only and the result is copied.
static int run_blocks(tld_denoiser* h, int batch, const float* kv0, long long kv0_stride, const float* kv1,
                      long long kv1_stride, const int* step_ptr, float* out, cudaStream_t st, int distinct = 0) {
  const int D = h->D, H4 = h->H4, N = h->N;
  const int T = batch * N;
  const bool share0 = g_share_cfg_prefix && distinct > 0 && distinct < batch && batch % distinct == 0 && !use_ln_fold(h);
  const bool fold = use_ln_fold(h);
  const int n_part = D / 32;
  int cur = 0;   // which xb / part buffer holds the current residual rows
  if (fold && launch_rowstats_cast(h->x_res, h->xb[0], h->part[0], T, D, st)) return 1;   // the embedding's rows
  for (int l = 0; l < h->L; ++l) {
    const auto& ly = h->layers[l];
    const auto& fl = h->fold[l];
    // x = SelfAttention(LN1(x)) + x
    if (fold) {   // norm1 folded: A = bf16(x), W = gamma (.) Wqkv, mean / rstd applied on the accumulator
      LnFoldArgs ln{fl.s_qkv, h->part[cur], n_part, 1e-5f, nullptr, 0, nullptr};
      if (launch_gemm(EPI_LNFOLD_BF16, h->xb[cur], D, fl.wqkv_f, D, T, 3 * D, D, h->qkv, 3 * D, fl.c_qkv, nullptr, st, &ln)) return 1;
    }
    const int ab = (l == 0 && share0) ? distinct : batch;   // samples the self-attention of this block runs on
    const int Ta = ab * N;
    if (!fold) {
      if (launch_layernorm_bf16(h->x_res, ly.ln1w, ly.ln1b, h->xn, Ta, D, st)) return 1;
      if (!use_fused_qkv(h) && launch_gemm(EPI_BF16, h->xn, D, ly.wqkv, D, Ta, 3 * D, D, h->qkv, 3 * D, nullptr, nullptr, st)) return 1;
    }
    if (use_fused_qkv(h)) {   // the CTA pair that owns a (sample, head) projects q, k, v itself: qkv never touches HBM
      if (launch_qkv_attention(h->xn, ly.wqkv, h->x_res, ab, N, D, st)) return 1;
    } else if (launch_self_attention(h->qkv, h->x_res, ab, N, D, st, g_attention_impl)) return 1;
    if (ab != batch)
      for (int c = 1; c < batch / distinct; ++c)
        TLD_CUDA_OK(cudaMemcpyAsync(h->x_res + (size_t)c * Ta * D, h->x_res, sizeof(float) * (size_t)Ta * D, cudaMemcpyDeviceToDevice, st));
    // x = CrossAttention(LN2(x), y) + x
    if (use_fused_xattn(h)) {   // norm2, the (folded) q projection, the 2-key softmax, the residual and norm3 in one row-wise pass
      const long long kvs_all = (long long)h->L * 2 * D, uks = (long long)h->L * (D / 64) * D;
      const float* uk0 = h->uk + ((kv0 - h->kv) / kvs_all) * uks + (size_t)l * (D / 64) * D;
      const float* uk1 = h->uk + ((kv1 - h->kv) / kvs_all) * uks + (size_t)l * (D / 64) * D;
      if (launch_ln_xattn_ln(h->x_res, ly.ln2w, ly.ln2b, ly.ln3w, ly.ln3b, uk0, kv0_stride == 0 ? 0 : uks, uk1,
                             kv1_stride == 0 ? 0 : uks, kv0 + (size_t)l * 2 * D, kv0_stride, kv1 + (size_t)l * 2 * D, kv1_stride,
                             step_ptr, h->xn, T, N, D, st))
        return 1;
    } else {
    if (launch_layernorm_bf16(h->x_res, ly.ln2w, ly.ln2b, h->xn, T, D, st)) return 1;
    XattnArgs xa;
    xa.kv0 = kv0 + (size_t)l * 2 * D;
    xa.kv1 = kv1 + (size_t)l * 2 * D;
    xa.kv0_stride = kv0_stride;
    xa.kv1_stride = kv1_stride;
    xa.step_ptr = step_ptr;
    xa.n_tok = N;
    xa.embed_dim = D;
    if (fold) {   // producer of norm3's inputs: new rows also as bf16 + their statistics partials
      LnFoldArgs ln{nullptr, nullptr, 0, 1e-5f, h->xb[cur ^ 1], D, h->part[cur ^ 1]};
      if (launch_gemm(EPI_XATTN_RESID_LNP, h->xn, D, ly.wq, D, T, D, D, h->x_res, D, nullptr, &xa, st, &ln)) return 1;
      cur ^= 1;
    } else {
      if (launch_gemm(EPI_XATTN_RESID_F32, h->xn, D, ly.wq, D, T, D, D, h->x_res, D, nullptr, &xa, st)) return 1;
    }
    }
    // x = MLPSepConv(LN3(x)) + x
    const bf16* a_up = h->xn;
    if (fold) a_up = h->xb[cur];
    else if (!use_fused_xattn(h) && launch_layernorm_bf16(h->x_res, ly.ln3w, ly.ln3b, h->xn, T, D, st)) return 1;
    if (use_fused_mlp(h)) {
      if (launch_gemm_up_dwconv_gelu(a_up, D, fold ? fl.wup_f : ly.wup, D, T, H4, D, fold ? fl.c_up : ly.bup, fold ? fl.s_up : nullptr,
                                     fold ? h->part[cur] : nullptr, fold ? n_part : 0, 1e-5f, ly.dww9, ly.dwb, h->hid2, st))
        return 1;
    } else {
      if (fold) {
        LnFoldArgs ln{fl.s_up, h->part[cur], n_part, 1e-5f, nullptr, 0, nullptr};
        if (launch_gemm(EPI_LNFOLD_BF16, a_up, D, fl.wup_f, D, T, H4, D, h->hid, H4, fl.c_up, nullptr, st, &ln)) return 1;
      } else {
        if (launch_gemm(EPI_BIAS_BF16, a_up, D, ly.wup, D, T, H4, D, h->hid, H4, ly.bup, nullptr, st)) return 1;
      }
      if (launch_dwconv_gelu(h->hid, ly.dww9, ly.dwb, h->hid2, batch, h->G, H4, st)) return 1;
    }
    if (fold && l + 1 < h->L) {   // producer of the next block's norm1 inputs (the last block feeds the fp32 out-projection)
      LnFoldArgs ln{nullptr, nullptr, 0, 1e-5f, h->xb[cur ^ 1], D, h->part[cur ^ 1]};
      if (launch_gemm(EPI_BIAS_RESID_LNP, h->hid2, H4, ly.wdown, H4, T, D, H4, h->x_res, D, ly.bdown, nullptr, st, &ln)) return 1;
      cur ^= 1;
    } else {
      if (launch_gemm(EPI_BIAS_RESID_F32, h->hid2, H4, ly.wdown, H4, T, D, H4, h->x_res, D, ly.bdown, nullptr, st)) return 1;
    }
  }
  return launch_outproj(h->x_res, h->out_w, h->out_b, out, batch, h->C, h->img, h->patch, D, st);
}

static int kernels_per_forward(const tld_denoiser* h) {
  const int per_layer = 9 - (use_fused_mlp(h) ? 1 : 0) - (use_ln_fold(h) ? 2 : 0) - (use_fused_qkv(h) ? 1 : 0) -
                        (use_fused_xattn(h) ? 2 : 0);
  return 1 + (use_ln_fold(h) ? 1 : 0) + per_layer * h->L + 1;
}

}  // namespace tld

// =========================================================================================== C ABI
extern "C" {

const char* tld_last_error(void) { return tld::last_error(); }
int tld_version(void) { return 1; }

int tld_set_option(const char* key, int value) {
  TLD_CHECK(key != nullptr, "tld_set_option: null key");
  const std::string k(key);
  ++g_option_epoch;
  if (k == "gemm_ctas") {
    TLD_CHECK(value >= 0 && value <= 2, "gemm_ctas must be 0, 1 or 2");
    set_gemm_ctas(value);
    return 0;
  }
  if (k == "pdl") {
    set_pdl(value != 0);
    return 0;
  }
  if (k == "attention_impl") {
    TLD_CHECK(value == 0 || value == 1 || value == 3, "attention_impl must be 0 (auto), 1 (mma.sync) or 3 (tcgen05 persistent)");
    g_attention_impl = value;
    return 0;
  }
  if (k == "attention_bwd_impl") {
    TLD_CHECK(value >= 0 && value <= 2, "attention_bwd_impl must be 0 / 1 (mma.sync kernels, default) or 2 (tcgen05 kernel when tokens % 256 == 0)");
    set_attention_bwd_impl(value);
    return 0;
  }
  if (k == "qkv_exp_emu") {
    TLD_CHECK(value == 0 || value == 4 || value == 6 || value == 8, "qkv_exp_emu (exp2 pairs per 16 on the FMA pipe, fused qkv + attention kernel) must be 0, 4, 6 or 8");
    set_qkv_attention_exp_emu(value);
    return 0;
  }
  if (k == "share_cfg_prefix") {
    g_share_cfg_prefix = value != 0;
    return 0;
  }
  if (k == "fused_xattn") {
    g_fused_xattn = value != 0;
    return 0;
  }
  if (k == "xattn_rows") {
    TLD_CHECK(value == 2 || value == 4, "xattn_rows (rows per warp of the norm2 + cross-attention + norm3 row kernel) must be 2 or 4");
    set_xattn_rows(value);
    return 0;
  }
  if (k == "xattn_ctas") {
    TLD_CHECK(value == 1 || value == 2, "xattn_ctas (CTAs per SM of the norm2 + cross-attention + norm3 row kernel) must be 1 or 2");
    set_xattn_ctas(value);
    return 0;
  }
  if (k == "xattn_mma") {
    TLD_CHECK(value >= 0 && value <= 3, "xattn_mma must be 0 (FFMA row kernel, default), 1 (tf32 mma.sync dots, x rounded), 2 (x split) or 3 (x and folded keys split)");
    set_xattn_mma(value);
    return 0;
  }
  if (k == "fused_qkv") {
    g_fused_qkv = value != 0;
    return 0;
  }
  if (k == "fused_mlp") {
    g_fused_mlp = value != 0;
    return 0;
  }
  if (k == "ln_fold") {
    g_ln_fold = value != 0;
    return 0;
  }
  if (k == "attention_exp_emu") {
    TLD_CHECK(value == 0 || value == 4 || value == 6 || value == 8 || value == 10,
              "attention_exp_emu (exp2 pairs per 16 evaluated on the FMA pipe) must be 0, 4, 6, 8 or 10");
    set_attention_exp_emu(value);
    return 0;
  }
  return fail("tld_set_option: unknown key " + k);
}

int tld_denoiser_create(const tld_config* cfg, int device, tld_denoiser** out) {
  TLD_CHECK(cfg && out, "tld_denoiser_create: null argument");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
    return fail("tld_denoiser_create: no CUDA device (this library has no CPU fallback)");
  TLD_CHECK(device >= 0 && device < ndev, "tld_denoiser_create: bad device index");
  TLD_CUDA_OK(cudaSetDevice(device));
  cudaDeviceProp prop;
  TLD_CUDA_OK(cudaGetDeviceProperties(&prop, device));
  TLD_CHECK(prop.major == 10, "tld_denoiser_create: kernels are built for sm_100a (B200) only, found sm_" +
                                  std::to_string(prop.major) + std::to_string(prop.minor));
  TLD_CHECK(cfg->embed_dim % 64 == 0 && cfg->embed_dim >= 64 && cfg->embed_dim <= 1024,
            "embed_dim must be a multiple of 64 in [64,1024] (heads = embed_dim / 64, transformer_blocks.py:126-129)");
  TLD_CHECK(cfg->patch_size > 0 && cfg->image_size % cfg->patch_size == 0, "image_size must be divisible by patch_size");
  const int G = cfg->image_size / cfg->patch_size;
  TLD_CHECK((G * G) % 64 == 0, "tokens per sample ((image_size/patch_size)^2) must be a multiple of 64");
  TLD_CHECK(cfg->n_channels * cfg->patch_size * cfg->patch_size <= 64, "n_channels*patch_size^2 must be <= 64");
  TLD_CHECK(cfg->noise_embed_dims % 2 == 0 && cfg->noise_embed_dims > 0, "noise_embed_dims must be even");
  TLD_CHECK(cfg->n_layers > 0 && cfg->mlp_multiplier > 0 && cfg->text_emb_size > 0, "bad layer configuration");
  TLD_CHECK((cfg->mlp_multiplier * cfg->embed_dim) % 64 == 0, "mlp width must be a multiple of 64");
  TLD_CHECK(cfg->dropout == 0.f, "dropout must be 0 on the inference path");
  tld_denoiser* h = new tld_denoiser();
  h->cfg = *cfg;
  h->device = device;
  h->D = cfg->embed_dim; h->L = cfg->n_layers; h->G = G; h->N = G * G;
  h->C = cfg->n_channels; h->patch = cfg->patch_size; h->img = cfg->image_size;
  h->pd = h->C * h->patch * h->patch; h->H4 = cfg->mlp_multiplier * h->D;
  h->E = cfg->noise_embed_dims; h->Te = cfg->text_emb_size;
  if (build_params(h)) { tld_denoiser_destroy(h); return 1; }
  if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_out, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_tables, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&h->ev_t0) != cudaSuccess || cudaEventCreate(&h->ev_t1) != cudaSuccess) {
    tld_denoiser_destroy(h);
    return fail("tld_denoiser_create: stream/event creation failed");
  }
  if (dev_alloc(h, &h->step_ptr, 1)) { tld_denoiser_destroy(h); return 1; }
  *out = h;
  return 0;
}

void tld_denoiser_destroy(tld_denoiser* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  free_workspace(h);
  for (void* p : h->allocs) cudaFree(p);
  void* extra[] = {h->ycond, h->kv, h->uk, h->tlevels, h->cond_scratch, h->x_t, h->x0_prev, h->x0_out, h->x0k, h->eps,
                   h->mask, h->step_table};
  for (void* p : extra)
    if (p) cudaFree(p);
  for (cudaEvent_t e : h->ev_grad)
    if (e) cudaEventDestroy(e);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  if (h->pin_host) cudaFreeHost(h->pin_host);
  cudaEvent_t evs[] = {h->ev_in, h->ev_out, h->ev_t0, h->ev_t1, h->ev_tables};
  for (cudaEvent_t e : evs)
    if (e) cudaEventDestroy(e);
  delete h;
}

int tld_denoiser_set_param(tld_denoiser* h, const char* key, const float* data, int64_t numel) {
  TLD_CHECK(h && key && data, "tld_denoiser_set_param: null argument");
  TLD_CUDA_OK(cudaSetDevice(h->device));
  auto it = h->slots.find(key);
  if (it == h->slots.end()) return fail(std::string("unexpected state_dict key: ") + key);
  Slot& s = it->second;
  if (numel != s.numel)
    return fail(std::string("size mismatch for ") + key + ": got " + std::to_string(numel) + ", expected " +
                std::to_string(s.numel));
  const int thr = 256;
  const int blocks = int((s.numel + thr - 1) / thr);
  if (s.kind == P_F32) {
    TLD_CUDA_OK(cudaMemcpy(s.dst, data, (size_t)numel * sizeof(float), cudaMemcpyDefault));
  } else {
    TLD_CUDA_OK(cudaMemcpy(h->staging, data, (size_t)numel * sizeof(float), cudaMemcpyDefault));
    if (s.shadow) TLD_CUDA_OK(cudaMemcpy(s.shadow, h->staging, (size_t)numel * sizeof(float), cudaMemcpyDeviceToDevice));
    if (s.kind == P_BF16)
      f32_to_bf16_kernel<<<blocks, thr>>>(h->staging, reinterpret_cast<bf16*>(s.dst), s.numel);
    else
      transpose_f32_kernel<<<blocks, thr>>>(h->staging, reinterpret_cast<float*>(s.dst), s.rows, s.cols);
    TLD_CUDA_OK(cudaGetLastError());
    TLD_CUDA_OK(cudaDeviceSynchronize());
  }
  s.filled = true;
  h->fold_dirty = true;
  return 0;
}

// Bulk, asynchronous refresh of the packed weights from DEVICE-resident fp32 tensors, enqueued on `stream` with no host
// synchronisation: plain copies for the fp32 slots, one conversion kernel per bf16 / transposed slot straight from the source.
// The Python mirror calls this before EVERY forward / generate / training step: parameters are modified in place by
// optimisers and EMA updates in ways torch's version counters do not always record (fused Adam, `.data` arithmetic as in
// tld/train.py:55-58), so a cached copy can never be trusted; the refresh costs one pass over the weights (~0.15 ms).
int tld_denoiser_set_params_async(tld_denoiser* h, int n, const char* const* keys, const float* const* data,
                                  const int64_t* numels, void* stream) {
  TLD_CHECK(h && keys && data && numels && n >= 0, "tld_denoiser_set_params_async: bad argument");
  TLD_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  RefreshBatch batch;
  int filled = 0;
  auto flush = [&]() -> int {
    if (filled == 0) return 0;
    refresh_params_kernel<<<dim3(64, filled), 256, 0, st>>>(batch);
    TLD_CUDA_OK(cudaGetLastError());
    filled = 0;
    return 0;
  };
  for (int i = 0; i < n; ++i) {
    TLD_CHECK(keys[i] && data[i], "tld_denoiser_set_params_async: null entry");
    auto it = h->slots.find(keys[i]);
    if (it == h->slots.end()) return fail(std::string("unexpected state_dict key: ") + keys[i]);
    Slot& s = it->second;
    if (numels[i] != s.numel)
      return fail(std::string("size mismatch for ") + keys[i] + ": got " + std::to_string(numels[i]) + ", expected " +
                  std::to_string(s.numel));
    RefreshEntry& e = batch.e[filled++];
    e.src = data[i];
    e.dst = s.dst;
    e.numel = s.numel;
    e.kind = s.kind == P_F32 ? 0 : (s.kind == P_BF16 ? 1 : 2);
    e.rows = s.rows;
    e.cols = s.cols > 0 ? s.cols : 1;
    e.pad = 0;
    s.filled = true;
    if (filled == REFRESH_BATCH && flush()) return 1;
    if (s.shadow && ln_fold_requested()) {   // the fp32 copy the LayerNorm-folded weights are rebuilt from (226 MB per refresh
                                             // at the 100M model: only written while the fold is switched on)
      RefreshEntry& e2 = batch.e[filled++];
      e2 = e;
      e2.dst = s.shadow;
      e2.kind = 0;
      if (filled == REFRESH_BATCH && flush()) return 1;
    }
  }
  h->fold_dirty = true;
  return flush();
}

long long tld_forward_serial(tld_denoiser* h) { return h ? h->fwd_serial : -1; }

int tld_denoiser_missing_params(tld_denoiser* h) {
  if (!h) return -1;
  int n = 0;
  for (auto& kv : h->slots) n += kv.second.filled ? 0 : 1;
  return n;
}

int tld_denoiser_forward(tld_denoiser* h, const float* x, const float* noise_level, const float* label, float* out,
                         int batch, void* stream) {
  TLD_CHECK(h && x && noise_level && label && out, "tld_denoiser_forward: null argument");
  TLD_CHECK(batch > 0, "tld_denoiser_forward: batch must be positive");
  TLD_CHECK(tld_denoiser_missing_params(h) == 0, "tld_denoiser_forward: parameters missing (call tld_denoiser_set_param for every state_dict key)");
  TLD_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (ensure_workspace(h, batch) || ensure_cond(h, 2 * batch)) return 1;
  ++h->fwd_serial;   // x_res and the conditioning rows are shared with the training path
  const long long kvs = (long long)h->L * 2 * h->D;
  // conditioning tokens: rows [0,B) noise token, rows [B,2B) label token (denoiser.py:117-122)
  if (launch_cond_noise(noise_level, batch, h->E, h->D, h->cond, h->ycond, h->cond_scratch, st)) return 1;
  if (launch_cond_label(label, batch, batch, h->Te, h->D, h->cond, h->ycond + (size_t)batch * h->D, h->cond_scratch, st))
    return 1;
  // K|V of both cond tokens for every layer in one GEMM (transformer_blocks.py:71)
  if (launch_gemm(EPI_F32, h->ycond, h->D, h->wkv_all, h->D, 2 * batch, int(kvs), h->D, h->kv, int(kvs), nullptr,
                  nullptr, st))
    return 1;
  if (fold_xattn_keys(h, 2 * batch, st)) return 1;
  if (launch_embed(x, batch, batch, h->C, h->img, h->patch, h->D, h->emb, h->x_res, st)) return 1;
  if (use_ln_fold(h) && ensure_fold(h, st)) return 1;
  return run_blocks(h, batch, h->kv, kvs, h->kv + (size_t)batch * kvs, kvs, nullptr, out, st);
}

// What tld_sampler_edit adds to a generate call; sampler_run takes nullptr for a plain generate.
struct EditInputs {
  const float* init_latent;  // x0k [B,C,H,W]
  const float* mask;         // [B,1,H,W] or nullptr (no blend: the generate step graph is replayed)
  bool from_pure_noise;      // start from eps with the first level forced to 0.99, as generate does
};

// The body of tld_sampler_generate and tld_sampler_edit (arguments already checked).  `noise` is the initial noise of a
// generate call, or the eps of an edit.
static int sampler_run(tld_denoiser* h, const float* labels, const float* noise, const EditInputs* edit,
                       float* latent_out, int num_imgs, const double* noise_levels, int n_levels, float class_guidance,
                       float sharp_f, float bright_f, int use_ddpm_plus, void* stream) {
  TLD_CUDA_OK(cudaSetDevice(h->device));
  cudaStream_t caller = reinterpret_cast<cudaStream_t>(stream);
  cudaStream_t st = h->own_stream;

  // ---- multistep coefficients on the host (diffusion.py:54-57,71-81), python-float (double) arithmetic
  std::vector<double> sig(noise_levels, noise_levels + n_levels);
  if (!edit || edit->from_pure_noise) sig[0] = 0.99;   // an edit from partway down the schedule uses its levels verbatim
  const int calls = (int)sig.size();
  std::vector<double> rs;
  if (use_ddpm_plus) {
    std::vector<double> lam(calls), hs;
    for (int i = 0; i < calls; ++i) lam[i] = log((1.0 - sig[i]) / sig[i]);
    for (int i = 1; i < calls; ++i) hs.push_back(lam[i] - lam[i - 1]);
    for (size_t i = 1; i < hs.size(); ++i) rs.push_back(hs[i - 1] / hs[i]);
  }
  std::vector<StepCoef> table(calls);
  std::vector<float> tl(calls);
  for (int i = 0; i < calls; ++i) {
    StepCoef sc{};
    sc.guidance = class_guidance;
    sc.one_minus_g = (float)(1.0 - (double)class_guidance);
    sc.sharp = sharp_f;
    sc.bright = bright_f;
    if (i < calls - 1) {
      const double cur = sig[i], next = sig[i + 1];
      tl[i] = (float)cur;
      sc.dsig = (float)(cur - next);
      sc.next = (float)next;
      sc.cur = (float)cur;
      sc.one_minus_next = (float)(1.0 - next);
      if (i > 0 && use_ddpm_plus) {
        sc.c1 = (float)(1.0 + 1.0 / (2.0 * rs[i - 1]));
        sc.c2 = (float)(1.0 / (2.0 * rs[i - 1]));
      } else {
        sc.c1 = 1.f;
        sc.c2 = 0.f;
      }
    } else {
      tl[i] = (float)sig[calls - 1];  // final prediction at next_noise (diffusion.py:85)
      sc.is_final = 1;
    }
    table[i] = sc;
  }

  // ---- buffers
  const int Beff = 2 * num_imgs;
  const long long hw = (long long)h->img * h->img;
  const long long img_elems = (long long)num_imgs * h->C * hw;
  if (ensure_workspace(h, Beff) || ensure_cond(h, calls + Beff)) return 1;
  ++h->fwd_serial;
  if (num_imgs > h->sampler_batch) {
    TLD_CUDA_OK(cudaDeviceSynchronize());
    float** bufs[] = {&h->x_t, &h->x0_prev, &h->x0_out, &h->x0k, &h->eps};
    for (float** b : bufs) {
      if (*b) cudaFree(*b);
      if (dev_alloc(h, b, img_elems, false)) return 1;
    }
    if (h->mask) cudaFree(h->mask);
    if (dev_alloc(h, &h->mask, num_imgs * hw, false)) return 1;
    h->sampler_batch = num_imgs;
    drop_step_graphs(h);
  }
  if (calls > h->step_table_cap) {
    TLD_CUDA_OK(cudaDeviceSynchronize());
    if (h->step_table) cudaFree(h->step_table);
    if (dev_alloc(h, &h->step_table, calls, false)) return 1;
    h->step_table_cap = calls;
    drop_step_graphs(h);
  }

  // ---- per-call host tables go through a library-owned pinned buffer: the copies are asynchronous and the host never
  // blocks here (at batch 1 of the 1024-px sweep a stream synchronize per call was visible); the only wait is for the
  // PREVIOUS call's copies to have left the buffer, which is long over by the time a caller comes back
  const size_t table_bytes = sizeof(StepCoef) * calls, tl_bytes = sizeof(float) * calls;
  if (table_bytes + tl_bytes > h->pin_cap) {
    if (h->pin_host) { TLD_CUDA_OK(cudaEventSynchronize(h->ev_tables)); cudaFreeHost(h->pin_host); h->pin_host = nullptr; h->pin_cap = 0; }
    const size_t want = 2 * (table_bytes + tl_bytes);
    TLD_CUDA_OK(cudaHostAlloc(&h->pin_host, want, cudaHostAllocDefault));
    h->pin_cap = want;
  } else {
    TLD_CUDA_OK(cudaEventSynchronize(h->ev_tables));
  }
  memcpy(h->pin_host, table.data(), table_bytes);
  memcpy(reinterpret_cast<char*>(h->pin_host) + table_bytes, tl.data(), tl_bytes);

  // order after the caller's stream
  TLD_CUDA_OK(cudaEventRecord(h->ev_in, caller));
  TLD_CUDA_OK(cudaStreamWaitEvent(st, h->ev_in, 0));
  TLD_CUDA_OK(cudaMemcpyAsync(h->step_table, h->pin_host, table_bytes, cudaMemcpyHostToDevice, st));
  TLD_CUDA_OK(cudaMemcpyAsync(h->tlevels, reinterpret_cast<char*>(h->pin_host) + table_bytes, tl_bytes, cudaMemcpyHostToDevice, st));
  TLD_CUDA_OK(cudaEventRecord(h->ev_tables, st));
  TLD_CUDA_OK(cudaMemsetAsync(h->step_ptr, 0, sizeof(int), st));
  if (!edit) {
    TLD_CUDA_OK(cudaMemcpyAsync(h->x_t, noise, sizeof(float) * img_elems, cudaMemcpyDeviceToDevice, st));
  } else {
    // the inputs go to handle-owned buffers: the masked step graph reads them at baked-in addresses
    TLD_CUDA_OK(cudaMemcpyAsync(h->eps, noise, sizeof(float) * img_elems, cudaMemcpyDeviceToDevice, st));
    TLD_CUDA_OK(cudaMemcpyAsync(h->x0k, edit->init_latent, sizeof(float) * img_elems, cudaMemcpyDeviceToDevice, st));
    if (edit->mask)
      TLD_CUDA_OK(cudaMemcpyAsync(h->mask, edit->mask, sizeof(float) * num_imgs * hw, cudaMemcpyDeviceToDevice, st));
    // x_t = sig[0]*eps + (1-sig[0])*x0k (the training corruption, tld/train.py:130), or eps from pure noise
    if (launch_edit_start(h->x_t, h->eps, h->x0k, (float)sig[0], (float)(1.0 - sig[0]), edit->from_pure_noise, img_elems, st))
      return 1;
  }

  // ---- conditioning hoisted out of the loop: the noise token depends only on the step, the label token only
  // on the sample (SURVEY.md §2.2 K13/K22).  rows [0, 2B): label tokens; rows [2B, 2B+calls): noise tokens.  The label
  // rows come FIRST so that every address the captured graph bakes in depends on the batch size alone: a second call
  // with the same batch and a different number of steps replays the same graph on correctly placed rows.
  const long long kvs = (long long)h->L * 2 * h->D;
  if (use_ln_fold(h) && ensure_fold(h, st)) return 1;
  if (launch_cond_label(labels, Beff, num_imgs, h->Te, h->D, h->cond, h->ycond, h->cond_scratch, st)) return 1;
  if (launch_cond_noise(h->tlevels, calls, h->E, h->D, h->cond, h->ycond + (size_t)Beff * h->D, h->cond_scratch, st))
    return 1;
  if (launch_gemm(EPI_F32, h->ycond, h->D, h->wkv_all, h->D, calls + Beff, int(kvs), h->D, h->kv, int(kvs), nullptr,
                  nullptr, st))
    return 1;
  if (fold_xattn_keys(h, calls + Beff, st)) return 1;
  const float* kv1 = h->kv;
  const float* kv0 = h->kv + (size_t)Beff * kvs;

  // ---- one diffusion step = one CUDA graph (embed of cat[x,x] -> L blocks -> out-proj -> CFG + update).  A masked edit has
  // its own graph, which differs in the update kernel only; an unmasked edit replays the generate graph.
  const bool masked = edit && edit->mask;
  cudaGraphExec_t& graph_exec = masked ? h->graph_exec_masked : h->graph_exec;
  int& graph_batch = masked ? h->graph_batch_masked : h->graph_batch;
  int& graph_epoch = masked ? h->graph_epoch_masked : h->graph_epoch;
  if (!graph_exec || graph_batch != num_imgs || graph_epoch != g_option_epoch) {
    if (graph_exec) { cudaGraphExecDestroy(graph_exec); graph_exec = nullptr; }
    cudaGraph_t graph = nullptr;
    TLD_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    int rc = launch_embed(h->x_t, num_imgs, Beff, h->C, h->img, h->patch, h->D, h->emb, h->x_res, st);
    if (!rc) rc = run_blocks(h, Beff, kv0, kvs /*row = *step_ptr*/, kv1, kvs, h->step_ptr, h->model_out, st, num_imgs);
    if (!rc)
      rc = launch_cfg_update(h->model_out, h->x_t, h->x0_prev, h->x0_out, h->step_table, h->step_ptr, num_imgs, h->C,
                             h->img * h->img, st, h->x0k, h->eps, masked ? h->mask : nullptr);
    if (!rc) rc = launch_advance_step(h->step_ptr, st);
    cudaError_t ce = cudaStreamEndCapture(st, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return 1; }
    TLD_CUDA_OK(ce);
    ce = cudaGraphInstantiate(&graph_exec, graph, 0);
    cudaGraphDestroy(graph);
    TLD_CUDA_OK(ce);
    graph_batch = num_imgs;
    graph_epoch = g_option_epoch;
  }
  TLD_CUDA_OK(cudaEventRecord(h->ev_t0, st));
  for (int i = 0; i < calls; ++i) TLD_CUDA_OK(cudaGraphLaunch(graph_exec, st));
  TLD_CUDA_OK(cudaEventRecord(h->ev_t1, st));
  TLD_CUDA_OK(cudaMemcpyAsync(latent_out, h->x0_out, sizeof(float) * img_elems, cudaMemcpyDeviceToDevice, st));
  TLD_CUDA_OK(cudaEventRecord(h->ev_out, st));
  TLD_CUDA_OK(cudaStreamWaitEvent(caller, h->ev_out, 0));
  h->last_launches = (long long)calls * (kernels_per_forward(h) + 2) + 3 + (use_fused_xattn(h) ? h->L : 0) + (edit ? 1 : 0);
  h->last_loop_ms = -1.f;
  return 0;
}

int tld_sampler_generate(tld_denoiser* h, const float* labels, const float* seeds, float* latent_out, int num_imgs,
                         const double* noise_levels, int n_levels, float class_guidance, float sharp_f,
                         float bright_f, int use_ddpm_plus, void* stream) {
  TLD_CHECK(h && labels && seeds && latent_out && noise_levels, "tld_sampler_generate: null argument");
  TLD_CHECK(num_imgs > 0, "tld_sampler_generate: num_imgs must be positive");
  TLD_CHECK(n_levels >= 2, "tld_sampler_generate: need at least 2 noise levels");
  TLD_CHECK(tld_denoiser_missing_params(h) == 0, "tld_sampler_generate: parameters missing");
  return sampler_run(h, labels, seeds, nullptr, latent_out, num_imgs, noise_levels, n_levels, class_guidance, sharp_f,
                     bright_f, use_ddpm_plus, stream);
}

int tld_sampler_edit(tld_denoiser* h, const float* labels, const float* noise, const float* init_latent, const float* mask,
                     float* latent_out, int num_imgs, const double* noise_levels, int n_levels, int from_pure_noise,
                     float class_guidance, int use_ddpm_plus, void* stream) {
  TLD_CHECK(h && labels && noise && init_latent && latent_out && noise_levels, "tld_sampler_edit: null argument");
  TLD_CHECK(num_imgs > 0, "tld_sampler_edit: num_imgs must be positive");
  TLD_CHECK(n_levels >= 2, "tld_sampler_edit: need at least 2 noise levels");
  TLD_CHECK(tld_denoiser_missing_params(h) == 0, "tld_sampler_edit: parameters missing");
  const EditInputs edit{init_latent, mask, from_pure_noise != 0};
  return sampler_run(h, labels, noise, &edit, latent_out, num_imgs, noise_levels, n_levels, class_guidance, 0.f, 0.f,
                     use_ddpm_plus, stream);
}

int tld_sampler_last_stats(tld_denoiser* h, float* loop_ms, int64_t* kernel_launches) {
  TLD_CHECK(h, "tld_sampler_last_stats: null handle");
  TLD_CUDA_OK(cudaSetDevice(h->device));
  if (h->last_loop_ms < 0.f) {
    TLD_CUDA_OK(cudaEventSynchronize(h->ev_t1));
    TLD_CUDA_OK(cudaEventElapsedTime(&h->last_loop_ms, h->ev_t0, h->ev_t1));
  }
  if (loop_ms) *loop_ms = h->last_loop_ms;
  if (kernel_launches) *kernel_launches = h->last_launches;
  return 0;
}

// ------------------------------------------------------------------------------------------ single ops
int tld_op_gemm(int epi, const uint16_t* A, const uint16_t* W, int M, int N, int K, void* out, const float* bias,
                void* stream) {
  TLD_CHECK(epi == EPI_BF16 || epi == EPI_BIAS_BF16 || epi == EPI_BIAS_RESID_F32 || epi == EPI_F32,
            "tld_op_gemm: epilogue must be 0, 1, 2 or 4");
  return launch_gemm(epi, reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(W), K, M, N, K, out, N,
                     bias, nullptr, reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_gemm_mn(int epi, const uint16_t* A, const uint16_t* B, int M, int N, int K, void* out, void* stream) {
  return launch_gemm_mn(epi, reinterpret_cast<const bf16*>(A), M, reinterpret_cast<const bf16*>(B), N, M, N, K, out, N,
                        reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_gemm_nn(int epi, const uint16_t* A, const uint16_t* B, int M, int N, int K, void* out, void* stream) {
  return launch_gemm_nn(epi, reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(B), N, M, N, K, out, N,
                        reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_gemm_xattn(const uint16_t* A, const uint16_t* Wq, int M, int D, float* x, const float* kv0,
                      const float* kv1, int n_tok, void* stream) {
  XattnArgs xa;
  xa.kv0 = kv0; xa.kv1 = kv1;
  xa.kv0_stride = 2LL * D; xa.kv1_stride = 2LL * D;
  xa.step_ptr = nullptr; xa.n_tok = n_tok; xa.embed_dim = D;
  return launch_gemm(EPI_XATTN_RESID_F32, reinterpret_cast<const bf16*>(A), D, reinterpret_cast<const bf16*>(Wq), D, M,
                     D, D, x, D, nullptr, &xa, reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_gemm_lnfold(const uint16_t* A, const uint16_t* Wf, int M, int N, int K, uint16_t* out, const float* col_c,
                       const float* col_s, const float* row_part, int n_part, void* stream) {
  LnFoldArgs ln{col_s, reinterpret_cast<const float2*>(row_part), n_part, 1e-5f, nullptr, 0, nullptr};
  return launch_gemm(EPI_LNFOLD_BF16, reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(Wf), K, M, N, K, out, N,
                     col_c, nullptr, reinterpret_cast<cudaStream_t>(stream), &ln);
}

int tld_op_gemm_bias_resid_lnp(const uint16_t* A, const uint16_t* W, int M, int N, int K, float* x, const float* bias,
                               uint16_t* xb_out, float* part_out, void* stream) {
  LnFoldArgs ln{nullptr, nullptr, 0, 1e-5f, reinterpret_cast<bf16*>(xb_out), N, reinterpret_cast<float2*>(part_out)};
  return launch_gemm(EPI_BIAS_RESID_LNP, reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(W), K, M, N, K, x, N,
                     bias, nullptr, reinterpret_cast<cudaStream_t>(stream), &ln);
}

int tld_op_gemm_xattn_lnp(const uint16_t* A, const uint16_t* Wq, int M, int D, float* x, const float* kv0, const float* kv1,
                          int n_tok, uint16_t* xb_out, float* part_out, void* stream) {
  XattnArgs xa;
  xa.kv0 = kv0; xa.kv1 = kv1;
  xa.kv0_stride = 2LL * D; xa.kv1_stride = 2LL * D;
  xa.step_ptr = nullptr; xa.n_tok = n_tok; xa.embed_dim = D;
  LnFoldArgs ln{nullptr, nullptr, 0, 1e-5f, reinterpret_cast<bf16*>(xb_out), D, reinterpret_cast<float2*>(part_out)};
  return launch_gemm(EPI_XATTN_RESID_LNP, reinterpret_cast<const bf16*>(A), D, reinterpret_cast<const bf16*>(Wq), D, M, D, D, x, D,
                     nullptr, &xa, reinterpret_cast<cudaStream_t>(stream), &ln);
}

int tld_op_rowstats_cast(const float* x, uint16_t* xb, float* part, int rows, int D, void* stream) {
  return launch_rowstats_cast(x, reinterpret_cast<bf16*>(xb), reinterpret_cast<float2*>(part), rows, D,
                              reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_ln_fold_weights(const float* W, const float* gamma, const float* beta, const float* bias, uint16_t* Wf, float* s,
                           float* c, int N, int K, void* stream) {
  return launch_ln_fold_weights(W, gamma, beta, bias, reinterpret_cast<bf16*>(Wf), s, c, N, K, reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_layernorm(const float* x, const float* gamma, const float* beta, uint16_t* y, int rows, int D,
                     void* stream) {
  return launch_layernorm_bf16(x, gamma, beta, reinterpret_cast<bf16*>(y), rows, D,
                               reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_self_attention(const uint16_t* qkv, float* x, int batch, int n_tok, int D, int impl, void* stream) {
  TLD_CHECK(impl == 0 || impl == 1 || impl == 3,
            "tld_op_self_attention: impl must be 0 (auto), 1 (mma.sync) or 3 (tcgen05 persistent)");
  return launch_self_attention(reinterpret_cast<const bf16*>(qkv), x, batch, n_tok, D,
                               reinterpret_cast<cudaStream_t>(stream), impl);
}

int tld_op_ln_xattn_ln(float* x, const float* g2, const float* b2, const float* g3, const float* b3, const uint16_t* Wq,
                       const float* kv0, const float* kv1, int batch, int n_tok, int D, float* uk_scratch, uint16_t* y, void* stream) {
  TLD_CHECK(uk_scratch != nullptr && D % 64 == 0, "tld_op_ln_xattn_ln: needs a [2 * batch, D / 64, D] fp32 scratch buffer");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long uks = (long long)(D / 64) * D;
  if (launch_xattn_fold_keys(kv0, 2LL * D, batch, reinterpret_cast<const bf16*>(Wq), uk_scratch, uks, D, st)) return 1;
  if (launch_xattn_fold_keys(kv1, 2LL * D, batch, reinterpret_cast<const bf16*>(Wq), uk_scratch + (size_t)batch * uks, uks, D, st)) return 1;
  return launch_ln_xattn_ln(x, g2, b2, g3, b3, uk_scratch, uks, uk_scratch + (size_t)batch * uks, uks, kv0, 2LL * D, kv1, 2LL * D,
                            nullptr, reinterpret_cast<bf16*>(y), batch * n_tok, n_tok, D, st);
}

int tld_op_qkv_attention(const uint16_t* xn, const uint16_t* Wqkv, float* x, int batch, int n_tok, int D, void* stream) {
  return launch_qkv_attention(reinterpret_cast<const bf16*>(xn), reinterpret_cast<const bf16*>(Wqkv), x, batch, n_tok, D,
                              reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_gemm_up_dwconv_gelu(const uint16_t* A, const uint16_t* W, const float* col_c, const float* col_s,
                               const float* row_sums, const float* dw_w9, const float* dw_b, uint16_t* out, int batch, int K,
                               int N, void* stream) {
  return launch_gemm_up_dwconv_gelu(reinterpret_cast<const bf16*>(A), K, reinterpret_cast<const bf16*>(W), K, batch * 256, N, K,
                                    col_c, col_s, reinterpret_cast<const float2*>(row_sums), 1, 1e-5f, dw_w9, dw_b,
                                    reinterpret_cast<bf16*>(out), reinterpret_cast<cudaStream_t>(stream));
}

int tld_op_dwconv_gelu(const uint16_t* hsrc, const float* w9, const float* bias, uint16_t* g, int batch, int grid,
                       int channels, void* stream) {
  return launch_dwconv_gelu(reinterpret_cast<const bf16*>(hsrc), w9, bias, reinterpret_cast<bf16*>(g), batch, grid,
                            channels, reinterpret_cast<cudaStream_t>(stream));
}

}  // extern "C"

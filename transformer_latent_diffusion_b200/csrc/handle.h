// The library handle shared by api.cu (inference) and train.cu (training step).
#pragma once
#include <map>
#include <string>
#include <vector>

#include "../../include/tld_b200.h"
#include "common.h"

namespace tld {

enum PackKind { P_F32, P_BF16, P_TRANSPOSE_F32 };
struct Slot {
  PackKind kind;
  void* dst;
  float* shadow = nullptr;  // optional fp32 copy (weights that are also folded with a LayerNorm's gamma)
  long long numel;
  int rows, cols;  // for P_TRANSPOSE_F32: source is [rows, cols]
  bool filled;
};

}  // namespace tld

using namespace tld;  // internal header: the handle is the C-ABI opaque type and lives in the global namespace

struct tld_denoiser {
  tld_config cfg;
  int device;
  int D, L, N, G, pd, H4, E, Te, C, img, patch;
  std::map<std::string, Slot> slots;
  std::vector<void*> allocs;
  float* staging = nullptr;
  long long staging_elems = 0;

  // parameters (device)
  CondW cond;
  EmbedW emb;
  float *out_w, *out_b;
  struct Layer {
    bf16 *wqkv, *wq, *wup, *wdown;
    float *ln1w, *ln1b, *ln2w, *ln2b, *ln3w, *ln3b, *bup, *dww9, *dwb, *bdown;
  };
  std::vector<Layer> layers;
  bf16* wkv_all = nullptr;  // [L*2D, D]
  // LayerNorm fold (inference path, gemm_tcgen05.cuh): norm1 -> qkv_linear and norm3 -> mlp.0.  W' = bf16(gamma (.) W) with the
  // column constants s_n = sum_k W'_nk, c_n = sum_k beta_k W_nk (+ bias), rebuilt from fp32 shadows whenever a parameter changed
  struct LayerFold {
    float *wqkv32, *wup32;          // fp32 shadows of the two foldable weights
    bf16 *wqkv_f, *wup_f;
    float *s_qkv, *c_qkv, *s_up, *c_up;
  };
  std::vector<LayerFold> fold;
  bool fold_dirty = true;

  // activation workspace, sized for ws_batch samples
  int ws_batch = 0;
  float* x_res = nullptr;   // [T, D] fp32 residual stream
  bf16* xn = nullptr;       // [T, D]
  bf16* qkv = nullptr;      // [T, 3D]
  bf16* hid = nullptr;      // [T, 4D]
  bf16* hid2 = nullptr;     // [T, 4D]
  float* model_out = nullptr;  // [B, C, H, W]
  bf16* xb[2] = {nullptr, nullptr};       // bf16 copy of the residual stream, ping-pong (producer epilogues write the other one)
  float2* part[2] = {nullptr, nullptr};   // [T, D/32] per-32-column (sum, sum of squares) partials of the residual rows
  // conditioning workspace
  int ws_cond_rows = 0;
  bf16* ycond = nullptr;    // [rows, D]
  float* kv = nullptr;      // [rows, L*2D]
  float* uk = nullptr;      // [rows, L, H, D] cross-attention keys folded through Wq (xattn_rowwise.cu); nullptr = table too large
  float* tlevels = nullptr; // [max steps]
  float* cond_scratch = nullptr;  // [rows, E + 2 D] fp32 intermediates of the conditioning MLP (inference path)

  // sampler state
  cudaStream_t own_stream = nullptr;
  cudaEvent_t ev_in = nullptr, ev_out = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
  float *x_t = nullptr, *x0_prev = nullptr, *x0_out = nullptr;
  float *x0k = nullptr, *eps = nullptr;  // tld_sampler_edit: known latent and noise [B,C,H,W]
  float* mask = nullptr;                 // tld_sampler_edit: [B,1,H,W], 1 = regenerate
  int sampler_batch = 0;
  StepCoef* step_table = nullptr;
  int step_table_cap = 0;
  int* step_ptr = nullptr;
  cudaGraphExec_t graph_exec = nullptr;
  int graph_batch = -1;
  int graph_epoch = -1;          // tld_set_option epoch the graph was captured under
  cudaGraphExec_t graph_exec_masked = nullptr;  // the same step with the masked update (both bake in the sampler buffers)
  int graph_batch_masked = -1;
  int graph_epoch_masked = -1;
  void* pin_host = nullptr;      // pinned staging of the per-call step table + noise levels
  size_t pin_cap = 0;
  cudaEvent_t ev_tables = nullptr;  // the previous call's table copies have left pin_host
  float last_loop_ms = 0.f;
  long long last_launches = 0;

  // every forward-like call (forward, sampler generate / edit, training forward) bumps fwd_serial; train_serial remembers the one whose
  // activations the training buffers (and x_res) currently hold, so a backward after any later forward is refused
  long long fwd_serial = 0;
  long long train_serial = -1;

  // ---- training step (train.cu) ----
  struct TrainLayer {
    float *xs0, *xs1, *xs2;        // residual stream before self-attn / cross-attn / MLP, fp32 [T,D]
    bf16 *qkv, *hid, *hid2;        // saved GEMM outputs
    bf16 *xn0, *xn1, *xn2;         // saved LayerNorm outputs (norm1/2/3): the A operands of the wgrad GEMMs, not recomputed
  };
  std::vector<TrainLayer> tl;
  int train_batch = 0;
  std::vector<void*> train_allocs;
  std::map<std::string, std::pair<float*, long long>> grads;  // reference-layout fp32 gradient of every parameter
  float* grad_arena = nullptr;
  long long grad_elems = 0;
  std::vector<cudaEvent_t> ev_grad;  // [L+1]: gradients of layer l complete (l < L) / whole backward complete (index L)
  // scratch (sized with train_batch)
  float *t_dx = nullptr, *t_dxn = nullptr, *t_xfinal = nullptr;
  bf16 *t_a = nullptr, *t_aT = nullptr, *t_big = nullptr, *t_bigT = nullptr, *t_big2 = nullptr, *t_xnT = nullptr, *t_q = nullptr;
  float *t_dkv = nullptr, *t_cond_pre = nullptr, *t_cond_h1 = nullptr, *t_cond_a1 = nullptr, *t_cond_emb = nullptr;
  float *t_small = nullptr;
};

// api.cu: (re)allocate the inference workspaces for `batch` samples and `cond_rows` conditioning rows
int tld_internal_ensure(tld_denoiser* h, int batch, int cond_rows);

// Internal launcher declarations shared by the translation units of libtld_b200.so.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

namespace tld {

typedef __nv_bfloat16 bf16;

// error plumbing: every launcher returns 0 or sets the thread-local message and returns non-zero
int fail(const std::string& msg);
const char* last_error();
#define TLD_CUDA_OK(expr)                                                                      \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return ::tld::fail(std::string(#expr) + " -> " + cudaGetErrorString(_e) + " @" + __FILE__ + ":" + \
                         std::to_string(__LINE__));                                            \
  } while (0)
#define TLD_CHECK(cond, msg)                  \
  do {                                        \
    if (!(cond)) return ::tld::fail(msg);     \
  } while (0)

int sm_count();
// Grow-only fp32 scratch buffer, one per (current device, slot): reduction partials of the backward / GroupNorm kernels.
// Per device so that handles on different GPUs of one process never share a pointer; returns nullptr on failure.
enum ScratchSlot { SCR_COLSUM = 0, SCR_LN_BWD, SCR_DWCONV_DW, SCR_SPLIT_K, SCR_GROUPNORM, SCR_ATTN_BWD, SCR_VAE_ATTN, SCR_COUNT };
float* device_scratch(ScratchSlot slot, size_t n_floats);
void set_pdl(int v);  // 1 = launch the step kernels with programmatic dependent launch, 0 = plain launches (default)

// ---------------------------------------------------------------- gemm.cu
struct XattnArgs {
  const float* kv0;
  const float* kv1;
  long long kv0_stride, kv1_stride;
  const int* step_ptr;
  int n_tok;
  int embed_dim;
};
// LayerNorm folding (gemm_tcgen05.cuh): consumer side = EPI_LNFOLD_BF16 (col_s, row_part, n_part = K / 32, ln_eps; `bias` is
// c_n); producer side = EPI_BIAS_RESID_LNP / EPI_XATTN_RESID_LNP (xb_out = bf16 copy of the new rows, part_out [M, N/32])
struct LnFoldArgs {
  const float* col_s;
  const float2* row_part;
  int n_part;
  float ln_eps;
  bf16* xb_out;
  int ldxb;
  float2* part_out;
};
// C[M,N] = A[M,K] * W[N,K]^T with a fused epilogue (see gemm_tcgen05.cuh). lda/ldw in elements.
int launch_gemm(int epi, const bf16* A, int lda, const bf16* W, int ldw, int M, int N, int K, void* out, int ldo,
                const float* bias, const XattnArgs* xa, cudaStream_t st, const LnFoldArgs* ln = nullptr);
// fp32 rows -> bf16 copy + per-32-column (sum, sum of squares) partials [rows, D/32] (the producer side of the LayerNorm fold
// for rows that no GEMM epilogue produced: the patch embedding)
int launch_rowstats_cast(const float* x, bf16* xb, float2* part, int rows, int D, cudaStream_t st);
// W'[n,k] = bf16(gamma[k] W[n,k]); s[n] = sum_k W'[n,k]; c[n] = sum_k beta[k] W[n,k] (+ bias[n])
int launch_ln_fold_weights(const float* W, const float* gamma, const float* beta, const float* bias, bf16* Wf, float* s,
                           float* c, int N, int K, cudaStream_t st);

// C[M,N] = A^T B with A stored [K,M], B stored [K,N] (weight-gradient shape, K = tokens); epi = EPI_F32 or EPI_BF16
int launch_gemm_mn(int epi, const bf16* A, int lda, const bf16* B, int ldb, int M, int N, int K, void* out, int ldo,
                   cudaStream_t st);
// C[M,N] = A B with A [M,K] as usual and B stored [K,N] (data-gradient shape dX = dY W, weight untransposed)
int launch_gemm_nn(int epi, const bf16* A, int lda, const bf16* B, int ldb, int M, int N, int K, void* out, int ldo,
                   cudaStream_t st);

// ---------------------------------------------------------------- rowwise.cu
int launch_layernorm_bf16(const float* x, const float* gamma, const float* beta, bf16* y, int rows, int D,
                          cudaStream_t st);
struct EmbedW {
  const float* conv_w;  // [pd, pd] (out, in) with in = (c, p1, p2)
  const float* conv_b;  // [pd]
  const float* ln1_w;   // [pd]
  const float* ln1_b;
  const float* lin_wT;  // [pd, D]  (transposed nn.Linear weight)
  const float* lin_b;   // [D]
  const float* ln2_w;   // [D]
  const float* ln2_b;
  const float* pos;     // [N, D]
};
struct EmbedSave {  // optional fp32 intermediates kept for the backward pass (training)
  float* u;    // [T, pd] gathered patch
  float* c16;  // [T, pd] conv output (pre-LN)
  float* t16;  // [T, pd] LN(pd) output
  float* e;    // [T, D]  Linear(pd->D) output (pre-LN)
};
// x[Bx,C,H,W] fp32 -> tokens[Bout,N,D] fp32; sample b reads image b % Bx (CFG duplication)
int launch_embed(const float* x, int Bx, int Bout, int C, int img, int patch, int D, const EmbedW& w, float* out,
                 cudaStream_t st, const EmbedSave* sv = nullptr);
struct CondW {
  const float* speeds;  // [E/2]
  const float* w1;      // [D, E]
  const float* b1;
  const float* w2;      // [D, D]
  const float* b2;
  const float* wl;      // [D, Te]
  const float* bl;
  const float* ln_w;    // [D]
  const float* ln_b;
};
struct CondSave {  // optional fp32 intermediates kept for the backward pass (training)
  float* emb;  // [R, E]  sinusoidal features
  float* a1;   // [R, D]  W1 emb + b1 (pre-GELU)
  float* h1;   // [R, D]  gelu(a1)
  float* pre;  // [R, D]  W2 h1 + b2 (pre-LayerNorm)
};
// noise token: y[r] = LN(W2 gelu(W1 sincos(t[r]) + b1) + b2)  -> bf16 [R, D]
// scratch: fp32 [R, E + 2 D] for the MLP intermediates (unused parts when sv supplies the buffers)
int launch_cond_noise(const float* t, int R, int E, int D, const CondW& w, bf16* y, float* scratch, cudaStream_t st,
                      const CondSave* sv = nullptr);
// label token: y[r] = LN(Wl label[r] + bl); label == nullptr or r >= R_real -> zero label (uncond half)
int launch_cond_label(const float* label, int R, int R_real, int Te, int D, const CondW& w, bf16* y, float* scratch,
                      cudaStream_t st, float* pre_save = nullptr);
// g = gelu(dwconv3x3(h) + b) over the token grid; h,g bf16 [B, grid, grid, C]; w tap-major [9, C]
int launch_dwconv_gelu(const bf16* h, const float* w9, const float* bias, bf16* g, int B, int grid, int C,
                       cudaStream_t st);
// 16x16-grid tile kernel in its backward modes: mode 1: out = second * gelu'(conv(in) + bias); mode 2: out = conv^T(in)
int launch_dwconv_g16_bwd(const bf16* in, const bf16* second, const float* w9, const float* bias, bf16* out, int B, int C,
                          int mode, cudaStream_t st);
// tokens[B,N,D] fp32 -> Linear(D->pd)+bias -> unpatchify -> out[B,C,H,W] fp32
int launch_outproj(const float* x, const float* w, const float* b, float* out, int B, int C, int img, int patch,
                   int D, cudaStream_t st);

struct StepCoef {  // one entry per model call of the sampler (device table)
  float guidance, one_minus_g;
  float c1, c2;        // D = c1*x0 - c2*x0_prev   (c2 == 0: D = x0)
  float dsig, next, cur;  // x_t = (dsig*D + next*x_t)/cur
  int is_final;        // last model call: emit x0 (+ channel shifts), no x_t update
  float sharp, bright;
  float one_minus_next;   // masked edit: the kept region of x_t is reset to next*eps + one_minus_next*x0k
};
// model_out[2B,...] (cond first, uncond second) -> CFG combine -> multistep update of x_t / x0_prev / x0_out.
// mask != nullptr (masked edit, mask [B,1,H,W] clamped to [0,1], 1 = regenerate): after each update
// x_t = m*x_t + (1-m)*(next*eps + (1-next)*x0k), and the final x0_out = m*x0 + (1-m)*x0k
int launch_cfg_update(const float* model_out, float* x_t, float* x0_prev, float* x0_out, const StepCoef* table,
                      const int* step_ptr, int B, int C, int hw, cudaStream_t st, const float* x0k = nullptr,
                      const float* eps = nullptr, const float* mask = nullptr);
int launch_advance_step(int* step_ptr, cudaStream_t st);
// start state of an edit: x_t = eps (from_noise) or s0*eps + one_minus_s0*x0k, n elements
int launch_edit_start(float* x_t, const float* eps, const float* x0k, float s0, float one_minus_s0, int from_noise,
                      long long n, cudaStream_t st);

// 3x3 'same' conv as implicit GEMM: x NHWC bf16, w bf16 [Cout, 9*Cin] with K order (ky,kx,cin), bias fp32 or null
int launch_conv3x3(const bf16* x, const bf16* w, const float* bias, bf16* out, int B, int H, int W, int Cin, int Cout,
                   cudaStream_t st, const bf16* resid = nullptr, float* gn_part = nullptr);
// MLPSepConv front half fused (gemm_dwconv.cu): g = GELU(dwconv3x3(A W^T [LayerNorm-folded] + c) + dw_b) for 16x16-token samples
int launch_gemm_up_dwconv_gelu(const bf16* A, int lda, const bf16* W, int ldw, int M, int N, int K, const float* col_c,
                               const float* col_s, const float2* row_part, int n_part, float ln_eps, const float* dw_w9,
                               const float* dw_b, bf16* out, cudaStream_t st, bf16* hid_out = nullptr);
void set_gemm_ctas(int v);  // 0 auto, 1 single-CTA tiles, 2 CTA-pair tiles (experiments / tests)

// 2-D row-major TMA descriptor (bf16 or fp32), box = [box_rows, 128 bytes], 128B swizzle (gemm.cu)
int make_tmap_2d(CUtensorMap* m, const void* base, bool is_f32, long long rows, long long cols, long long ld,
                 int box_rows);
int make_tmap_tokens3d(CUtensorMap* m, const void* base, int B, int npos, int C, int box_pos);  // [B][npos][C] bf16

// ---------------------------------------------------------------- attention.cu / attention_tc.cu
// x[T,D] fp32 += softmax(q k^T / 8) v per (sample, head); qkv bf16 [T,3D] (q | k | v), head_dim 64
// impl: 0 = auto (tcgen05 when n_tok % 128 == 0, else mma.sync), 1 = mma.sync kernel, 3 = tcgen05 persistent kernel
int launch_self_attention(const bf16* qkv, float* x, int B, int n_tok, int D, cudaStream_t st, int impl = 0);
int launch_self_attention_mma(const bf16* qkv, float* x, int B, int n_tok, int D, cudaStream_t st);
int launch_self_attention_tc2(const bf16* qkv, float* x, int B, int n_tok, int D, cudaStream_t st);
// norm2 + 2-token cross-attention + residual + norm3 as one row-wise kernel on keys folded through Wq: xattn_rowwise.cu
int launch_xattn_fold_keys(const float* kv, long long kv_stride, int R, const bf16* wq, float* uk, long long uk_stride, int D,
                           cudaStream_t st);
bool ln_xattn_ln_supported(int D, int n_tok);
void set_xattn_rows(int v);  // rows per warp of the FFMA row kernel: 4 (8 warps x 255 registers) or 2 (16 warps x 128)
void set_xattn_ctas(int v);  // CTAs per SM of the FFMA row kernel: 1 (32 / rows warps) or 2 (half the warps each)
void set_xattn_mma(int v);   // 0 = FFMA row kernel, 1 / 2 / 3 = tensor-pipe dot products (tf32 mma.sync), x rounded / x split / x and keys split
int launch_ln_xattn_ln(float* x, const float* g2, const float* b2, const float* g3, const float* b3, const float* uk0,
                       long long uk0_stride, const float* uk1, long long uk1_stride, const float* kv0, long long kv0_stride,
                       const float* kv1, long long kv1_stride, const int* step_ptr, bf16* y, int rows, int n_tok, int D,
                       cudaStream_t st);
// qkv projection + attention + residual add in one CTA-pair kernel (256 tokens per sample): qkv_attention.cu
int launch_qkv_attention(const bf16* xn, const bf16* wqkv, float* x, int B, int n_tok, int D, cudaStream_t st);
void set_qkv_attention_exp_emu(int v);
void set_attention_exp_emu(int pairs_of_16);
void set_attention_bwd_impl(int v);   // 0 / 1 mma.sync kernels (default), 2 tcgen05 kernel when tokens % 256 == 0  // attention_tc2: share of exp2 evaluated on the FMA pipe instead of MUFU

}  // namespace tld

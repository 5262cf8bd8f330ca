// HBM-bound row-wise kernels of the denoiser: LayerNorm, patch embedding, conditioning tokens,
// depthwise-3x3+GELU, output projection/unpatchify and the fused CFG + multistep sampler update.
// All statistics and transcendental math in fp32; bf16 only as the tensor-core operand format.
#include <math.h>

#include "common.h"
#include "dwconv_math.cuh"
#include "launch.h"
#include "ptx.cuh"

namespace tld {

static constexpr float LN_EPS = 1e-5f;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ uint32_t pack_bf16x2_dev(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// --------------------------------------------------------------------------------------------
// LayerNorm(D) fp32 -> bf16, one warp per row.  Reference: nn.LayerNorm at transformer_blocks.py:131-138.
// V = D/128 float4 per lane; the row lives in registers between the two passes.
// --------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(256) layernorm_bf16_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, bf16* __restrict__ y,
                                                             int rows) {
  constexpr int D = V * 128;
  pdl_launch_dependents();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  pdl_wait();
  const float4* xr = reinterpret_cast<const float4*>(x + (size_t)row * D);
  float4 v[V];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < V; ++j) {
    v[j] = xr[lane + 32 * j];
    s += (v[j].x + v[j].y) + (v[j].z + v[j].w);
  }
  const float mu = warp_sum(s) * (1.0f / D);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const float a = v[j].x - mu, b = v[j].y - mu, c = v[j].z - mu, d = v[j].w - mu;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / D) + LN_EPS);
  uint2* yr = reinterpret_cast<uint2*>(y + (size_t)row * D);
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + lane + 32 * j);
    const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + lane + 32 * j);
    __nv_bfloat162 lo = __floats2bfloat162_rn((v[j].x - mu) * rstd * g.x + b.x, (v[j].y - mu) * rstd * g.y + b.y);
    __nv_bfloat162 hi = __floats2bfloat162_rn((v[j].z - mu) * rstd * g.z + b.z, (v[j].w - mu) * rstd * g.w + b.w);
    uint2 o;
    o.x = *reinterpret_cast<uint32_t*>(&lo);
    o.y = *reinterpret_cast<uint32_t*>(&hi);
    yr[lane + 32 * j] = o;
  }
}

// embed_dim = 64 x odd (the reference takes any multiple of 64: heads = D // 64, transformer_blocks.py:126-129): same scheme
// with scalar lanes, column c = lane + 32 j (coalesced 128-byte warp accesses), row held in registers.
__global__ void __launch_bounds__(256) layernorm_bf16_generic_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                                     const float* __restrict__ beta, bf16* __restrict__ y,
                                                                     int rows, int D) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + (size_t)row * D;
  const int n = D / 32;   // <= 32
  float v[32];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    v[j] = j < n ? xr[lane + 32 * j] : 0.f;
    s += v[j];
  }
  const float mu = warp_sum(s) / D;
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j)
    if (j < n) q += (v[j] - mu) * (v[j] - mu);
  const float rstd = rsqrtf(warp_sum(q) / D + LN_EPS);
#pragma unroll
  for (int j = 0; j < 32; ++j)
    if (j < n) {
      const int c = lane + 32 * j;
      y[(size_t)row * D + c] = __float2bfloat16((v[j] - mu) * rstd * __ldg(gamma + c) + __ldg(beta + c));
    }
}

int launch_layernorm_bf16(const float* x, const float* gamma, const float* beta, bf16* y, int rows, int D,
                          cudaStream_t st) {
  TLD_CHECK(D % 64 == 0 && D >= 64 && D <= 1024, "layernorm: embed_dim must be a multiple of 64 in [64,1024]");
  const int grid = (rows + 7) / 8;
  if (D % 128 != 0) {
    layernorm_bf16_generic_kernel<<<grid, 256, 0, st>>>(x, gamma, beta, y, rows, D);
    TLD_CUDA_OK(cudaGetLastError());
    return 0;
  }
  switch (D / 128) {
#define LN_CASE(V) \
  case V: if (launch_pdl(layernorm_bf16_kernel<V>, dim3(grid), dim3(256), 0, st, x, gamma, beta, y, rows)) return 1; break;
    LN_CASE(1) LN_CASE(2) LN_CASE(3) LN_CASE(4) LN_CASE(5) LN_CASE(6) LN_CASE(7) LN_CASE(8)
#undef LN_CASE
  }
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}

// --------------------------------------------------------------------------------------------
// LayerNorm fold, producer side for rows no GEMM epilogue wrote (the patch embedding): fp32 row -> bf16 copy + per-32-column
// (sum, sum of squares) partials [rows, D/32].  One warp per row; lane l holds columns 128 j + 4 l .. + 3, so a 32-column
// group is 8 consecutive lanes (xor-shuffle 1, 2, 4).  HBM-bound (D * 6 bytes per row), once per forward.
// --------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(256) rowstats_cast_kernel(const float* __restrict__ x, bf16* __restrict__ xb,
                                                            float2* __restrict__ part, int rows) {
  constexpr int D = V * 128;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float4* xr = reinterpret_cast<const float4*>(x + (size_t)row * D);
  uint2* yr = reinterpret_cast<uint2*>(xb + (size_t)row * D);
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const float4 v = xr[lane + 32 * j];
    __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<uint32_t*>(&lo);
    o.y = *reinterpret_cast<uint32_t*>(&hi);
    yr[lane + 32 * j] = o;
    float ps = (v.x + v.y) + (v.z + v.w), pq = (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
#pragma unroll
    for (int o2 = 1; o2 < 8; o2 <<= 1) {
      ps += __shfl_xor_sync(0xffffffffu, ps, o2);
      pq += __shfl_xor_sync(0xffffffffu, pq, o2);
    }
    if ((lane & 7) == 0) part[(size_t)row * (D / 32) + 4 * j + (lane >> 3)] = make_float2(ps, pq);
  }
}

int launch_rowstats_cast(const float* x, bf16* xb, float2* part, int rows, int D, cudaStream_t st) {
  TLD_CHECK(D % 128 == 0 && D >= 128 && D <= 1024, "rowstats_cast: embed_dim must be a multiple of 128 in [128,1024]");
  const int grid = (rows + 7) / 8;
  switch (D / 128) {
#define RS_CASE(V) \
  case V: rowstats_cast_kernel<V><<<grid, 256, 0, st>>>(x, xb, part, rows); break;
    RS_CASE(1) RS_CASE(2) RS_CASE(3) RS_CASE(4) RS_CASE(5) RS_CASE(6) RS_CASE(7) RS_CASE(8)
#undef RS_CASE
  }
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}

// LayerNorm fold, weight side: W'[n,k] = bf16(gamma[k] W[n,k]), s[n] = sum_k float(W'[n,k]) (the ROUNDED weights: the
// epilogue subtracts mean * s from an accumulator that was built from them), c[n] = sum_k beta[k] W[n,k] + bias[n].
// One warp per output row; runs once per weight refresh.
__global__ void __launch_bounds__(256) ln_fold_weights_kernel(const float* __restrict__ W, const float* __restrict__ gamma,
                                                              const float* __restrict__ beta, const float* __restrict__ bias,
                                                              bf16* __restrict__ Wf, float* __restrict__ s_out,
                                                              float* __restrict__ c_out, int N, int K) {
  const int n = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  const float* wr = W + (size_t)n * K;
  bf16* fr = Wf + (size_t)n * K;
  float s = 0.f, c = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float w = wr[k];
    const bf16 f = __float2bfloat16(w * __ldg(gamma + k));
    fr[k] = f;
    s += __bfloat162float(f);
    c = fmaf(__ldg(beta + k), w, c);
  }
  s = warp_sum(s);
  c = warp_sum(c);
  if (lane == 0) {
    s_out[n] = s;
    c_out[n] = c + (bias ? bias[n] : 0.f);
  }
}

int launch_ln_fold_weights(const float* W, const float* gamma, const float* beta, const float* bias, bf16* Wf, float* s,
                           float* c, int N, int K, cudaStream_t st) {
  ln_fold_weights_kernel<<<(N + 7) / 8, 256, 0, st>>>(W, gamma, beta, bias, Wf, s, c, N, K);
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}

// --------------------------------------------------------------------------------------------
// Patch embedding (denoiser.py:34-45,75-77): one warp per token.
//   u = 2x2xC patch -> t = W0 u + b0 -> LN(pd) -> e = W3 t + b3 -> LN(D) -> + pos[n]
// pd <= 64.  The D-wide vector is distributed 4 floats per lane per 128-column group.
// --------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(256) embed_kernel(const float* __restrict__ x, int Bx, int Bout, int C, int img,
                                                    int patch, EmbedW w, float* __restrict__ out, EmbedSave sv) {
  constexpr int D = V * 128;
  __shared__ float s_t[8][64];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = img / patch, N = g * g, pd = C * patch * patch;
  // tokens of the Bx distinct images; output image b + k Bx (k < Bout / Bx: the CFG pair embeds the same x_t twice) gets a copy
  const long long tok = (long long)blockIdx.x * 8 + wib;
  pdl_launch_dependents();
  if (tok >= (long long)Bx * N) return;
  pdl_wait();
  const int b = int(tok / N), n = int(tok % N);
  const int gy = n / g, gx = n % g;
  const float* xb = x + (size_t)b * C * img * img;
  // gather the patch (c, p1, p2) and apply the strided conv as a pd x pd mat-vec
  float* t = s_t[wib];
  for (int i = lane; i < pd; i += 32) {
    const int c = i / (patch * patch), p1 = (i / patch) % patch, p2 = i % patch;
    t[i] = xb[(size_t)c * img * img + (size_t)(gy * patch + p1) * img + gx * patch + p2];
  }
  __syncwarp();
  if (sv.u)
    for (int i = lane; i < pd; i += 32) sv.u[(size_t)tok * pd + i] = t[i];
  float conv[2] = {0.f, 0.f};
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int o = lane + 32 * r;
    if (o < pd) {
      float acc = w.conv_b[o];
      for (int i = 0; i < pd; ++i) acc += w.conv_w[o * pd + i] * t[i];
      conv[r] = acc;
      s += acc;
    }
  }
  const float mu1 = warp_sum(s) / pd;
  float q = 0.f;
#pragma unroll
  for (int r = 0; r < 2; ++r)
    if (lane + 32 * r < pd) q += (conv[r] - mu1) * (conv[r] - mu1);
  const float rstd1 = rsqrtf(warp_sum(q) / pd + LN_EPS);
  __syncwarp();
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int o = lane + 32 * r;
    if (o < pd) {
      t[o] = (conv[r] - mu1) * rstd1 * w.ln1_w[o] + w.ln1_b[o];
      if (sv.c16) {
        sv.c16[(size_t)tok * pd + o] = conv[r];
        sv.t16[(size_t)tok * pd + o] = t[o];
      }
    }
  }
  __syncwarp();
  // Linear pd -> D with the transposed weight [pd, D] (coalesced float4 per lane)
  float4 e[V];
  float s2 = 0.f;
#pragma unroll
  for (int j = 0; j < V; ++j) {
    float4 acc = __ldg(reinterpret_cast<const float4*>(w.lin_b) + lane + 32 * j);
    for (int i = 0; i < pd; ++i) {
      const float4 wv = __ldg(reinterpret_cast<const float4*>(w.lin_wT + (size_t)i * D) + lane + 32 * j);
      const float ti = t[i];
      acc.x += wv.x * ti;
      acc.y += wv.y * ti;
      acc.z += wv.z * ti;
      acc.w += wv.w * ti;
    }
    e[j] = acc;
    if (sv.e) reinterpret_cast<float4*>(sv.e + (size_t)tok * D)[lane + 32 * j] = acc;
    s2 += (acc.x + acc.y) + (acc.z + acc.w);
  }
  const float mu2 = warp_sum(s2) * (1.0f / D);
  float q2 = 0.f;
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const float a = e[j].x - mu2, bb = e[j].y - mu2, c = e[j].z - mu2, d = e[j].w - mu2;
    q2 += (a * a + bb * bb) + (c * c + d * d);
  }
  const float rstd2 = rsqrtf(warp_sum(q2) * (1.0f / D) + LN_EPS);
  const float4* prow = reinterpret_cast<const float4*>(w.pos + (size_t)n * D);
#pragma unroll
  for (int j = 0; j < V; ++j) {
    const float4 gm = __ldg(reinterpret_cast<const float4*>(w.ln2_w) + lane + 32 * j);
    const float4 bt = __ldg(reinterpret_cast<const float4*>(w.ln2_b) + lane + 32 * j);
    const float4 p = __ldg(prow + lane + 32 * j);
    float4 o;
    o.x = (e[j].x - mu2) * rstd2 * gm.x + bt.x + p.x;
    o.y = (e[j].y - mu2) * rstd2 * gm.y + bt.y + p.y;
    o.z = (e[j].z - mu2) * rstd2 * gm.z + bt.z + p.z;
    o.w = (e[j].w - mu2) * rstd2 * gm.w + bt.w + p.w;
    for (int bb = b; bb < Bout; bb += Bx) reinterpret_cast<float4*>(out + ((size_t)bb * N + n) * D)[lane + 32 * j] = o;
  }
}

// embed_dim = 64 x odd: the same computation with scalar lanes (column c = lane + 32 j); inference only (no EmbedSave)
__global__ void __launch_bounds__(256) embed_generic_kernel(const float* __restrict__ x, int Bx, int Bout, int C, int img,
                                                            int patch, int D, EmbedW w, float* __restrict__ out) {
  __shared__ float s_t[8][64];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = img / patch, N = g * g, pd = C * patch * patch;
  const long long tok = (long long)blockIdx.x * 8 + wib;
  if (tok >= (long long)Bout * N) return;
  const int b = int(tok / N), n = int(tok % N);
  const int gy = n / g, gx = n % g;
  const float* xb = x + (size_t)(b % Bx) * C * img * img;
  float* t = s_t[wib];
  for (int i = lane; i < pd; i += 32) {
    const int c = i / (patch * patch), p1 = (i / patch) % patch, p2 = i % patch;
    t[i] = xb[(size_t)c * img * img + (size_t)(gy * patch + p1) * img + gx * patch + p2];
  }
  __syncwarp();
  float conv[2] = {0.f, 0.f};
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int o = lane + 32 * r;
    if (o < pd) {
      float acc = w.conv_b[o];
      for (int i = 0; i < pd; ++i) acc += w.conv_w[o * pd + i] * t[i];
      conv[r] = acc;
      s += acc;
    }
  }
  const float mu1 = warp_sum(s) / pd;
  float q = 0.f;
#pragma unroll
  for (int r = 0; r < 2; ++r)
    if (lane + 32 * r < pd) q += (conv[r] - mu1) * (conv[r] - mu1);
  const float rstd1 = rsqrtf(warp_sum(q) / pd + LN_EPS);
  __syncwarp();
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int o = lane + 32 * r;
    if (o < pd) t[o] = (conv[r] - mu1) * rstd1 * w.ln1_w[o] + w.ln1_b[o];
  }
  __syncwarp();
  const int nj = D / 32;   // <= 32
  float e[32];
  float s2 = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    e[j] = 0.f;
    if (j < nj) {
      const int c = lane + 32 * j;
      float acc = __ldg(w.lin_b + c);
      for (int i = 0; i < pd; ++i) acc += __ldg(w.lin_wT + (size_t)i * D + c) * t[i];
      e[j] = acc;
      s2 += acc;
    }
  }
  const float mu2 = warp_sum(s2) / D;
  float q2 = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j)
    if (j < nj) q2 += (e[j] - mu2) * (e[j] - mu2);
  const float rstd2 = rsqrtf(warp_sum(q2) / D + LN_EPS);
#pragma unroll
  for (int j = 0; j < 32; ++j)
    if (j < nj) {
      const int c = lane + 32 * j;
      out[(size_t)tok * D + c] = (e[j] - mu2) * rstd2 * __ldg(w.ln2_w + c) + __ldg(w.ln2_b + c) + __ldg(w.pos + (size_t)n * D + c);
    }
}

int launch_embed(const float* x, int Bx, int Bout, int C, int img, int patch, int D, const EmbedW& w, float* out,
                 cudaStream_t st, const EmbedSave* svp) {
  const EmbedSave sv = svp ? *svp : EmbedSave{nullptr, nullptr, nullptr, nullptr};
  TLD_CHECK(D % 64 == 0 && D >= 64 && D <= 1024, "embed: embed_dim must be a multiple of 64 in [64,1024]");
  if (D % 128 != 0) {
    TLD_CHECK(svp == nullptr, "embed: the training path needs embed_dim % 128 == 0");
    TLD_CHECK(C * patch * patch <= 64 && img % patch == 0, "embed: bad patch geometry");
    const long long toks_g = (long long)Bout * (img / patch) * (img / patch);
    embed_generic_kernel<<<int((toks_g + 7) / 8), 256, 0, st>>>(x, Bx, Bout, C, img, patch, D, w, out);
    TLD_CUDA_OK(cudaGetLastError());
    return 0;
  }
  TLD_CHECK(C * patch * patch <= 64, "embed: patch_dim (n_channels*patch^2) must be <= 64");
  TLD_CHECK(img % patch == 0, "embed: image_size must be divisible by patch_size");
  TLD_CHECK(Bx > 0 && Bout % Bx == 0, "embed: the output batch must be a whole number of copies of the input batch");
  TLD_CHECK(svp == nullptr || Bx == Bout, "embed: the training path embeds every image once");
  const long long toks = (long long)Bx * (img / patch) * (img / patch);
  const int grid = int((toks + 7) / 8);
  switch (D / 128) {
#define EM_CASE(V) \
  case V: if (launch_pdl(embed_kernel<V>, dim3(grid), dim3(256), 0, st, x, Bx, Bout, C, img, patch, w, out, sv)) return 1; break;
    EM_CASE(1) EM_CASE(2) EM_CASE(3) EM_CASE(4) EM_CASE(5) EM_CASE(6) EM_CASE(7) EM_CASE(8)
#undef EM_CASE
  }
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}

// --------------------------------------------------------------------------------------------
// Conditioning tokens (denoiser.py:117-122, transformer_blocks.py:17-21).  The sinusoid and both MLP layers are fp32
// on purpose (SURVEY.md §0: bf16 sin(6283 t) is garbage).  All R rows go through each layer together: a 16x16-tiled
// fp32 dense kernel reads every weight once per 16 rows (the first version ran one CTA per row and re-streamed the
// 3 MB of MLP weights R times: 0.5 ms for 128 rows), then one CTA per row does the LayerNorm -> bf16.
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cond_sincos_kernel(const float* __restrict__ t, const float* __restrict__ speeds,
                                                          float* __restrict__ emb, int R, int E) {
  const int i = blockIdx.x * 256 + threadIdx.x, half = E / 2;
  if (i >= R * half) return;
  const int r = i / half, j = i % half;
  const float a = speeds[j] * t[r];  // fp32 product, as the reference's fp32 path
  emb[(size_t)r * E + j] = sinf(a);
  emb[(size_t)r * E + half + j] = cosf(a);
}

// out[r, o] = act(bias[o] + sum_i in[r, i] W[o, i]);  in == nullptr or r >= R_real: zero input row.  pre (optional) keeps the
// value before the activation.  16 rows x 16 outputs per CTA, K walked in 16-wide smem tiles.
__global__ void __launch_bounds__(256) cond_dense_kernel(const float* __restrict__ in, int R, int R_real,
                                                         const float* __restrict__ W, const float* __restrict__ bias,
                                                         float* __restrict__ out, float* __restrict__ pre, int n_out,
                                                         int n_in, int gelu) {
  __shared__ float sA[16][17], sW[16][17];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int r = blockIdx.y * 16 + ty, o = blockIdx.x * 16 + tx;
  const int rl = blockIdx.y * 16 + ty, ol = blockIdx.x * 16 + ty;   // rows of the two tiles this thread loads
  float acc = 0.f;
  for (int k0 = 0; k0 < n_in; k0 += 16) {
    const int k = k0 + tx;
    sA[ty][tx] = (in != nullptr && rl < R_real && k < n_in) ? in[(size_t)rl * n_in + k] : 0.f;
    sW[ty][tx] = (ol < n_out && k < n_in) ? __ldg(W + (size_t)ol * n_in + k) : 0.f;
    __syncthreads();
#pragma unroll
    for (int q = 0; q < 16; ++q) acc = fmaf(sA[ty][q], sW[tx][q], acc);
    __syncthreads();
  }
  if (r < R && o < n_out) {
    acc += bias[o];
    if (pre) pre[(size_t)r * n_out + o] = acc;
    out[(size_t)r * n_out + o] = gelu ? gelu_erf(acc) : acc;
  }
}

__device__ void block_layernorm_store(const float* __restrict__ v, const float* __restrict__ gw,
                                      const float* __restrict__ gb, bf16* __restrict__ y, int D, float* red) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float s = 0.f;
  for (int i = threadIdx.x; i < D; i += blockDim.x) s += v[i];
  s = warp_sum(s);
  if (lane == 0) red[wib] = s;
  __syncthreads();
  float tot = 0.f;
  for (int i = 0; i < nw; ++i) tot += red[i];
  const float mu = tot / D;
  __syncthreads();
  float q = 0.f;
  for (int i = threadIdx.x; i < D; i += blockDim.x) q += (v[i] - mu) * (v[i] - mu);
  q = warp_sum(q);
  if (lane == 0) red[wib] = q;
  __syncthreads();
  tot = 0.f;
  for (int i = 0; i < nw; ++i) tot += red[i];
  const float rstd = rsqrtf(tot / D + LN_EPS);
  for (int i = threadIdx.x; i < D; i += blockDim.x) y[i] = __float2bfloat16((v[i] - mu) * rstd * gw[i] + gb[i]);
}

__global__ void __launch_bounds__(256) cond_ln_kernel(const float* __restrict__ pre, const float* __restrict__ gw,
                                                      const float* __restrict__ gb, bf16* __restrict__ y, int D) {
  __shared__ float red[8];
  const int r = blockIdx.x;
  block_layernorm_store(pre + (size_t)r * D, gw, gb, y + (size_t)r * D, D, red);
}

int launch_cond_noise(const float* t, int R, int E, int D, const CondW& w, bf16* y, float* scratch, cudaStream_t st,
                      const CondSave* sv) {
  if (R <= 0) return 0;
  TLD_CHECK(scratch != nullptr || (sv && sv->emb && sv->a1 && sv->h1 && sv->pre), "cond_noise: no scratch buffer");
  float* emb = (sv && sv->emb) ? sv->emb : scratch;
  float* h1 = (sv && sv->h1) ? sv->h1 : scratch + (size_t)R * E;
  float* pre = (sv && sv->pre) ? sv->pre : scratch + (size_t)R * (E + D);
  cond_sincos_kernel<<<(R * (E / 2) + 255) / 256, 256, 0, st>>>(t, w.speeds, emb, R, E);
  const dim3 grid((D + 15) / 16, (R + 15) / 16);
  cond_dense_kernel<<<grid, 256, 0, st>>>(emb, R, R, w.w1, w.b1, h1, sv ? sv->a1 : nullptr, D, E, 1);
  cond_dense_kernel<<<grid, 256, 0, st>>>(h1, R, R, w.w2, w.b2, pre, nullptr, D, D, 0);
  cond_ln_kernel<<<R, 256, 0, st>>>(pre, w.ln_w, w.ln_b, y, D);
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_cond_label(const float* label, int R, int R_real, int Te, int D, const CondW& w, bf16* y, float* scratch,
                      cudaStream_t st, float* pre_save) {
  if (R <= 0) return 0;
  TLD_CHECK(scratch != nullptr || pre_save != nullptr, "cond_label: no scratch buffer");
  float* pre = pre_save ? pre_save : scratch;
  const dim3 grid((D + 15) / 16, (R + 15) / 16);
  cond_dense_kernel<<<grid, 256, 0, st>>>(label, R, label ? R_real : 0, w.wl, w.bl, pre, nullptr, D, Te, 0);
  cond_ln_kernel<<<R, 256, 0, st>>>(pre, w.ln_w, w.ln_b, y, D);
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}

// --------------------------------------------------------------------------------------------
// Depthwise 3x3 ('same', zero pad) + bias + exact GELU over the token grid (transformer_blocks.py:96-103).
// Layout: h, g bf16 [B, grid, grid, C] (token-major == NHWC).  One thread owns 4 channels of one grid row and
// slides along x with a 3x3 fp32 register window (each loaded value is unpacked once): 3 new 8-byte loads per
// 4 outputs; the 36 weights stay in registers.  The kernel is ALU-bound (9 FMA + GELU per element at
// 100 M elements per layer), so erf uses Abramowitz-Stegun 7.1.26 (|err| <= 1.5e-7, far below the bf16
// rounding of the output) on the MUFU ex2/rcp units instead of the ~25-instruction libdevice erff.
// --------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_fast_erf(float v) {
  const float z = fabsf(v) * 0.70710678118654752f;
  const float t = __fdividef(1.0f, fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(1.061405429f, t, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  const float e = __expf(-z * z);
  const float erf_abs = fmaf(-p * t, e, 1.0f);  // erf(|v|/sqrt2)
  const float hv = 0.5f * v;
  return fmaf(hv, copysignf(erf_abs, v), hv);
}

__device__ __forceinline__ void unpack4(const uint2& v, float (&f)[4]) {
  f[0] = __uint_as_float(v.x << 16);
  f[1] = __uint_as_float(v.x & 0xffff0000u);
  f[2] = __uint_as_float(v.y << 16);
  f[3] = __uint_as_float(v.y & 0xffff0000u);
}

__global__ void __launch_bounds__(256) dwconv_gelu_generic_kernel(const bf16* __restrict__ h, const float* __restrict__ w9,
                                                          const float* __restrict__ bias, bf16* __restrict__ g, int B,
                                                          int grid, int C) {
  const int c4n = C / 4;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)B * grid * c4n) return;
  const int c4 = int(idx % c4n);
  const int gy = int((idx / c4n) % grid);
  const int b = int(idx / ((long long)c4n * grid));
  const int c0 = c4 * 4;
  float w[9][4], bs[4];
#pragma unroll
  for (int tp = 0; tp < 9; ++tp) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(w9 + (size_t)tp * C + c0));
    w[tp][0] = a.x; w[tp][1] = a.y; w[tp][2] = a.z; w[tp][3] = a.w;
  }
  {
    const float4 a = __ldg(reinterpret_cast<const float4*>(bias + c0));
    bs[0] = a.x; bs[1] = a.y; bs[2] = a.z; bs[3] = a.w;
  }
  const size_t img_base = (size_t)b * grid * grid * C + c0;
  const bool up = gy > 0, dn = gy + 1 < grid;
  // col[k][dy][ch]: three window columns in rotating roles
  float col[3][3][4];
  auto load_col = [&](float (&dst)[3][4], int xx) {
    const bool okx = xx >= 0 && xx < grid;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
      const bool ok = okx && (dy == 1 || (dy == 0 ? up : dn));
      uint2 v = make_uint2(0u, 0u);
      if (ok) v = *reinterpret_cast<const uint2*>(h + img_base + ((size_t)(gy + dy - 1) * grid + xx) * C);
      unpack4(v, dst[dy]);
    }
  };
#pragma unroll
  for (int dy = 0; dy < 3; ++dy)
#pragma unroll
    for (int j = 0; j < 4; ++j) col[0][dy][j] = 0.f;
  load_col(col[1], 0);
  load_col(col[2], 1);
  for (int x0 = 0; x0 < grid; x0 += 3) {
#pragma unroll
    for (int u = 0; u < 3; ++u) {
      const int xq = x0 + u;
      if (xq < grid) {
        // window columns: left = col[u%3], centre = col[(u+1)%3], right = col[(u+2)%3]
        float acc[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j] = bs[j];
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
          for (int dx = 0; dx < 3; ++dx)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[j] = fmaf(w[dy * 3 + dx][j], col[(u + dx) % 3][dy][j], acc[j]);
        uint2 o;
        o.x = pack_bf16x2_dev(gelu_fast_erf(acc[0]), gelu_fast_erf(acc[1]));
        o.y = pack_bf16x2_dev(gelu_fast_erf(acc[2]), gelu_fast_erf(acc[3]));
        *reinterpret_cast<uint2*>(g + img_base + ((size_t)gy * grid + xq) * C) = o;
        load_col(col[u % 3], xq + 2);  // the old left column becomes the next right column
      }
    }
  }
}

// d/dv gelu(v) = Phi(v) + v phi(v) on a channel pair (training backward): Phi through the same erf polynomial,
// phi(v) = exp(-v^2/2) / sqrt(2 pi) on MUFU.EX2
__device__ __forceinline__ float2 dgelu2(float2 v) {
  const float2 vc = make_float2(fminf(fmaxf(v.x, -3.96f), 3.96f), fminf(fmaxf(v.y, -3.96f), 3.96f));
  const float2 u = fmul2(vc, vc);
  float2 r = ffma2(make_float2(-3.3440241686832906e-09f, -3.3440241686832906e-09f), u,
                   make_float2(2.5340079901070567e-07f, 2.5340079901070567e-07f));
  r = ffma2(r, u, make_float2(-8.418431207246613e-06f, -8.418431207246613e-06f));
  r = ffma2(r, u, make_float2(0.00016371029778383672f, 0.00016371029778383672f));
  r = ffma2(r, u, make_float2(-0.002110206289216876f, -0.002110206289216876f));
  r = ffma2(r, u, make_float2(0.019370341673493385f, 0.019370341673493385f));
  r = ffma2(r, u, make_float2(-0.13240252435207367f, -0.13240252435207367f));
  r = ffma2(r, u, make_float2(0.7977136969566345f, 0.7977136969566345f));
  const float2 cdf = ffma2(fmul2(vc, r), make_float2(0.5f, 0.5f), make_float2(0.5f, 0.5f));
  const float2 arg = fmul2(v, fmul2(v, make_float2(-0.72134752044448170f, -0.72134752044448170f)));
  const float2 pdf = make_float2(ex2_approx(arg.x) * 0.3989422804014327f, ex2_approx(arg.y) * 0.3989422804014327f);
  return ffma2(v, pdf, cdf);
}

// Specialised kernel for a compile-time token grid G (8/16/32/64): one thread = 4 channels (two FFMA2 pairs) of one
// grid row, sliding along x.  y-borders: row index clamped + that tap row's weights zeroed (branch-free);
// x-borders: zero columns.  Loads run 4 columns ahead of their use through a 6-deep raw-register ring.
template <int G>
__global__ void __launch_bounds__(256) dwconv_gelu_grid_kernel(const bf16* __restrict__ h, const float* __restrict__ w9,
                                                               const float* __restrict__ bias, bf16* __restrict__ g,
                                                               int B, int C) {
  const int c4n = C >> 2;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * G * c4n) return;
  const int c4 = idx % c4n;
  const int rowid = idx / c4n;       // b * G + gy
  const int gy = rowid % G;
  const int c0 = c4 * 4;
  const bool up = gy > 0, dn = gy + 1 < G;
  float2 w[9][2];
#pragma unroll
  for (int tp = 0; tp < 9; ++tp) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(w9 + (size_t)tp * C + c0));
    const bool live = (tp / 3 == 1) || (tp / 3 == 0 ? up : dn);
    w[tp][0] = live ? make_float2(a.x, a.y) : make_float2(0.f, 0.f);
    w[tp][1] = live ? make_float2(a.z, a.w) : make_float2(0.f, 0.f);
  }
  const float4 bq = __ldg(reinterpret_cast<const float4*>(bias + c0));
  const float2 b0 = make_float2(bq.x, bq.y), b1 = make_float2(bq.z, bq.w);
  const size_t rowC = (size_t)G * C;
  const bf16* r1 = h + (size_t)rowid * rowC + c0;
  const bf16* r0 = up ? r1 - rowC : r1;   // clamped rows: their weights are zero when out of range
  const bf16* r2 = dn ? r1 + rowC : r1;
  bf16* orow = g + (size_t)rowid * rowC + c0;

  uint2 ring[6][3];       // raw columns, ring[c % 6]
  float2 win[3][3][2];    // unpacked columns win[c % 3][dy][pair]
  auto fetch = [&](uint2 (&dst)[3], int colx) {
    if (colx < G) {
      const size_t o = (size_t)colx * C;
      dst[0] = *reinterpret_cast<const uint2*>(r0 + o);
      dst[1] = *reinterpret_cast<const uint2*>(r1 + o);
      dst[2] = *reinterpret_cast<const uint2*>(r2 + o);
    } else {
      dst[0] = dst[1] = dst[2] = make_uint2(0u, 0u);
    }
  };
  auto unpack = [&](float2 (&dst)[3][2], const uint2 (&src)[3]) {
#pragma unroll
    for (int dy = 0; dy < 3; ++dy) {
      dst[dy][0] = unpack_bf16x2(src[dy].x);
      dst[dy][1] = unpack_bf16x2(src[dy].y);
    }
  };
#pragma unroll
  for (int c = 0; c < 6; ++c) fetch(ring[c], c);
#pragma unroll
  for (int dy = 0; dy < 3; ++dy) win[2][dy][0] = win[2][dy][1] = make_float2(0.f, 0.f);  // column -1
  unpack(win[0], ring[0]);
  unpack(win[1], ring[1]);

  constexpr int U = (G % 12 == 0) ? 12 : (G <= 16 ? G : 12);
#pragma unroll 1
  for (int x0 = 0; x0 < G; x0 += U) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int xq = x0 + u;
      if (G % U == 0 || xq < G) {
        // x0 is a multiple of U (itself a multiple of 6 unless the loop runs once), so u stands in for xq in the
        // compile-time ring/window indices
        float2 a0 = b0, a1 = b1;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            a0 = ffma2(w[dy * 3 + dx][0], win[(u + dx + 2) % 3][dy][0], a0);
            a1 = ffma2(w[dy * 3 + dx][1], win[(u + dx + 2) % 3][dy][1], a1);
          }
        const float2 g0 = gelu2(a0), g1 = gelu2(a1);
        uint2 o;
        o.x = pack_bf16x2_dev(g0.x, g0.y);
        o.y = pack_bf16x2_dev(g1.x, g1.y);
        *reinterpret_cast<uint2*>(orow + (size_t)xq * C) = o;
        unpack(win[(u + 2) % 3], ring[(u + 2) % 6]);   // column xq+2 replaces column xq-1
        fetch(ring[u % 6], xq + 6);                    // column xq+6 reuses the slot of column xq
      }
    }
  }
}

// 16x16 token grid (256-px latents), shared-memory version: one CTA = one image x 64 channels.  The whole
// [256 positions x 64 ch] bf16 slab (32 KB) arrives with ONE TMA load (128B swizzle); lane = channel pair, so every
// warp-wide LDS reads one full 128-byte row (conflict-free); warp w produces grid rows 2w and 2w+1 sliding along x
// with a 4-row x 3-column fp32 window.  All shared-memory offsets are compile-time constants after unrolling.
// MODE 0: g = gelu(conv(h) + b)                         (forward)
// MODE 1: out = second * gelu'(conv(h) + b)              (backward A: du = dg * gelu'(u), u recomputed)
// MODE 2: out = conv^T(in): flipped taps, no bias        (backward B: dh = dwconv^T(du))
// MODE 3: tap / bias gradients of this image:  partial[b][tap][c] = sum_{y,x} du[y,x,c] h[y+dy-1, x+dx-1, c],
//         partial[b][9][c] = sum du   (tile = h, second = du, g reinterpreted as the fp32 partial buffer [B][10][C])
template <int MODE>
__global__ void __launch_bounds__(256) dwconv_gelu_g16_kernel(const __grid_constant__ CUtensorMap tmap_h,
                                                              const float* __restrict__ w9,
                                                              const float* __restrict__ bias, bf16* __restrict__ g,
                                                              int C, const bf16* __restrict__ second) {
  constexpr int G = 16;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* tile = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar = reinterpret_cast<uint64_t*>(tile + G * G * 128);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c0 = blockIdx.x * 64, b = blockIdx.y;
  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
    pdl_wait();  // h is the previous kernel's output
    mbar_expect_tx(bar, G * G * 128);
    tma_load_2d(tile, &tmap_h, bar, c0, b * G * G);
  }
  // weights / bias of this lane's channel pair while the tile is in flight
  const int ch = c0 + 2 * lane;
  float2 w[9];
#pragma unroll
  for (int tp = 0; tp < 9; ++tp)
    w[tp] = MODE == 3 ? make_float2(0.f, 0.f)
                      : __ldg(reinterpret_cast<const float2*>(w9 + (size_t)(MODE == 2 ? 8 - tp : tp) * C + ch));
  const float2 bs = MODE >= 2 ? make_float2(0.f, 0.f) : __ldg(reinterpret_cast<const float2*>(bias + ch));
  __syncthreads();  // barrier init visible before anyone polls it
  pdl_wait();       // every thread: the output buffer may still be read by an earlier kernel
  mbar_wait(bar, 0);

  const int y0 = 2 * warp;  // output rows y0, y0+1; input rows y0-1 .. y0+2
  const bool up = y0 > 0, dn = y0 + 2 < G;
  // byte offset of (row rr of the 4-row window, column x) for this lane: p = y*16 + x, p & 7 == x & 7
  const uint32_t rows = smem_u32(tile) + (y0 - 1) * G * 128;  // shared-window address (may point one row above)
  const int lane_chunk = lane >> 2, lane_off = (lane & 3) * 4;
  auto ldcol = [&](float2 (&dst)[4], int x) {
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const bool ok = (rr == 1 || rr == 2) || (rr == 0 ? up : dn);
      uint32_t v = 0u;
      if (ok) {
        const uint32_t addr = rows + (rr * G + x) * 128 + ((lane_chunk ^ (x & 7)) << 4) + lane_off;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
      }
      dst[rr] = unpack_bf16x2(v);
    }
  };
  float2 win[3][4];
#pragma unroll
  for (int rr = 0; rr < 4; ++rr) win[2][rr] = make_float2(0.f, 0.f);  // column -1
  ldcol(win[0], 0);
  ldcol(win[1], 1);
  bf16* out = g + ((size_t)b * G * G + (size_t)y0 * G) * C + ch;
  if constexpr (MODE == 3) {
    // weight-gradient mode: the same sliding window, but the products are accumulated per tap instead of per position
    const bf16* du = second + ((size_t)b * G * G + (size_t)y0 * G) * C + ch;
    float2 acc[9], accb = make_float2(0.f, 0.f);
#pragma unroll
    for (int t = 0; t < 9; ++t) acc[t] = make_float2(0.f, 0.f);
#pragma unroll
    for (int x = 0; x < G; ++x) {
      const float2 d0 = unpack_bf16x2(__ldg(reinterpret_cast<const uint32_t*>(du + (size_t)x * C)));
      const float2 d1 = unpack_bf16x2(__ldg(reinterpret_cast<const uint32_t*>(du + (size_t)(G + x) * C)));
      accb = fadd2(accb, fadd2(d0, d1));
#pragma unroll
      for (int dy = 0; dy < 3; ++dy)
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          acc[dy * 3 + dx] = ffma2(d0, win[(x + dx + 2) % 3][dy], acc[dy * 3 + dx]);
          acc[dy * 3 + dx] = ffma2(d1, win[(x + dx + 2) % 3][dy + 1], acc[dy * 3 + dx]);
        }
      if (x + 2 < G) {
        ldcol(win[(x + 2) % 3], x + 2);
      } else {
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) win[(x + 2) % 3][rr] = make_float2(0.f, 0.f);
      }
    }
    // the 8 warps (row pairs) of the CTA -> one [10][64] block of this image's partial sums (fixed order: deterministic)
    float* red = reinterpret_cast<float*>(tile + G * G * 128 + 64);   // [8][10][64] fp32 behind the tile and its barrier
#pragma unroll
    for (int t = 0; t < 9; ++t) *reinterpret_cast<float2*>(red + (warp * 10 + t) * 64 + 2 * lane) = acc[t];
    *reinterpret_cast<float2*>(red + (warp * 10 + 9) * 64 + 2 * lane) = accb;
    __syncthreads();
    float* partial = reinterpret_cast<float*>(g);
    for (int i = threadIdx.x; i < 10 * 64; i += 256) {
      float t = 0.f;
#pragma unroll
      for (int wq = 0; wq < 8; ++wq) t += red[wq * 640 + i];
      partial[((size_t)b * 10 + i / 64) * C + c0 + (i & 63)] = t;
    }
    return;
  }
#pragma unroll
  for (int x = 0; x < G; ++x) {
    float2 a0 = bs, a1 = bs;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        a0 = ffma2(w[dy * 3 + dx], win[(x + dx + 2) % 3][dy], a0);
        a1 = ffma2(w[dy * 3 + dx], win[(x + dx + 2) % 3][dy + 1], a1);
      }
    float2 g0, g1;
    if constexpr (MODE == 0) {
      g0 = gelu2(a0);
      g1 = gelu2(a1);
    } else if constexpr (MODE == 1) {
      const bf16* sec = second + (out - g);
      const float2 d0 = unpack_bf16x2(__ldg(reinterpret_cast<const uint32_t*>(sec + (size_t)x * C)));
      const float2 d1 = unpack_bf16x2(__ldg(reinterpret_cast<const uint32_t*>(sec + (size_t)(G + x) * C)));
      g0 = fmul2(d0, dgelu2(a0));
      g1 = fmul2(d1, dgelu2(a1));
    } else {
      g0 = a0;
      g1 = a1;
    }
    *reinterpret_cast<uint32_t*>(out + (size_t)x * C) = pack_bf16x2_dev(g0.x, g0.y);
    *reinterpret_cast<uint32_t*>(out + (size_t)(G + x) * C) = pack_bf16x2_dev(g1.x, g1.y);
    if (x + 2 < G) {
      ldcol(win[(x + 2) % 3], x + 2);
    } else {
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) win[(x + 2) % 3][rr] = make_float2(0.f, 0.f);
    }
  }
}

// Larger token grids (32x32: 512-px model, 64x64: 1024-px model): the same shared-memory scheme on ROW TILES.  One CTA =
// one image x 64 channels x RT output rows; the RT+2 input rows (one halo row above and below) arrive as TMA boxes of two
// grid rows each from a 3-D [image][position][channel] view, so rows outside the image are zero-filled by the TMA unit
// (= the conv's zero padding, no border flags).  A warp produces two output rows over a segment of G/XS columns, sliding
// along x with a 4-row x 3-column fp32 window; lane = channel pair (conflict-free 128-byte LDS rows, FFMA2 arithmetic).
template <int G, int RT, int XS>
__global__ void __launch_bounds__(32 * (RT / 2) * XS) dwconv_gelu_rows_kernel(const __grid_constant__ CUtensorMap tmap_h,
                                                                            const float* __restrict__ w9,
                                                                            const float* __restrict__ bias,
                                                                            bf16* __restrict__ g, int C) {
  static_assert(RT % 2 == 0 && G % RT == 0 && G % XS == 0 && (2 * G) % 8 == 0 && 2 * G <= 256, "bad row tiling");
  constexpr int TROWS = RT + 2, XW = G / XS;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* tile = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bar = reinterpret_cast<uint64_t*>(tile + TROWS * G * 128);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c0 = blockIdx.x * 64;
  const int tiles_per_img = G / RT;
  const int b = blockIdx.y / tiles_per_img, ty0 = (blockIdx.y % tiles_per_img) * RT;   // first output row of this CTA
  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    fence_mbar_init();
    pdl_wait();  // h is the previous kernel's output
    mbar_expect_tx(bar, TROWS * G * 128);
#pragma unroll
    for (int r2 = 0; r2 < TROWS / 2; ++r2)   // box = two grid rows; the first starts one row above the tile (may be row -1)
      tma_load_3d(tile + r2 * 2 * G * 128, &tmap_h, bar, c0, (ty0 - 1 + 2 * r2) * G, b);
  }
  const int ch = c0 + 2 * lane;
  float2 w[9];
#pragma unroll
  for (int tp = 0; tp < 9; ++tp) w[tp] = __ldg(reinterpret_cast<const float2*>(w9 + (size_t)tp * C + ch));
  const float2 bs = __ldg(reinterpret_cast<const float2*>(bias + ch));
  __syncthreads();  // barrier init visible before anyone polls it
  pdl_wait();
  mbar_wait(bar, 0);

  const int wr = warp / XS, ws = warp % XS;      // row pair / column segment of this warp
  const int y0 = 2 * wr, x0 = ws * XW;           // output rows ty0+y0, ty0+y0+1 = tile rows y0+1, y0+2; inputs y0 .. y0+3
  const uint32_t rows = smem_u32(tile) + y0 * G * 128;
  const int lane_chunk = lane >> 2, lane_off = (lane & 3) * 4;
  auto ldcol = [&](float2 (&dst)[4], int x) {
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int tp = rr * G + x;   // (y0 * G) is a multiple of 8, so the swizzle phase of the row is tp & 7 == x & 7
      uint32_t v;
      asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(rows + tp * 128 + ((lane_chunk ^ (x & 7)) << 4) + lane_off));
      dst[rr] = unpack_bf16x2(v);
    }
  };
  float2 win[3][4];
  // window columns x0-1, x0, x0+1 in slots 2, 0, 1 (slot of column x = (x - x0) mod 3, column x0-1 takes slot 2)
  if (x0 > 0) {
    ldcol(win[2], x0 - 1);
  } else {
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) win[2][rr] = make_float2(0.f, 0.f);
  }
  ldcol(win[0], x0);
  ldcol(win[1], x0 + 1);
  bf16* out = g + ((size_t)b * G * G + (size_t)(ty0 + y0) * G + x0) * C + ch;
#pragma unroll
  for (int xi = 0; xi < XW; ++xi) {
    float2 a0 = bs, a1 = bs;
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        a0 = ffma2(w[dy * 3 + dx], win[(xi + dx + 2) % 3][dy], a0);
        a1 = ffma2(w[dy * 3 + dx], win[(xi + dx + 2) % 3][dy + 1], a1);
      }
    const float2 g0 = gelu2(a0), g1 = gelu2(a1);
    *reinterpret_cast<uint32_t*>(out + (size_t)xi * C) = pack_bf16x2_dev(g0.x, g0.y);
    *reinterpret_cast<uint32_t*>(out + (size_t)(G + xi) * C) = pack_bf16x2_dev(g1.x, g1.y);
    if (x0 + xi + 2 < G) {
      ldcol(win[(xi + 2) % 3], x0 + xi + 2);
    } else {
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) win[(xi + 2) % 3][rr] = make_float2(0.f, 0.f);
    }
  }
}

template <int G, int RT, int XS>
static int launch_dwconv_rows(const bf16* h, const float* w9, const float* bias, bf16* g, int B, int C, cudaStream_t st) {
  constexpr int smem = 1024 + (RT + 2) * G * 128 + 64;
  auto kern = dwconv_gelu_rows_kernel<G, RT, XS>;
  static bool attr_set = false;
  if (!attr_set) {
    TLD_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set = true;
  }
  CUtensorMap th;
  if (make_tmap_tokens3d(&th, h, B, G * G, C, 2 * G)) return 1;
  return launch_pdl(kern, dim3(C / 64, B * (G / RT)), dim3(32 * (RT / 2) * XS), smem, st, th, w9, bias, g, C);
}

int launch_dwconv_gelu(const bf16* h, const float* w9, const float* bias, bf16* g, int B, int grid, int C,
                       cudaStream_t st) {
  TLD_CHECK(C % 4 == 0, "dwconv: channel count must be a multiple of 4");
  TLD_CHECK(grid >= 2, "dwconv: token grid must be at least 2x2");
  const long long threads = (long long)B * grid * (C / 4);
  TLD_CHECK(threads < (1LL << 31), "dwconv: problem too large for 32-bit thread indexing");
  const int blocks = int((threads + 255) / 256);
  if (grid == 16 && C % 64 == 0 && B <= 65535) {
    constexpr int smem = 1024 + 16 * 16 * 128 + 64;
    CUtensorMap th;
    if (make_tmap_2d(&th, h, false, (long long)B * 256, C, C, 256)) return 1;
    return launch_pdl(dwconv_gelu_g16_kernel<0>, dim3(C / 64, B), dim3(256), smem, st, th, w9, bias, g, C,
                      (const bf16*)nullptr);
  }
  if (C % 64 == 0 && (long long)B * grid <= 65535) {
    if (grid == 32) return launch_dwconv_rows<32, 16, 1>(h, w9, bias, g, B, C, st);   // 18 rows x 32 = 72 KB, 8 warps
    if (grid == 64) return launch_dwconv_rows<64, 8, 2>(h, w9, bias, g, B, C, st);    // 10 rows x 64 = 80 KB, 8 warps
  }
  switch (grid) {
    case 8: dwconv_gelu_grid_kernel<8><<<blocks, 256, 0, st>>>(h, w9, bias, g, B, C); break;
    case 16: dwconv_gelu_grid_kernel<16><<<blocks, 256, 0, st>>>(h, w9, bias, g, B, C); break;
    case 32: dwconv_gelu_grid_kernel<32><<<blocks, 256, 0, st>>>(h, w9, bias, g, B, C); break;
    case 64: dwconv_gelu_grid_kernel<64><<<blocks, 256, 0, st>>>(h, w9, bias, g, B, C); break;
    default: dwconv_gelu_generic_kernel<<<blocks, 256, 0, st>>>(h, w9, bias, g, B, grid, C);
  }
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}

// backward passes A and B of the MLP middle on the 16x16 grid (same tile kernel, other point-wise tail)
int launch_dwconv_g16_bwd(const bf16* in, const bf16* second, const float* w9, const float* bias, bf16* out, int B, int C,
                          int mode, cudaStream_t st) {
  TLD_CHECK(C % 64 == 0 && B <= 65535 && mode >= 1 && mode <= 3, "dwconv_g16_bwd: bad arguments");
  constexpr int smem = 1024 + 16 * 16 * 128 + 64;
  CUtensorMap th;
  if (make_tmap_2d(&th, in, false, (long long)B * 256, C, C, 256)) return 1;
  if (mode == 3) {  // out = fp32 partial sums [B][10][C]; extra [8][10][64] fp32 reduction buffer behind the tile
    constexpr int smem3 = smem + 8 * 10 * 64 * 4;
    static bool attr_set = false;
    if (!attr_set) {
      TLD_CUDA_OK(cudaFuncSetAttribute(dwconv_gelu_g16_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem3));
      attr_set = true;
    }
    return launch_pdl(dwconv_gelu_g16_kernel<3>, dim3(C / 64, B), dim3(256), smem3, st, th, w9, bias, out, C, second);
  }
  if (mode == 1)
    return launch_pdl(dwconv_gelu_g16_kernel<1>, dim3(C / 64, B), dim3(256), smem, st, th, w9, bias, out, C, second);
  return launch_pdl(dwconv_gelu_g16_kernel<2>, dim3(C / 64, B), dim3(256), smem, st, th, w9, bias, out, C,
                    (const bf16*)nullptr);
}

// --------------------------------------------------------------------------------------------
// Output projection + unpatchify (denoiser.py:47-52,72,82): one warp per token.
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) outproj_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                      const float* __restrict__ bias, float* __restrict__ out, int B,
                                                      int C, int img, int patch, int D) {
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = img / patch, N = g * g, pd = C * patch * patch;
  const long long tok = (long long)blockIdx.x * 8 + wib;
  if (tok >= (long long)B * N) return;
  const int b = int(tok / N), n = int(tok % N), gy = n / g, gx = n % g;
  const float* xr = x + (size_t)tok * D;
  for (int o = 0; o < pd; ++o) {
    const float* wr = w + (size_t)o * D;
    float acc = 0.f;
    for (int i = lane * 4; i < D; i += 128) {
      const float4 xv = *reinterpret_cast<const float4*>(xr + i);
      const float4 wv = __ldg(reinterpret_cast<const float4*>(wr + i));
      acc += xv.x * wv.x + xv.y * wv.y + xv.z * wv.z + xv.w * wv.w;
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      const int c = o / (patch * patch), p1 = (o / patch) % patch, p2 = o % patch;
      out[((size_t)b * C + c) * img * img + (size_t)(gy * patch + p1) * img + gx * patch + p2] = acc + bias[o];
    }
  }
}

// Fast path for patch_dim 16 (4 channels x 2x2): the [16, D] weight lives in shared memory, a warp keeps FOUR token rows in
// registers (every weight element read from shared memory feeds 4 tokens: the one-token version was shared-memory bound,
// 96 LDS.128 per token) and loops over groups of tokens (persistent grid).  Four-row sums by a 6-shuffle transpose-reduce:
// afterwards the 8 lanes with (bit4, bit3) = r hold the sum of token r; lane (r, l) keeps outputs l and l + 8.
template <int V>
__global__ void __launch_bounds__(256) outproj16_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                        const float* __restrict__ bias, float* __restrict__ out,
                                                        long long T, int C, int img, int patch) {
  constexpr int D = V * 128;
  extern __shared__ __align__(16) float s_w[];  // [16][D]
  pdl_launch_dependents();
  for (int i = threadIdx.x; i < 16 * D / 4; i += 256) reinterpret_cast<float4*>(s_w)[i] = __ldg(reinterpret_cast<const float4*>(w) + i);
  __syncthreads();
  pdl_wait();
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = img / patch, N = g * g;
  const bool hi4 = lane & 16, hi3 = lane & 8;
  const int my_r = (hi4 ? 2 : 0) + (hi3 ? 1 : 0), l3 = lane & 7;
  const long long groups = (T + 3) / 4;
  for (long long grp = (long long)blockIdx.x * 8 + wib; grp < groups; grp += (long long)gridDim.x * 8) {
    float4 xv[4][V];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const long long tok = grp * 4 + r;
      const float4* xr = reinterpret_cast<const float4*>(x + (size_t)(tok < T ? tok : T - 1) * D);
#pragma unroll
      for (int j = 0; j < V; ++j) xv[r][j] = xr[lane + 32 * j];
    }
    float mine[2] = {0.f, 0.f};   // outputs l3 and l3 + 8 of token my_r
#pragma unroll
    for (int o = 0; o < 16; ++o) {
      float a[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < V; ++j) {
        const float4 wv = reinterpret_cast<const float4*>(s_w + o * D)[lane + 32 * j];
#pragma unroll
        for (int r = 0; r < 4; ++r) a[r] += xv[r][j].x * wv.x + xv[r][j].y * wv.y + xv[r][j].z * wv.z + xv[r][j].w * wv.w;
      }
      float k0 = hi4 ? a[2] : a[0], k1 = hi4 ? a[3] : a[1];
      k0 += __shfl_xor_sync(0xffffffffu, hi4 ? a[0] : a[2], 16);
      k1 += __shfl_xor_sync(0xffffffffu, hi4 ? a[1] : a[3], 16);
      float k = hi3 ? k1 : k0;
      k += __shfl_xor_sync(0xffffffffu, hi3 ? k0 : k1, 8);
      k += __shfl_xor_sync(0xffffffffu, k, 4);
      k += __shfl_xor_sync(0xffffffffu, k, 2);
      k += __shfl_xor_sync(0xffffffffu, k, 1);
      if ((o & 7) == l3) mine[o >> 3] = k;
    }
    const long long tok = grp * 4 + my_r;
    if (tok < T) {
      const int b = int(tok / N), n = int(tok % N), gy = n / g, gx = n % g;
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int o = l3 + 8 * u;
        const int c = o / (patch * patch), p1 = (o / patch) % patch, p2 = o % patch;
        out[((size_t)b * C + c) * img * img + (size_t)(gy * patch + p1) * img + gx * patch + p2] = mine[u] + bias[o];
      }
    }
  }
}

int launch_outproj(const float* x, const float* w, const float* b, float* out, int B, int C, int img, int patch,
                   int D, cudaStream_t st) {
  TLD_CHECK(D % 4 == 0, "outproj: embed_dim must be a multiple of 4");
  const long long toks = (long long)B * (img / patch) * (img / patch);
  if (C * patch * patch == 16 && D % 128 == 0 && D <= 768) {
    const int smem = 16 * D * 4;
    long long nb = (toks + 31) / 32;   // 8 warps x 4 tokens per CTA
    if (nb > (long long)sm_count()) nb = sm_count();   // 194 registers: one CTA per SM
    switch (D / 128) {
#define OP_CASE(V)                                                                                               \
  case V: {                                                                                                      \
    static bool set = false;                                                                                     \
    if (!set) {                                                                                                  \
      TLD_CUDA_OK(cudaFuncSetAttribute(outproj16_kernel<V>, cudaFuncAttributeMaxDynamicSharedMemorySize, 49152)); \
      set = true;                                                                                                \
    }                                                                                                            \
    if (launch_pdl(outproj16_kernel<V>, dim3((int)nb), dim3(256), smem, st, x, w, b, out, toks, C, img, patch)) return 1; \
  } break;
      OP_CASE(1) OP_CASE(2) OP_CASE(3) OP_CASE(4) OP_CASE(5) OP_CASE(6)
#undef OP_CASE
    }
    TLD_CUDA_OK(cudaGetLastError());
    return 0;
  }
  outproj_kernel<<<int((toks + 7) / 8), 256, 0, st>>>(x, w, b, out, B, C, img, patch, D);
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}

// --------------------------------------------------------------------------------------------
// CFG combine + DPM-Solver++(2M)/DDIM update (diffusion.py:66-89,122-125), coefficients from a device table.
// Separate rounded multiplies/adds (no FMA contraction) to follow the eager reference op by op.
// MASKED (masked edit): the kept region (mask 0) of x_t is reset to the known latent re-noised to the next level with the
// same eps after every update, and the final prediction keeps the known latent there; x0_prev keeps the unblended x0.
// --------------------------------------------------------------------------------------------
template <bool MASKED>
__global__ void __launch_bounds__(256) cfg_update_kernel(const float* __restrict__ mo, float* __restrict__ x_t,
                                                         float* __restrict__ x0_prev, float* __restrict__ x0_out,
                                                         const StepCoef* __restrict__ table,
                                                         const int* __restrict__ step_ptr, int B, int C, int hw,
                                                         const float* __restrict__ x0k, const float* __restrict__ eps,
                                                         const float* __restrict__ mask) {
  pdl_launch_dependents();
  pdl_wait();
  const StepCoef sc = table[*step_ptr];
  const long long n = (long long)B * C * hw;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float m = 1.f;
  if constexpr (MASKED) m = fminf(fmaxf(mask[(i / ((long long)C * hw)) * hw + i % hw], 0.f), 1.f);  // one value per pixel
  const float c = mo[i], u = mo[n + i];
  const float x0 = __fadd_rn(__fmul_rn(sc.guidance, c), __fmul_rn(sc.one_minus_g, u));
  if (sc.is_final) {
    const int ch = int((i / hw) % C);
    float v = x0;
    if (ch == 3) v = __fadd_rn(v, sc.sharp);
    if (ch == 0) v = __fadd_rn(v, sc.bright);
    if constexpr (MASKED) v = __fadd_rn(__fmul_rn(m, v), __fmul_rn(__fsub_rn(1.f, m), x0k[i]));
    x0_out[i] = v;
    return;
  }
  float d = x0;
  if (sc.c2 != 0.f) d = __fsub_rn(__fmul_rn(sc.c1, x0), __fmul_rn(sc.c2, x0_prev[i]));
  const float num = __fadd_rn(__fmul_rn(sc.dsig, d), __fmul_rn(sc.next, x_t[i]));
  float xn = __fdiv_rn(num, sc.cur);
  if constexpr (MASKED) {
    const float kept = __fadd_rn(__fmul_rn(sc.next, eps[i]), __fmul_rn(sc.one_minus_next, x0k[i]));
    xn = __fadd_rn(__fmul_rn(m, xn), __fmul_rn(__fsub_rn(1.f, m), kept));
  }
  x_t[i] = xn;
  x0_prev[i] = x0;
}

__global__ void edit_start_kernel(float* __restrict__ x_t, const float* __restrict__ eps, const float* __restrict__ x0k,
                                  float s0, float one_minus_s0, int from_noise, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  x_t[i] = from_noise ? eps[i] : __fadd_rn(__fmul_rn(s0, eps[i]), __fmul_rn(one_minus_s0, x0k[i]));
}

__global__ void advance_step_kernel(int* step_ptr) {
  pdl_launch_dependents();
  pdl_wait();
  *step_ptr += 1;
}

int launch_cfg_update(const float* model_out, float* x_t, float* x0_prev, float* x0_out, const StepCoef* table,
                      const int* step_ptr, int B, int C, int hw, cudaStream_t st, const float* x0k, const float* eps,
                      const float* mask) {
  const long long n = (long long)B * C * hw;
  if (mask)
    return launch_pdl(cfg_update_kernel<true>, dim3(int((n + 255) / 256)), dim3(256), 0, st, model_out, x_t, x0_prev, x0_out,
                      table, step_ptr, B, C, hw, x0k, eps, mask);
  return launch_pdl(cfg_update_kernel<false>, dim3(int((n + 255) / 256)), dim3(256), 0, st, model_out, x_t, x0_prev, x0_out,
                    table, step_ptr, B, C, hw, nullptr, nullptr, nullptr);
}
int launch_edit_start(float* x_t, const float* eps, const float* x0k, float s0, float one_minus_s0, int from_noise,
                      long long n, cudaStream_t st) {
  edit_start_kernel<<<int((n + 255) / 256), 256, 0, st>>>(x_t, eps, x0k, s0, one_minus_s0, from_noise, n);
  TLD_CUDA_OK(cudaGetLastError());
  return 0;
}
int launch_advance_step(int* step_ptr, cudaStream_t st) {
  return launch_pdl(advance_step_kernel, dim3(1), dim3(1), 0, st, step_ptr);
}

}  // namespace tld

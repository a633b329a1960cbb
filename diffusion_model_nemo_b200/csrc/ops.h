// ops.h -- host-side launch interface of the engine kernels (internal; the public ABI is include/dmn_b200.h).
//
// Engine data layout: activations are NHWC ("pixel-major": [batch][H*W][C]) in fp32 or bf16; GroupNorm
// statistics are {sum, sum-of-squares} per (sample, group) in fp32, accumulated by the producing kernel's
// epilogue and turned into mean/rstd by the consumer's prologue.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/dmn_b200.h"

namespace dmn {

typedef long long stat_t;   // fixed-point GroupNorm statistics (common.cuh)

enum { ACT_F32 = 0, ACT_BF16 = 1 };
enum { CONV_SAME = 0, CONV_DOWN = 1, CONV_UP = 2 };
enum { PRO_NONE = 0, PRO_GN = 1, PRO_SILU = 2, PRO_TEMB = 4, PRO_LRELU = 8 };   // PRO_LRELU: LeakyReLU(0.2), FiLM signal path (no GroupNorm)

// One convolution (+ fused prologue on its input, + fused epilogue on its output).
struct ConvP {
  // sources: channel-concatenation of src1 (C1 channels) and src2 (C2 channels, 0 = none); never materialised
  const void* src1 = nullptr;
  const void* src2 = nullptr;
  int C1 = 0, C2 = 0;
  int B = 0, Hin = 0, Win = 0, Hout = 0, Wout = 0, Cout = 0;
  int mode = CONV_SAME, ksize = 3;
  // weights: SIMT engine  -> fp32 [tap][Cin][Cout];  tcgen05 engine -> bf16 blocked (see conv_tcgen05.cu)
  const void* w = nullptr;
  const float* bias = nullptr;
  // prologue applied to src1 while loading (GroupNorm of the producer, SiLU, time-embedding add)
  int pro = PRO_NONE;
  const stat_t* pstats = nullptr;  // [B][pgroups][2]
  int pgroups = 0;
  const float* pgamma = nullptr;
  const float* pbeta = nullptr;
  const float* temb = nullptr;     // effective row = temb + (d_row ? *d_row * temb_rstride : 0) + b * temb_bstride
  long temb_bstride = 0, temb_rstride = 0;
  const int* d_row = nullptr;
  // GroupNorm(1) of the INPUT folded through a 1x1 conv (to_qkv): with W' = W * diag(gamma) packed as the weights,
  //   out[n] = rstd_b * (W' x)[n] - mean_b * rstd_b * s1[n] + s2[n],  s1[n] = sum_c W'[n][c],  s2[n] = sum_c W[n][c] * beta[c]
  // so the operand is loaded raw (no prologue) and the normalisation is an affine in the epilogue.  Uses pstats (pgroups == 1).
  const float* fold_s1 = nullptr;
  const float* fold_s2 = nullptr;
  // epilogue
  void* out = nullptr;             // raw conv output (+bias, +res)
  const void* res = nullptr;       // optional residual added to the output (same layout as out)
  stat_t* ostats = nullptr;        // [B][ogroups][2] accumulated with integer atomics (must be zeroed beforehand)
  int ogroups = 0;
};

int conv_simt(const ConvP& p, int act, cudaStream_t s);
int conv_tcgen05(const ConvP& p, cudaStream_t s);              // bf16 activations only
bool conv_tcgen05_supported(const ConvP& p);
// bytes of the blocked bf16 weight image for the tcgen05 engine, and the host-side packer
size_t conv_tcgen05_weight_bytes(int mode, int ksize, int cin, int cout);
void conv_tcgen05_pack_weights(int mode, int ksize, int cin, int cout, const float* w_torch, void* dst_host);
// SIMT packer: torch layout -> [tap][Cin][Cout] fp32 (optionally rounded to bf16 values)
void conv_simt_pack_weights(int mode, int ksize, int cin, int cout, const float* w_torch, float* dst_host, bool round_bf16);

// init_conv 7x7 pad 3 on the fp32 NCHW sampler state -> NHWC activations (+ class embedding)
struct InitConvP {
  const float* x = nullptr;        // [B][Cin][S][S]
  const float* w = nullptr;        // [49*Cin][Cout] fp32
  const float* bias = nullptr;
  const float* cls_w = nullptr;    // [num_classes+1][Cout] or null
  const int64_t* classes = nullptr;
  int pad_class = 0;               // row used when classes == null
  void* out = nullptr;
  int B = 0, Cin = 0, S = 0, Cout = 0;
};
int init_conv(const InitConvP& p, int act, cudaStream_t s);
// tensor-core stem (bf16 activations): w = blocked bf16 image from init_conv_tcgen05_pack_weights
int init_conv_tcgen05(const InitConvP& p, cudaStream_t s);
bool init_conv_tcgen05_supported(int Cin, int S, int Cout, int B);
size_t init_conv_tcgen05_weight_bytes(int cout);
void init_conv_tcgen05_pack_weights(int cin, int cout, const float* w_torch, void* dst_host);

// y = act(GroupNorm(raw)) [+ res];  optional statistics of y for the next norm
struct FinalizeP {
  const void* raw = nullptr;
  const stat_t* stats = nullptr;
  int groups = 0;
  const float* gamma = nullptr;
  const float* beta = nullptr;
  int silu = 0;
  const void* res = nullptr;
  void* out = nullptr;
  stat_t* ostats = nullptr;
  int ogroups = 0;
  int B = 0, HW = 0, C = 0;
};
int gn_finalize(const FinalizeP& p, int act, cudaStream_t s);

// final_conv tail: eps = conv1x1(SiLU(GroupNorm(y)))  -> fp32 NCHW
struct FinalProjP {
  const void* y = nullptr;
  const stat_t* stats = nullptr;
  int groups = 0;
  const float* gamma = nullptr;
  const float* beta = nullptr;
  const float* w = nullptr;        // [Cout][C] fp32
  const float* bias = nullptr;
  float* out = nullptr;            // [B][Cout][HW]
  int B = 0, HW = 0, C = 0, Cout = 0;
  int plain = 0;                   // 1: eps = conv1x1(y) only ('conv_bn_act' tail, unet.py:115-116); stats / gamma / beta unused
};
int final_proj(const FinalProjP& p, int act, cudaStream_t s);

int linattn_core(const void* qkv, void* out, int B, int heads, int dh, int N, int act, cudaStream_t s);
int attn_core(const void* qkv, void* out, int B, int heads, int dh, int N, int act, cudaStream_t s);
// bf16 tensor-core LinearAttention core (heads = 4, dim_head = 32); linattn_core dispatches to it for ACT_BF16
int linattn_core_bf16_mma(const void* qkv, void* out, int B, int N, cudaStream_t s);

// Residual(PreNorm(dim, LinearAttention(dim))) as one tcgen05 kernel (attn_fused.cu): out = GroupNorm(1)(to_out(attn(GN1(x)))) + x.
// bf16 NHWC activations; wqkv = row-major bf16 [384][C] with the PreNorm gamma folded in, wo = row-major bf16 [C][128];
// s1 / s2 = the fold vectors of ConvP (384 floats each); pstats = GroupNorm(1) statistics of x.
struct LinAttnFusedP {
  const void* x = nullptr;
  void* out = nullptr;
  const stat_t* pstats = nullptr;
  const void* wqkv = nullptr;
  const void* wo = nullptr;
  const float* s1 = nullptr;
  const float* s2 = nullptr;
  const float* bo = nullptr;       // to_out.0.bias [C]
  const float* go = nullptr;       // to_out.1.weight [C]
  const float* beo = nullptr;      // to_out.1.bias [C]
  int B = 0, N = 0, C = 0;
};
bool linattn_fused_supported(int B, int N, int C);
int linattn_fused(const LinAttnFusedP& p, cudaStream_t s);
// Residual(PreNorm(dim, Attention(dim))) (the bottleneck softmax attention, at most 64 tokens): same parameter block, go / beo unused
bool attn_softmax_fused_supported(int B, int N, int C);
int attn_softmax_fused(const LinAttnFusedP& p, cudaStream_t s);
// plumbing self-test of the TMA tensor copies + 128-byte-swizzle UMMA descriptors: D[M][N] = A[M][K] . B[N][K]^T (row-major bf16 in, fp32 out)
int selftest_tma_sw128_gemm(const void* a_bf16, const void* b_bf16, float* d, int M, int N, int K, cudaStream_t s);

// time path
struct TimeP {
  const float* times = nullptr;    // [rows]
  const float* freqs = nullptr;    // [dim/2]
  const float* w1t = nullptr;      // [dim][4dim]   (transposed Linear weights: [in][out])
  const float* b1 = nullptr;
  const float* w3t = nullptr;      // [4dim][4dim]
  const float* b3 = nullptr;
  const float* wct = nullptr;      // [4dim][sumC]  all ResnetBlock.mlp weights side by side
  const float* bc = nullptr;       // [sumC]
  float* tmp = nullptr;            // [rows][2*4dim] scratch
  float* table = nullptr;          // [rows][sumC]
  int rows = 0, dim = 0, sumC = 0;
};
int time_table(const TimeP& p, cudaStream_t s);

// FiLM positional encoding of a continuous noise level (parts/film.py:17-26): table[r][c] = sin | cos (5000 * level[r] * freq[c]);
// is_cos[c] selects the half.  freq / is_cos are per table column (all FiLM layers side by side).
int film_pe_table(const float* levels, const float* freq, const float* is_cos, float* table, int rows, int sumC, cudaStream_t s);

// FiLM apply: out = x * scale + shift (elementwise, NHWC activations; out may alias x)   (modules/unet.py:259,262)
int film_modulate(const void* x, const void* scale, const void* shift, void* out, long n, int act, cudaStream_t s);
// x[b][pix][c] += class_embed[classes[b] or pad_class][c], in place (WaveGradUNet adds the class embedding after FiLM 0, unet.py:219-226)
int class_embed_add(void* x, const float* cls_w, const int64_t* classes, int pad_class, int B, int HW, int C, int act, cudaStream_t s);

// layout conversion at the public ABI boundary
int nchw_to_nhwc(const float* in, void* out, int B, int C, int HW, int act, cudaStream_t s);
int nhwc_to_nchw(const void* in, float* out, int B, int C, int HW, int act, cudaStream_t s);
int stats_to_mean_rstd(const stat_t* stats, float* out, int n, float inv_count, cudaStream_t s);

// ---- probability-flow ODE, device-side RK45 (ode.cu) ----
// solver constants of one solve (baked into the cached graph)
struct OdeParams {
  int sde_kind = 0, N = 0, max_nfe = 0;
  double beta_0 = 0, beta_1 = 0, sigma_min = 0, sigma_max = 0;
  double t0 = 0, t1 = 0, rtol = 0, atol = 0;
};
// solver record in device memory; the controller owns it between attempts
struct OdeRec {
  double t, t_new, h, h_abs, min_step;
  double h0, d1;                         // select_initial_step carry
  int cur;                               // y[cur] = y, y[cur ^ 1] = y_new
  int k0, k6;                            // physical K slots of the FSAL pair (swapped on accept)
  int rejected;                          // a rejection happened in the current step (growth capped at 1)
  int status, nfev, n_acc, n_rej;
  float labels[6], fx[6], sc[6], g2[6];  // per stage of an attempt: U-Net time label, f(x,t) = fx * x, score scale, g(t)^2
};
// views into the caller's work buffer
struct OdeWork {
  long n = 0;                            // batch * C * H * W
  OdeRec* rec = nullptr;
  int32_t* rows = nullptr;               // {0..5}: time-table row of each stage (row_dev of the U-Net forwards)
  double* y = nullptr;                   // [2][n]
  float* K = nullptr;                    // [7][n]
  float* x32 = nullptr;                  // [n] U-Net input
  float* mo = nullptr;                   // [n] U-Net output
  double* partials = nullptr;            // [ode_grid(n)][2]
  dmn_ode_result* result = nullptr;
};
size_t ode_work_layout(long n, char* base, OdeWork* w);    // bytes; fills w when given
int ode_grid(long n);
int launch_ode_init(const OdeWork& w, const OdeParams& P, cudaStream_t st);
int launch_ode_init_elem(const OdeWork& w, const OdeParams& P, const float* state, int mode, cudaStream_t st);
int launch_ode_init_step(const OdeWork& w, const OdeParams& P, int mode, cudaGraphConditionalHandle hnd, int use_cond, cudaStream_t st);
int launch_ode_stage(const OdeWork& w, const OdeParams& P, int s, cudaStream_t st);
int launch_ode_control(const OdeWork& w, const OdeParams& P, cudaGraphConditionalHandle hnd, int use_cond, cudaStream_t st);
int launch_ode_finish(const OdeWork& w, float* state, cudaStream_t st);

}  // namespace dmn

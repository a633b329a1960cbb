// api_layers.cu -- layer-level C ABI entry points (include/dmn_b200.h, "Layer-level entry points").
// fp32 NCHW tensors at the boundary; converted to the engine's NHWC layout in caller-provided scratch.
#include <vector>

#include "../../include/dmn_b200.h"
#include "common.cuh"
#include "ops.h"

using namespace dmn;

namespace {
size_t al(size_t v) { return (v + 255) / 256 * 256; }

struct ConvScratch {
  size_t x, y, w, w2, stats_in, stats_out, total;
};
ConvScratch conv_layout(const dmn_conv_args* a) {
  const size_t esz = a->act == DMN_ACT_F32 ? 4 : 2;
  const int hout = a->mode == CONV_DOWN ? a->hin / 2 : (a->mode == CONV_UP ? a->hin * 2 : a->hin);
  const int wout = a->mode == CONV_DOWN ? a->win / 2 : (a->mode == CONV_UP ? a->win * 2 : a->win);
  const int k = a->mode == CONV_SAME ? a->ksize : 4;
  ConvScratch s;
  size_t o = 0;
  s.x = o; o += al((size_t)a->batch * a->hin * a->win * a->cin * esz);
  s.y = o; o += al((size_t)a->batch * hout * wout * a->cout * esz);
  s.w = o; o += al((size_t)a->cin * a->cout * k * k * 4);
  s.w2 = o; o += al((size_t)a->cin * a->cout * k * k * 2);
  s.stats_in = o; o += al((size_t)a->batch * 64 * 2 * 8);
  s.stats_out = o; o += al((size_t)a->batch * 64 * 2 * 8);
  s.total = o;
  return s;
}

// per-(sample, group) sum / sum-of-squares of an NHWC tensor (test path only: one thread block per (b, g))
template <typename T>
__global__ void group_stats_kernel(const T* x, stat_t* stats, int HW, int C, int G) {
  const int b = blockIdx.x / G, g = blockIdx.x % G;
  const int cpg = C / G;
  float s = 0.f, ss = 0.f;
  for (int i = threadIdx.x; i < HW * cpg; i += blockDim.x) {
    const int pix = i / cpg, c = g * cpg + i % cpg;
    const float v = to_f<T>(x[((long)b * HW + pix) * C + c]);
    s += v;
    ss += v * v;
  }
  __shared__ float rs[32], rss[32];
  s = warp_sum(s);
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) { rs[threadIdx.x >> 5] = s; rss[threadIdx.x >> 5] = ss; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, c2 = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) { a += rs[i]; c2 += rss[i]; }
    stats[2 * blockIdx.x] = __float2ll_rn(a * kStatScaleSum);
    stats[2 * blockIdx.x + 1] = __float2ll_rn(c2 * kStatScaleSq);
  }
}
}  // namespace

namespace dmn {
int conv_tcgen05_read_trace(long long* out, int n);
int conv_tcgen05_read_log(int32_t* out, int cap);
int fa_read_trace(long long* out, int n);
}

extern "C" {

/* debug only (not part of the documented ABI): timeline of one CTA of the last tcgen05 conv launched with DMN_TC_TRACE=1 */
int dmn_debug_conv_trace(long long* out, int n) { return conv_tcgen05_read_trace(out, n); }
/* debug only: one record of 64 int32 per tcgen05 conv launch since the previous call (see conv_tcgen05.cu,
 * conv_tcgen05_read_log); copies at most `cap` records, clears the log and returns how many there were.  Recording starts with the
 * first call. */
int dmn_debug_conv_log(int32_t* out, int cap) { return conv_tcgen05_read_log(out, cap); }
/* debug only: phase timeline of CTA 0 of the last fused attention launch with DMN_FA_TRACE=1 (clock64 at: image start, phase A done,
 * context built, phase B done, phase C done; slots 0..4 first image, 8..12 last image of the CTA) */
int dmn_debug_fa_trace(long long* out, int n) { return fa_read_trace(out, n); }

size_t dmn_conv_scratch_bytes(const dmn_conv_args* a) { return a ? conv_layout(a).total : 0; }

// x2 / cin2: second source of a channel concatenation (cin2 = 0: none)
static int conv_forward(const dmn_conv_args* a, const float* x2, int cin2, void* stream) {
  if (!a) return fail(DMN_EINVAL, "null args");
  DMN_REQUIRE(a->x && a->w && a->y && a->scratch_dev, "null tensor");
  DMN_REQUIRE(cin2 >= 0 && cin2 < a->cin && (cin2 == 0 || x2), "concat source");
  DMN_REQUIRE(cin2 == 0 || a->gn_groups == 0, "the concat form takes a plain operand (gn_groups = 0)");
  DMN_REQUIRE(a->mode >= 0 && a->mode <= 2, "mode");
  DMN_REQUIRE(a->act == DMN_ACT_F32 || a->act == DMN_ACT_BF16, "act");
  DMN_REQUIRE(a->engine == DMN_CONV_SIMT || a->act == DMN_ACT_BF16, "tcgen05 engine needs bf16 activations");
  DMN_REQUIRE(a->gn_groups <= 64 && a->out_groups <= 64, "too many groups");
  const ConvScratch L = conv_layout(a);
  DMN_REQUIRE(a->scratch_bytes >= L.total, "scratch too small (dmn_conv_scratch_bytes)");
  cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)a->scratch_dev;
  const int hout = a->mode == CONV_DOWN ? a->hin / 2 : (a->mode == CONV_UP ? a->hin * 2 : a->hin);
  const int wout = a->mode == CONV_DOWN ? a->win / 2 : (a->mode == CONV_UP ? a->win * 2 : a->win);
  const int k = a->mode == CONV_SAME ? a->ksize : 4;
  int rc;
  // both sources NHWC back to back in the x region
  const int cin1 = a->cin - cin2;
  const size_t x2_off = L.x + (size_t)a->batch * a->hin * a->win * cin1 * (a->act == DMN_ACT_F32 ? 4 : 2);
  if ((rc = nchw_to_nhwc(a->x, base + L.x, a->batch, cin1, a->hin * a->win, a->act, st))) return rc;
  if (cin2 && (rc = nchw_to_nhwc(x2, base + x2_off, a->batch, cin2, a->hin * a->win, a->act, st))) return rc;

  ConvP c;
  c.src1 = base + L.x; c.C1 = cin1; c.C2 = cin2;
  c.src2 = cin2 ? base + x2_off : nullptr;
  c.B = a->batch; c.Hin = a->hin; c.Win = a->win; c.Hout = hout; c.Wout = wout; c.Cout = a->cout;
  c.mode = a->mode; c.ksize = a->ksize;
  c.bias = a->bias;
  if (a->gn_groups > 0) {
    DMN_REQUIRE(a->gn_gamma && a->gn_beta, "GroupNorm prologue needs gamma/beta");
    if (a->act == DMN_ACT_F32) group_stats_kernel<float><<<a->batch * a->gn_groups, 256, 0, st>>>((const float*)(base + L.x), (stat_t*)(base + L.stats_in), a->hin * a->win, a->cin, a->gn_groups);
    else group_stats_kernel<bf16><<<a->batch * a->gn_groups, 256, 0, st>>>((const bf16*)(base + L.x), (stat_t*)(base + L.stats_in), a->hin * a->win, a->cin, a->gn_groups);
    DMN_LAUNCH_CHECK("group_stats");
    c.pro = PRO_GN | (a->silu ? PRO_SILU : 0) | (a->temb ? PRO_TEMB : 0);
    c.pstats = (const stat_t*)(base + L.stats_in); c.pgroups = a->gn_groups; c.pgamma = a->gn_gamma; c.pbeta = a->gn_beta;
    if (a->temb) { c.temb = a->temb; c.temb_bstride = a->cin; }
  }
  c.out = base + L.y;
  if (a->out_groups > 0) {
    DMN_REQUIRE(a->out_stats, "out_stats is null");
    DMN_CUDA_CHECK(cudaMemsetAsync(base + L.stats_out, 0, (size_t)a->batch * a->out_groups * 2 * 8, st));
    c.ostats = (stat_t*)(base + L.stats_out); c.ogroups = a->out_groups;
  }
  // weights: device fp32 in torch layout -> host repack -> device (validation path; sync copies are fine here)
  const size_t nw = (size_t)a->cin * a->cout * k * k;
  std::vector<float> hw(nw);
  DMN_CUDA_CHECK(cudaMemcpyAsync(hw.data(), a->w, nw * 4, cudaMemcpyDeviceToHost, st));
  DMN_CUDA_CHECK(cudaStreamSynchronize(st));
  if (a->engine == DMN_CONV_TCGEN05) {
    if (!conv_tcgen05_supported(c)) return fail(DMN_ENOTSUP, "conv shape not supported by the tcgen05 engine");
    std::vector<char> img(conv_tcgen05_weight_bytes(a->mode, a->ksize, a->cin, a->cout));
    conv_tcgen05_pack_weights(a->mode, a->ksize, a->cin, a->cout, hw.data(), img.data());
    DMN_CUDA_CHECK(cudaMemcpyAsync(base + L.w2, img.data(), img.size(), cudaMemcpyHostToDevice, st));
    DMN_CUDA_CHECK(cudaStreamSynchronize(st));
    c.w = base + L.w2;
    if ((rc = conv_tcgen05(c, st))) return rc;
  } else {
    std::vector<float> pw(nw);
    conv_simt_pack_weights(a->mode, a->ksize, a->cin, a->cout, hw.data(), pw.data(), a->act == DMN_ACT_BF16);
    DMN_CUDA_CHECK(cudaMemcpyAsync(base + L.w, pw.data(), nw * 4, cudaMemcpyHostToDevice, st));
    DMN_CUDA_CHECK(cudaStreamSynchronize(st));
    c.w = base + L.w;
    if ((rc = conv_simt(c, a->act, st))) return rc;
  }
  if ((rc = nhwc_to_nchw(base + L.y, a->y, a->batch, a->cout, hout * wout, a->act, st))) return rc;
  if (a->out_groups > 0) {
    const int cpg = a->cout / a->out_groups;
    if ((rc = stats_to_mean_rstd((const stat_t*)(base + L.stats_out), a->out_stats, a->batch * a->out_groups,
                                 1.f / (float)(hout * wout * cpg), st)))
      return rc;
  }
  return 0;
}

int dmn_conv_forward(const dmn_conv_args* a, void* stream) { return conv_forward(a, nullptr, 0, stream); }
int dmn_conv_forward_cat(const dmn_conv_args* a, const float* x2, int32_t cin2, void* stream) {
  if (cin2 <= 0) return fail(DMN_EINVAL, "dmn_conv_forward_cat: cin2 must be positive");
  return conv_forward(a, x2, cin2, stream);
}

static int attn_common(bool linear, const float* qkv, float* out, int batch, int heads, int dh, int n, int act, void* scratch,
                       size_t scratch_bytes, void* stream) {
  DMN_REQUIRE(qkv && out && scratch, "null tensor");
  const size_t esz = act == DMN_ACT_F32 ? 4 : 2;
  const size_t a_in = al((size_t)batch * n * 3 * heads * dh * esz), a_out = al((size_t)batch * n * heads * dh * esz);
  DMN_REQUIRE(scratch_bytes >= a_in + a_out, "scratch too small: need batch*n*4*heads*dim_head elements (+512 B)");
  cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)scratch;
  int rc;
  if ((rc = nchw_to_nhwc(qkv, base, batch, 3 * heads * dh, n, act, st))) return rc;
  rc = linear ? linattn_core(base, base + a_in, batch, heads, dh, n, act, st) : attn_core(base, base + a_in, batch, heads, dh, n, act, st);
  if (rc) return rc;
  return nhwc_to_nchw(base + a_in, out, batch, heads * dh, n, act, st);
}

int dmn_linear_attention_core(const float* qkv, float* out, int batch, int heads, int dim_head, int n_tokens, int act,
                              void* scratch_dev, size_t scratch_bytes, void* stream) {
  return attn_common(true, qkv, out, batch, heads, dim_head, n_tokens, act, scratch_dev, scratch_bytes, stream);
}
int dmn_attention_core(const float* qkv, float* out, int batch, int heads, int dim_head, int n_tokens, int act,
                       void* scratch_dev, size_t scratch_bytes, void* stream) {
  return attn_common(false, qkv, out, batch, heads, dim_head, n_tokens, act, scratch_dev, scratch_bytes, stream);
}

// plain GEMM through the tcgen05 engine: a 1x1 "convolution" over M pixels (H = M, W = 1)
__global__ void bf16_to_f32_kernel(const bf16* in, float* out, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __bfloat162float(in[i]);
}
int dmn_selftest_umma_gemm(const void* a_bf16, const void* b_bf16, float* d, int M, int N, int K, void* stream) {
  // b_bf16 must already be in the engine's blocked layout (host: conv_tcgen05_pack_weights via dmn_conv_forward);
  // this entry point takes row-major B[N][K] bf16 on the DEVICE and repacks through the host for simplicity.
  DMN_REQUIRE(a_bf16 && b_bf16 && d, "null tensor");
  cudaStream_t st = (cudaStream_t)stream;
  std::vector<bf16> hb((size_t)N * K);
  DMN_CUDA_CHECK(cudaMemcpyAsync(hb.data(), b_bf16, hb.size() * 2, cudaMemcpyDeviceToHost, st));
  DMN_CUDA_CHECK(cudaStreamSynchronize(st));
  std::vector<float> hf(hb.size());
  for (size_t i = 0; i < hb.size(); ++i) hf[i] = __bfloat162float(hb[i]);
  std::vector<char> img(conv_tcgen05_weight_bytes(CONV_SAME, 1, K, N));
  conv_tcgen05_pack_weights(CONV_SAME, 1, K, N, hf.data(), img.data());
  void* wdev = nullptr;
  void* odev = nullptr;
  // self-test only: the one place the library allocates (and frees) device memory itself
  DMN_CUDA_CHECK(cudaMalloc(&wdev, img.size()));
  DMN_CUDA_CHECK(cudaMalloc(&odev, (size_t)M * N * 2));
  DMN_CUDA_CHECK(cudaMemcpyAsync(wdev, img.data(), img.size(), cudaMemcpyHostToDevice, st));
  ConvP c;
  c.src1 = a_bf16; c.C1 = K; c.B = 1; c.Hin = M; c.Win = 1; c.Hout = M; c.Wout = 1; c.Cout = N;
  c.mode = CONV_SAME; c.ksize = 1; c.w = wdev; c.out = odev;
  int rc = conv_tcgen05(c, st);
  if (!rc) {
    bf16_to_f32_kernel<<<(unsigned)(((long)M * N + 255) / 256), 256, 0, st>>>((const bf16*)odev, d, (long)M * N);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = fail(DMN_ECUDA, std::string("selftest: ") + cudaGetErrorString(e));
  }
  cudaFree(wdev);
  cudaFree(odev);
  return rc;
}

int dmn_selftest_tma_sw128_gemm(const void* a_bf16, const void* b_bf16, float* d, int M, int N, int K, void* stream) {
  DMN_REQUIRE(a_bf16 && b_bf16 && d, "null tensor");
  int rc = selftest_tma_sw128_gemm(a_bf16, b_bf16, d, M, N, K, (cudaStream_t)stream);
  if (rc) return rc;
  cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
  if (e != cudaSuccess) return fail(DMN_ECUDA, std::string("selftest_tma_sw128_gemm: ") + cudaGetErrorString(e));
  return 0;
}

namespace {
struct AttnScratch {
  size_t x, y, wqkv, wo, s12, stats, total;
};
AttnScratch attn_layout(const dmn_attn_block_args* a) {
  AttnScratch s;
  size_t o = 0;
  const size_t act = (size_t)a->batch * a->n_tokens * a->dim * 2;
  s.x = o; o += al(act);
  s.y = o; o += al(act);
  s.wqkv = o; o += al((size_t)384 * a->dim * 2);
  s.wo = o; o += al((size_t)a->dim * 128 * 2);
  s.s12 = o; o += al((size_t)2 * 384 * 4);
  s.stats = o; o += al((size_t)a->batch * 2 * 8);
  s.total = o;
  return s;
}
}  // namespace

size_t dmn_linear_attention_block_scratch_bytes(const dmn_attn_block_args* a) { return a ? attn_layout(a).total : 0; }

int dmn_linear_attention_block(const dmn_attn_block_args* a, void* stream) {
  if (!a) return fail(DMN_EINVAL, "null args");
  DMN_REQUIRE(a->x && a->y && a->norm_w && a->norm_b && a->w_qkv && a->w_out && a->b_out && a->scratch_dev, "null tensor");
  DMN_REQUIRE(a->softmax || (a->out_norm_w && a->out_norm_b), "null tensor (to_out GroupNorm parameters)");
  if (a->softmax ? !attn_softmax_fused_supported(a->batch, a->n_tokens, a->dim) : !linattn_fused_supported(a->batch, a->n_tokens, a->dim))
    return fail(DMN_ENOTSUP, "fused attention block: n_tokens must be a multiple of 128 (or of 8, below 128; softmax form: at most 64) and dim 128 or 256");
  const AttnScratch L = attn_layout(a);
  DMN_REQUIRE(a->scratch_bytes >= L.total, "scratch too small (dmn_linear_attention_block_scratch_bytes)");
  cudaStream_t st = (cudaStream_t)stream;
  char* base = (char*)a->scratch_dev;
  const int C_ = a->dim;
  int rc;
  if ((rc = nchw_to_nhwc(a->x, base + L.x, a->batch, C_, a->n_tokens, ACT_BF16, st))) return rc;
  group_stats_kernel<bf16><<<a->batch, 256, 0, st>>>((const bf16*)(base + L.x), (stat_t*)(base + L.stats), a->n_tokens, C_, 1);
  DMN_LAUNCH_CHECK("group_stats");
  // host side: fold the PreNorm gamma / beta through to_qkv exactly as the plan does (plan.cu, dmn_plan_load_param)
  std::vector<float> g(C_), be(C_), wq((size_t)384 * C_), wo((size_t)C_ * 128);
  DMN_CUDA_CHECK(cudaMemcpyAsync(g.data(), a->norm_w, C_ * 4, cudaMemcpyDeviceToHost, st));
  DMN_CUDA_CHECK(cudaMemcpyAsync(be.data(), a->norm_b, C_ * 4, cudaMemcpyDeviceToHost, st));
  DMN_CUDA_CHECK(cudaMemcpyAsync(wq.data(), a->w_qkv, wq.size() * 4, cudaMemcpyDeviceToHost, st));
  DMN_CUDA_CHECK(cudaMemcpyAsync(wo.data(), a->w_out, wo.size() * 4, cudaMemcpyDeviceToHost, st));
  DMN_CUDA_CHECK(cudaStreamSynchronize(st));
  std::vector<bf16> wqb(wq.size()), wob(wo.size());
  std::vector<float> s12((size_t)2 * 384);
  for (int n = 0; n < 384; ++n) {
    double s1 = 0.0, s2 = 0.0;
    for (int c = 0; c < C_; ++c) {
      const bf16 wb = __float2bfloat16_rn(wq[(size_t)n * C_ + c] * g[c]);
      wqb[(size_t)n * C_ + c] = wb;
      s1 += (double)__bfloat162float(wb);
      s2 += (double)wq[(size_t)n * C_ + c] * (double)be[c];
    }
    s12[n] = (float)s1;
    s12[384 + n] = (float)s2;
  }
  for (size_t i = 0; i < wo.size(); ++i) wob[i] = __float2bfloat16_rn(wo[i]);
  DMN_CUDA_CHECK(cudaMemcpyAsync(base + L.wqkv, wqb.data(), wqb.size() * 2, cudaMemcpyHostToDevice, st));
  DMN_CUDA_CHECK(cudaMemcpyAsync(base + L.wo, wob.data(), wob.size() * 2, cudaMemcpyHostToDevice, st));
  DMN_CUDA_CHECK(cudaMemcpyAsync(base + L.s12, s12.data(), s12.size() * 4, cudaMemcpyHostToDevice, st));
  DMN_CUDA_CHECK(cudaStreamSynchronize(st));
  LinAttnFusedP q;
  q.x = base + L.x; q.out = base + L.y; q.pstats = (const stat_t*)(base + L.stats);
  q.wqkv = base + L.wqkv; q.wo = base + L.wo;
  q.s1 = (const float*)(base + L.s12); q.s2 = q.s1 + 384;
  q.bo = a->b_out; q.go = a->out_norm_w; q.beo = a->out_norm_b;
  q.B = a->batch; q.N = a->n_tokens; q.C = C_;
  if ((rc = a->softmax ? attn_softmax_fused(q, st) : linattn_fused(q, st))) return rc;
  return nhwc_to_nchw(base + L.y, a->y, a->batch, C_, a->n_tokens, ACT_BF16, st);
}

}  // extern "C"

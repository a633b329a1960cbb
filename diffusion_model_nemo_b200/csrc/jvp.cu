// jvp.cu -- tangent kernels of the forward-mode JVP of the U-Net (fp32 parity mode, SIMT engine).
//
// dmn_unet_jvp (plan.cu) runs the forward program op by op and, after each op, its tangent op.  Convolutions, the stem and the
// final 1x1 are linear in their operand, so their tangents reuse conv_simt / init_conv / final_proj with a null bias.  The
// nonlinear pieces are here:
//  * gn_tangent  : tangent of y = act(GroupNorm(h)) [+ res] from the primal statistics:
//                    dy = act'(a) * gamma * rstd * (dh - mean_g(dh) - hn * mean_g(hn * dh)) [+ dres],  hn = (h - mu) * rstd,
//                    a = gamma * hn + beta.  One block per (group, sample): a fixed-order sum of dh and hn * dh, then the
//                    elementwise pass.  It materialises the operand of a tangent convolution whose primal has a GroupNorm
//                    prologue, and is the whole tangent of gn_finalize.
//  * linattn_jvp : tangent of the LinearAttention core (parts/mha.py:44-58), ds = s * (dx - sum s dx) for both softmaxes.
//  * attn_jvp    : tangent of the softmax Attention core (parts/mha.py:16-29).
// Every reduction has a fixed order, so a JVP is bit-reproducible run to run.
#include <math.h>

#include "common.cuh"
#include "ops.h"

namespace dmn {

// =====================================================================================================
// GroupNorm(+SiLU) tangent
// =====================================================================================================
__global__ void __launch_bounds__(256) gn_tangent_kernel(const GnTangentP p) {
  __shared__ float red[2][256];
  const int g = blockIdx.x, b = blockIdx.y, t = threadIdx.x;
  const int cpg = p.C / p.groups;
  const long cnt = (long)p.HW * cpg;
  float mean, rstd;
  gn_mean_rstd(p.stats + ((long)b * p.groups + g) * 2, 1.f / (float)cnt, kGnEps, mean, rstd);
  const long base = (long)b * p.HW * p.C + (long)g * cpg;
  float s1 = 0.f, s2 = 0.f;
  for (long i = t; i < cnt; i += 256) {
    const long idx = base + (i / cpg) * p.C + i % cpg;
    const float dh = p.dh[idx];
    s1 += dh;
    s2 = fmaf((p.h[idx] - mean) * rstd, dh, s2);
  }
  red[0][t] = s1;
  red[1][t] = s2;
  __syncthreads();
  for (int w = 128; w > 0; w >>= 1) {
    if (t < w) { red[0][t] += red[0][t + w]; red[1][t] += red[1][t + w]; }
    __syncthreads();
  }
  const float m1 = red[0][0] / (float)cnt, m2 = red[1][0] / (float)cnt;
  for (long i = t; i < cnt; i += 256) {
    const long idx = base + (i / cpg) * p.C + i % cpg;
    const int c = g * cpg + (int)(i % cpg);
    const float hn = (p.h[idx] - mean) * rstd;
    float d = p.gamma[c] * rstd * (p.dh[idx] - m1 - hn * m2);
    if (p.silu) {
      const float a = fmaf(hn, p.gamma[c], p.beta[c]);
      const float sg = 1.f / (1.f + expf(-a));
      d *= sg * (1.f + a * (1.f - sg));
    }
    if (p.dres) d += p.dres[idx];
    p.out[idx] = d;
  }
}

int gn_tangent(const GnTangentP& p, cudaStream_t st) {
  DMN_REQUIRE(p.groups > 0 && p.C % p.groups == 0 && p.HW > 0 && p.B > 0, "gn_tangent: bad shape");
  gn_tangent_kernel<<<dim3(p.groups, p.B), 256, 0, st>>>(p);
  count_launch();
  DMN_LAUNCH_CHECK("gn_tangent");
  return 0;
}

// =====================================================================================================
// LinearAttention core tangent.  Per (sample, head), q / k / v are [32][N] (d x n):
//   ks = softmax_n(k), qs = softmax_d(q), ctx[d][e] = sum_n ks[d][n] v[e][n], out[e][n] = scale * sum_d ctx[d][e] qs[d][n]
//   dks = ks * (dk - sum_n ks dk), dqs = qs * (dq - sum_d qs dq)
//   dctx = dks v^T + ks dv^T,  dout = scale * (dctx^T qs + ctx^T dqs)
// One block (256 threads) per (sample, head); qkv / dqkv: [B][N][384] (channel = which*128 + head*32 + d), dout: [B][N][128].
// =====================================================================================================
__global__ void __launch_bounds__(256) linattn_jvp_kernel(const float* __restrict__ qkv, const float* __restrict__ dqkv,
                                                          float* __restrict__ dout, int N) {
  constexpr int TN = 64;
  __shared__ __align__(16) float tk[TN][32], tdk[TN][32], tv[TN][32], tdv[TN][32];
  __shared__ float ctx[32][32], dctx[32][32];
  __shared__ float red[2][8][32];
  __shared__ float kmax[32], kinv[32], kmd[32];
  const int b = blockIdx.x >> 2, h = blockIdx.x & 3, t = threadIdx.x;
  const float* X = qkv + (long)b * N * 384;
  const float* DX = dqkv + (long)b * N * 384;
  const int ko = 128 + h * 32, vo = 256 + h * 32, qo = h * 32;

  // phase 1: per channel d of k, the max, the sum of exp and the sum of exp * dk over tokens (thread = (d, part))
  {
    const int d = t & 31, part = t >> 5;
    float m = -INFINITY;
    for (int n = part; n < N; n += 8) m = fmaxf(m, X[(long)n * 384 + ko + d]);
    red[0][part][d] = m;
    __syncthreads();
    if (t < 32) {
      float mm = red[0][0][t];
      for (int i = 1; i < 8; ++i) mm = fmaxf(mm, red[0][i][t]);
      kmax[t] = mm;
    }
    __syncthreads();
    float s = 0.f, sd = 0.f;
    const float km = kmax[d];
    for (int n = part; n < N; n += 8) {
      const float e = expf(X[(long)n * 384 + ko + d] - km);
      s += e;
      sd = fmaf(e, DX[(long)n * 384 + ko + d], sd);
    }
    red[0][part][d] = s;
    red[1][part][d] = sd;
    __syncthreads();
    if (t < 32) {
      float ss = 0.f, ssd = 0.f;
      for (int i = 0; i < 8; ++i) { ss += red[0][i][t]; ssd += red[1][i][t]; }
      kinv[t] = 1.f / ss;
      kmd[t] = ssd / ss;
    }
    __syncthreads();
  }
  // phase 2: ctx and dctx.  thread -> row d = t / 8, columns e0 .. e0 + 3
  const int d = t >> 3, e0 = (t & 7) * 4;
  float acc[4] = {0.f, 0.f, 0.f, 0.f}, dacc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int n0 = 0; n0 < N; n0 += TN) {
    for (int i = t; i < TN * 32; i += 256) {
      const int r = i >> 5, c = i & 31;
      float k = 0.f, dk = 0.f, v = 0.f, dv = 0.f;
      if (n0 + r < N) {
        const long row = (long)(n0 + r) * 384;
        k = expf(X[row + ko + c] - kmax[c]) * kinv[c];
        dk = k * (DX[row + ko + c] - kmd[c]);
        v = X[row + vo + c];
        dv = DX[row + vo + c];
      }
      tk[r][c] = k; tdk[r][c] = dk; tv[r][c] = v; tdv[r][c] = dv;
    }
    __syncthreads();
    for (int r = 0; r < TN; ++r) {
      const float kd = tk[r][d], dkd = tdk[r][d];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc[j] = fmaf(kd, tv[r][e0 + j], acc[j]);
        dacc[j] = fmaf(dkd, tv[r][e0 + j], fmaf(kd, tdv[r][e0 + j], dacc[j]));
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) { ctx[d][e0 + j] = acc[j]; dctx[d][e0 + j] = dacc[j]; }
  __syncthreads();

  // phase 3: warp per token, lane = d for the softmax of q and its tangent, then lane = e:
  //   dout[e] = scale * sum_d (dctx[d][e] qs[d] + ctx[d][e] dqs[d])  (qs / dqs broadcast by shuffles, fixed order)
  const float scale = rsqrtf(32.f);
  const int lane = t & 31;
  for (int n = t >> 5; n < N; n += 8) {
    const float q = X[(long)n * 384 + qo + lane], dq = DX[(long)n * 384 + qo + lane];
    const float e = expf(q - warp_max(q));
    const float qs = e / warp_sum(e);
    const float dqs = qs * (dq - warp_sum(qs * dq));
    float o = 0.f;
    for (int i = 0; i < 32; ++i)
      o = fmaf(dctx[i][lane], __shfl_sync(0xffffffffu, qs, i), fmaf(ctx[i][lane], __shfl_sync(0xffffffffu, dqs, i), o));
    dout[((long)b * N + n) * 128 + h * 32 + lane] = o * scale;
  }
}

int linattn_jvp(const void* qkv, const void* dqkv, void* dout, int B, int heads, int dh, int N, cudaStream_t st) {
  DMN_REQUIRE(dh == 32 && heads == 4, "linattn_jvp: heads must be 4 and dim_head 32");
  linattn_jvp_kernel<<<B * 4, 256, 0, st>>>((const float*)qkv, (const float*)dqkv, (float*)dout, N);
  count_launch();
  DMN_LAUNCH_CHECK("linattn_jvp");
  return 0;
}

// =====================================================================================================
// softmax Attention core tangent.  Per (sample, head) and query i (q pre-scaled by 32^-1/2 as the reference does):
//   s_j = q . k_j, ds_j = dq . k_j + q . dk_j, attn = softmax_j(s), dattn = attn * (ds - sum_j attn ds)
//   dout = sum_j dattn_j v_j + attn_j dv_j = (sum_j p_j (ds_j v_j + dv_j) - (sum_j p_j ds_j / S) sum_j p_j v_j) / S,  p = exp(s - max)
// One block per (sample, head), thread per query; k, dk, v, dv of the head in shared memory.
// =====================================================================================================
__global__ void __launch_bounds__(256) attn_jvp_kernel(const float* __restrict__ qkv, const float* __restrict__ dqkv, float* __restrict__ dout,
                                                       int heads, int N) {
  constexpr int D = 32;
  extern __shared__ float akv[];   // k | dk | v | dv, each [N][D]
  float* ks = akv;
  float* dks = akv + (long)N * D;
  float* vs = akv + 2L * N * D;
  float* dvs = akv + 3L * N * D;
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int C3 = 3 * heads * D;
  const float* X = qkv + (long)b * N * C3;
  const float* DX = dqkv + (long)b * N * C3;
  const int qo = h * D, ko = heads * D + h * D, vo = 2 * heads * D + h * D;
  for (int i = threadIdx.x; i < N * D; i += blockDim.x) {
    const long r = (long)(i / D) * C3;
    const int d = i % D;
    ks[i] = X[r + ko + d];
    dks[i] = DX[r + ko + d];
    vs[i] = X[r + vo + d];
    dvs[i] = DX[r + vo + d];
  }
  __syncthreads();
  const float scale = rsqrtf((float)D);
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float q[D], dq[D], o[D], a[D];
#pragma unroll
    for (int d = 0; d < D; ++d) {
      q[d] = X[(long)i * C3 + qo + d] * scale;
      dq[d] = DX[(long)i * C3 + qo + d] * scale;
      o[d] = 0.f;
      a[d] = 0.f;
    }
    float mx = -INFINITY;
    for (int j = 0; j < N; ++j) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < D; ++d) s = fmaf(q[d], ks[j * D + d], s);
      mx = fmaxf(mx, s);
    }
    float S = 0.f, SD = 0.f;
    for (int j = 0; j < N; ++j) {
      float s = 0.f, ds = 0.f;
#pragma unroll
      for (int d = 0; d < D; ++d) {
        s = fmaf(q[d], ks[j * D + d], s);
        ds = fmaf(dq[d], ks[j * D + d], fmaf(q[d], dks[j * D + d], ds));
      }
      const float pj = expf(s - mx);
      S += pj;
      SD = fmaf(pj, ds, SD);
#pragma unroll
      for (int d = 0; d < D; ++d) {
        o[d] = fmaf(pj, vs[j * D + d], o[d]);
        a[d] = fmaf(pj, fmaf(ds, vs[j * D + d], dvs[j * D + d]), a[d]);
      }
    }
    const float inv = 1.f / S, m = SD * inv;
    float* op = dout + ((long)b * N + i) * (heads * D) + h * D;
#pragma unroll
    for (int d = 0; d < D; ++d) op[d] = (a[d] - m * o[d]) * inv;
  }
}

int attn_jvp(const void* qkv, const void* dqkv, void* dout, int B, int heads, int dh, int N, cudaStream_t st) {
  DMN_REQUIRE(dh == 32, "attn_jvp: dim_head must be 32");
  const size_t smem = (size_t)4 * N * 32 * sizeof(float);
  DMN_REQUIRE(smem <= 128 * 1024, "attn_jvp: too many tokens for the bottleneck attention tangent kernel");
  static DeviceOnce attr;
  if (attr.first()) DMN_CUDA_CHECK(cudaFuncSetAttribute(attn_jvp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
  int threads = ((N + 31) / 32) * 32;
  if (threads > 256) threads = 256;
  attn_jvp_kernel<<<B * heads, threads, smem, st>>>((const float*)qkv, (const float*)dqkv, (float*)dout, heads, N);
  count_launch();
  DMN_LAUNCH_CHECK("attn_jvp");
  return 0;
}

}  // namespace dmn

// kernels_simt.cu -- CUDA-core kernels of the sampling path.
//
//  * conv_simt      : generic implicit-GEMM convolution with fp32 FMA accumulation.  It is the arithmetic of the
//                     fp32 parity mode (1e-4 gate) and the cross-check for the tcgen05 engine; it carries the
//                     same fused prologue (GroupNorm-apply + SiLU + time-embedding add of the *producer*) and
//                     epilogue (bias, residual, GroupNorm statistics) as the tensor-core engine.
//  * init_conv      : 7x7 stem reading the fp32 NCHW sampler state directly          (modules/unet.py:41)
//  * gn_finalize    : y = SiLU(GroupNorm(raw)) + res, plus statistics for the next norm (parts/convnext.py:35-45,86)
//  * final_proj     : GroupNorm + SiLU + 1x1 conv to out_dim, fp32 NCHW out            (modules/unet.py:112-116)
//  * linattn_core / attn_core : parts/mha.py:44-58 / 16-29
//  * time_table     : sinusoid -> Linear -> GELU -> Linear -> (SiLU -> Linear) x blocks (unet.py:61-66, convnext.py:68-72)
#include <math.h>

#include "common.cuh"
#include "ops.h"

namespace dmn {

// =====================================================================================================
// generic convolution
// =====================================================================================================
template <typename T>
__global__ void __launch_bounds__(256) conv_simt_kernel(const ConvP p) {
  constexpr int BM = 64, BN = 64, BK = 16;
  __shared__ float As[BK][BM + 4];
  __shared__ __align__(16) float Bs[BK][BN];

  const int tid = threadIdx.x;
  const int Cin = p.C1 + p.C2;
  const int HWo = p.Hout * p.Wout;
  const long M = (long)p.B * HWo;
  const long m0 = (long)blockIdx.x * BM;
  const int n0 = blockIdx.y * BN;

  // A-loader role: one row (output pixel), 4 consecutive input channels
  const int arow = tid >> 2, akq = (tid & 3) * 4;
  const long am = m0 + arow;
  const bool arow_ok = am < M;
  int ab = 0, aoy = 0, aox = 0;
  if (arow_ok) {
    ab = (int)(am / HWo);
    int r = (int)(am - (long)ab * HWo);
    aoy = r / p.Wout;
    aox = r - aoy * p.Wout;
  }
  // B-loader role
  const int bk = tid >> 4, bn = (tid & 15) * 4;
  // compute role
  const int ty = tid >> 4, tx = tid & 15;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const float* temb_row = nullptr;
  if (p.pro & PRO_TEMB)
    temb_row = p.temb + (p.d_row ? (long)(*p.d_row) * p.temb_rstride : 0) + (long)ab * p.temb_bstride;
  const int cpg_in = (p.pro & PRO_GN) ? (p.C1 / p.pgroups) : 1;
  const float inv_cnt = 1.f / (float)(p.Hin * p.Win * cpg_in);

  const int kw_ = (p.mode == CONV_SAME) ? p.ksize : 4;
  const int ntaps = kw_ * kw_;
  for (int tap = 0; tap < ntaps; ++tap) {
    const int ky = tap / kw_, kx = tap - ky * kw_;
    int iy, ix;
    bool ok = arow_ok;
    if (p.mode == CONV_SAME) {
      const int pad = p.ksize >> 1;
      iy = aoy + ky - pad;
      ix = aox + kx - pad;
    } else if (p.mode == CONV_DOWN) {
      iy = aoy * 2 - 1 + ky;
      ix = aox * 2 - 1 + kx;
    } else {  // transposed conv k4 s2 p1: oy = 2*iy - 1 + ky
      const int ty_ = aoy + 1 - ky, tx_ = aox + 1 - kx;
      ok = ok && !(ty_ & 1) && !(tx_ & 1) && ty_ >= 0 && tx_ >= 0;
      iy = ty_ >> 1;
      ix = tx_ >> 1;
    }
    ok = ok && iy >= 0 && iy < p.Hin && ix >= 0 && ix < p.Win;
    const long pix = ((long)ab * p.Hin + iy) * p.Win + ix;

    for (int c0 = 0; c0 < Cin; c0 += BK) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      const int c = c0 + akq;
      if (ok && c < Cin) {
        if (c < p.C1) v = load4<T>((const T*)p.src1 + pix * p.C1 + c);
        else v = load4<T>((const T*)p.src2 + pix * p.C2 + (c - p.C1));
        if (p.pro & PRO_GN) {
          float mean, rstd;
          gn_mean_rstd(p.pstats + ((long)ab * p.pgroups + c / cpg_in) * 2, inv_cnt, kGnEps, mean, rstd);
          const float4 ga = *reinterpret_cast<const float4*>(p.pgamma + c);
          const float4 be = *reinterpret_cast<const float4*>(p.pbeta + c);
          v.x = (v.x - mean) * rstd * ga.x + be.x;
          v.y = (v.y - mean) * rstd * ga.y + be.y;
          v.z = (v.z - mean) * rstd * ga.z + be.z;
          v.w = (v.w - mean) * rstd * ga.w + be.w;
        }
        if (p.pro & PRO_SILU) {
          v.x = silu_f(v.x); v.y = silu_f(v.y); v.z = silu_f(v.z); v.w = silu_f(v.w);
        }
        if (p.pro & PRO_LRELU) {      // LeakyReLU(0.2), parts/film.py:22
          v.x = v.x > 0.f ? v.x : 0.2f * v.x; v.y = v.y > 0.f ? v.y : 0.2f * v.y;
          v.z = v.z > 0.f ? v.z : 0.2f * v.z; v.w = v.w > 0.f ? v.w : 0.2f * v.w;
        }
        if (p.pro & PRO_TEMB) {
          const float4 te = *reinterpret_cast<const float4*>(temb_row + c);
          v.x += te.x; v.y += te.y; v.z += te.z; v.w += te.w;
        }
      }
      As[akq + 0][arow] = v.x;
      As[akq + 1][arow] = v.y;
      As[akq + 2][arow] = v.z;
      As[akq + 3][arow] = v.w;

      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      const int kk = c0 + bk;
      if (kk < Cin && n0 + bn < p.Cout)
        w = *reinterpret_cast<const float4*>((const float*)p.w + ((long)tap * Cin + kk) * p.Cout + n0 + bn);
      *reinterpret_cast<float4*>(&Bs[bk][bn]) = w;
      __syncthreads();
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
        const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
        const float av[4] = {a.x, a.y, a.z, a.w};
        const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
      }
      __syncthreads();
    }
  }

  // epilogue: bias, residual, store, GroupNorm statistics of the output
  const int n = n0 + tx * 4;
  if (n >= p.Cout) return;
  float4 bias = make_float4(0.f, 0.f, 0.f, 0.f);
  if (p.bias) bias = *reinterpret_cast<const float4*>(p.bias + n);
  const int cpg_out = p.ostats ? (p.Cout / p.ogroups) : 1;
  float s = 0.f, ss = 0.f;
  int sb = -1;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const long m = m0 + ty * 4 + i;
    if (m >= M) break;
    float4 o = make_float4(acc[i][0] + bias.x, acc[i][1] + bias.y, acc[i][2] + bias.z, acc[i][3] + bias.w);
    if (p.res) {
      const float4 r = load4<T>((const T*)p.res + m * p.Cout + n);
      o.x += r.x; o.y += r.y; o.z += r.z; o.w += r.w;
    }
    store4<T>((T*)p.out + m * p.Cout + n, o);
    if (p.ostats) {
      const int b = (int)(m / HWo);
      if (b != sb && sb >= 0) {
        stat_add(p.ostats + ((long)sb * p.ogroups + n / cpg_out) * 2, s, ss);
        s = ss = 0.f;
      }
      sb = b;
      s += o.x + o.y + o.z + o.w;
      ss += o.x * o.x + o.y * o.y + o.z * o.z + o.w * o.w;
    }
  }
  if (p.ostats && sb >= 0) stat_add(p.ostats + ((long)sb * p.ogroups + n / cpg_out) * 2, s, ss);
}

int conv_simt(const ConvP& p, int act, cudaStream_t st) {
  const int Cin = p.C1 + p.C2;
  DMN_REQUIRE(p.C1 % 4 == 0 && p.C2 % 4 == 0 && p.Cout % 4 == 0 && Cin > 0, "conv_simt: channels must be multiples of 4");
  DMN_REQUIRE(!(p.pro & PRO_GN) || (p.C2 == 0 && p.pgroups > 0 && (p.C1 / p.pgroups) % 4 == 0 && p.C1 % p.pgroups == 0),
              "conv_simt: GroupNorm prologue needs a single source and channels-per-group % 4 == 0");
  DMN_REQUIRE(!p.ostats || (p.ogroups > 0 && p.Cout % p.ogroups == 0 && (p.Cout / p.ogroups) % 4 == 0),
              "conv_simt: output statistics need channels-per-group % 4 == 0");
  DMN_REQUIRE(p.mode != CONV_SAME || p.ksize == 1 || p.ksize == 3, "conv_simt: ksize must be 1 or 3");
  const long M = (long)p.B * p.Hout * p.Wout;
  dim3 grid((unsigned)((M + 63) / 64), (unsigned)((p.Cout + 63) / 64));
  if (act == ACT_F32) conv_simt_kernel<float><<<grid, 256, 0, st>>>(p);
  else conv_simt_kernel<bf16><<<grid, 256, 0, st>>>(p);
  count_launch();
  DMN_LAUNCH_CHECK("conv_simt");
  return 0;
}

void conv_simt_pack_weights(int mode, int ksize, int cin, int cout, const float* w, float* dst, bool round_bf16) {
  const int k = (mode == CONV_SAME) ? ksize : 4;
  for (int ky = 0; ky < k; ++ky)
    for (int kx = 0; kx < k; ++kx)
      for (int ci = 0; ci < cin; ++ci)
        for (int co = 0; co < cout; ++co) {
          // Conv2d weight [co][ci][ky][kx]; ConvTranspose2d weight [ci][co][ky][kx]
          const long src = (mode == CONV_UP) ? ((((long)ci * cout + co) * k + ky) * k + kx)
                                             : ((((long)co * cin + ci) * k + ky) * k + kx);
          float v = w[src];
          if (round_bf16) v = __bfloat162float(__float2bfloat16_rn(v));
          dst[(((long)(ky * k + kx)) * cin + ci) * cout + co] = v;
        }
}

// =====================================================================================================
// init conv 7x7 (pad 3) on fp32 NCHW input
// =====================================================================================================
template <typename T>
__global__ void init_conv_kernel(const InitConvP p) {
  extern __shared__ float patch[];   // [7][S+6][Cin]
  const int b = blockIdx.y, y = blockIdx.x, S = p.S, Cin = p.Cin;
  const int PW = S + 6;
  for (int i = threadIdx.x; i < 7 * PW * Cin; i += blockDim.x) {
    const int ci = i % Cin;
    const int px = (i / Cin) % PW;
    const int r = i / (Cin * PW);
    const int iy = y + r - 3, ix = px - 3;
    float v = 0.f;
    if (iy >= 0 && iy < S && ix >= 0 && ix < S) v = p.x[(((long)b * Cin + ci) * S + iy) * S + ix];
    patch[i] = v;
  }
  __syncthreads();
  int cls = p.pad_class;
  if (p.cls_w && p.classes) cls = (int)p.classes[b];
  for (int co = threadIdx.x; co < p.Cout; co += blockDim.x) {
    float base = p.bias ? p.bias[co] : 0.f;
    if (p.cls_w) base += p.cls_w[(long)cls * p.Cout + co];
    for (int x0 = 0; x0 < S; x0 += 32) {
      float acc[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = 0.f;
      for (int ky = 0; ky < 7; ++ky)
        for (int kx = 0; kx < 7; ++kx)
          for (int ci = 0; ci < Cin; ++ci) {
            const float wv = p.w[((long)(ky * 7 + kx) * Cin + ci) * p.Cout + co];
            const float* pr = patch + ((long)ky * PW + x0 + kx) * Cin + ci;
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (x0 + i < S) acc[i] = fmaf(pr[(long)i * Cin], wv, acc[i]);
          }
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (x0 + i < S) ((T*)p.out)[(((long)b * S + y) * S + x0 + i) * p.Cout + co] = from_f<T>(acc[i] + base);
    }
  }
}

int init_conv(const InitConvP& p, int act, cudaStream_t st) {
  const size_t smem = (size_t)7 * (p.S + 6) * p.Cin * sizeof(float);
  DMN_REQUIRE(smem <= 48 * 1024, "init_conv: input row patch does not fit in shared memory");
  dim3 grid(p.S, p.B);
  const int threads = p.Cout >= 128 ? 128 : (p.Cout >= 64 ? 64 : 32);
  if (act == ACT_F32) init_conv_kernel<float><<<grid, threads, smem, st>>>(p);
  else init_conv_kernel<bf16><<<grid, threads, smem, st>>>(p);
  count_launch();
  DMN_LAUNCH_CHECK("init_conv");
  return 0;
}

// =====================================================================================================
// GroupNorm finalize: y = act(GN(raw)) + res ; statistics of y for the next norm.  HBM-bound: 3 x esz bytes / element.
// grid = (blocks_per_image, B), 256 threads, 16-byte accesses (8 bf16 / 4 fp32 channels per thread); the item stride is a
// multiple of C/VEC so each thread keeps one channel vector (=> one input group, one output group) for its whole loop.
// =====================================================================================================
template <typename T, int V> struct VecIO;
template <> struct VecIO<float, 4> {
  static constexpr int N = 4;
  typedef float4 Raw;
  static __device__ __forceinline__ void unpack(const Raw& t, float* v) { v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
  static __device__ __forceinline__ void load(const float* p, float* v) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void store(float* p, const float* v) { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};
template <> struct VecIO<bf16, 4> {
  static constexpr int N = 4;
  typedef uint2 Raw;
  static __device__ __forceinline__ void unpack(const Raw& u, float* v) {
    v[0] = __uint_as_float(u.x << 16); v[1] = __uint_as_float(u.x & 0xffff0000u);
    v[2] = __uint_as_float(u.y << 16); v[3] = __uint_as_float(u.y & 0xffff0000u);
  }
  static __device__ __forceinline__ void load(const bf16* p, float* v) {
    const float4 t = load4<bf16>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void store(bf16* p, const float* v) { store4<bf16>(p, make_float4(v[0], v[1], v[2], v[3])); }
};
template <> struct VecIO<bf16, 8> {
  static constexpr int N = 8;
  typedef uint4 Raw;
  static __device__ __forceinline__ void unpack(const Raw& u, float* v) { unpack8(u, v); }
  static __device__ __forceinline__ void load(const bf16* p, float* v) { unpack8(*reinterpret_cast<const uint4*>(p), v); }
  static __device__ __forceinline__ void store(bf16* p, const float* v) { *reinterpret_cast<uint4*>(p) = pack8(v); }
};

// raw conv output and residual are dead (raw) or cold (residual) after this kernel while the result is read by the very next kernel:
// streaming loads (evict-first) keep the 126 MB L2 for the output
#define DMN_FIN_LD(ptr) __ldcs(ptr)
template <typename T, int V>
__global__ void __launch_bounds__(256, 3) gn_finalize_kernel(const FinalizeP p) {
  pdl_trigger();
  pdl_wait();
  __shared__ unsigned long long sm_stats[2 * 64];
  const int b = blockIdx.y;
  const int CV = p.C / V;
  const long items = (long)p.HW * CV;
  const int c = (threadIdx.x % CV) * V;
  const int cpg = p.C / p.groups;
  float mean, rstd;
  gn_mean_rstd(p.stats + ((long)b * p.groups + c / cpg) * 2, 1.f / (float)(p.HW * cpg), kGnEps, mean, rstd);
  float sc[V], sh[V];
#pragma unroll
  for (int e = 0; e < V; ++e) {
    sc[e] = rstd * p.gamma[c + e];
    sh[e] = p.beta[c + e] - mean * sc[e];
  }
  if (p.ostats) {
    for (int i = threadIdx.x; i < 2 * p.ogroups; i += blockDim.x) sm_stats[i] = 0ull;
    __syncthreads();
  }
  float s = 0.f, ss = 0.f;
  const T* raw = (const T*)p.raw + (long)b * p.HW * p.C;
  const T* res = p.res ? (const T*)p.res + (long)b * p.HW * p.C : nullptr;
  T* out = (T*)p.out + (long)b * p.HW * p.C;
  const long stride = (long)gridDim.x * blockDim.x;
  // 4 independent 16-byte items per thread and iteration (8 loads in flight with the residual): latency is covered by ILP
  constexpr int U = 4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < items; i += U * stride) {
    typedef typename VecIO<T, V>::Raw Raw;
    Raw vr[U], rr[U];                       // packed: 16 bytes per item until it is processed
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (i + u * stride < items) vr[u] = DMN_FIN_LD(reinterpret_cast<const Raw*>(raw + (i + u * stride) * V));
    if (res) {
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (i + u * stride < items) rr[u] = DMN_FIN_LD(reinterpret_cast<const Raw*>(res + (i + u * stride) * V));
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i + u * stride < items) {
        float v[V], r[V];
        VecIO<T, V>::unpack(vr[u], v);
        if (res) VecIO<T, V>::unpack(rr[u], r);
#pragma unroll
        for (int e = 0; e < V; ++e) {
          float t = fmaf(v[e], sc[e], sh[e]);
          if (p.silu) t = sizeof(T) == 2 ? silu_fast(t) : silu_f(t);
          if (res) t += r[e];
          v[e] = t;
          s += t;
          ss += t * t;
        }
        VecIO<T, V>::store(out + (i + u * stride) * V, v);
      }
    }
  }
  if (p.ostats) {
    const int og = c / (p.C / p.ogroups);
    // lanes that share the output group form aligned power-of-two classes: butterfly over them, then one fixed-point integer
    // atomic per class (order independent => deterministic)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const int og2 = __shfl_xor_sync(0xffffffffu, og, o);
      const float s2 = __shfl_xor_sync(0xffffffffu, s, o), ss2 = __shfl_xor_sync(0xffffffffu, ss, o);
      if (og2 == og) { s += s2; ss += ss2; }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, og);
    if ((threadIdx.x & 31) == __ffs(peers) - 1) {
      atomicAdd(&sm_stats[og * 2], (unsigned long long)__float2ll_rn(s * kStatScaleSum));
      atomicAdd(&sm_stats[og * 2 + 1], (unsigned long long)__float2ll_rn(ss * kStatScaleSq));
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * p.ogroups; i += blockDim.x)
      atomicAdd(reinterpret_cast<unsigned long long*>(p.ostats) + (long)b * p.ogroups * 2 + i, sm_stats[i]);
  }
}

int gn_finalize(const FinalizeP& p, int act, cudaStream_t st) {
  int V = act == ACT_F32 ? 4 : 8;
  if (V == 8 && ((p.C / p.groups) % 8 || (p.ostats && (p.C / p.ogroups) % 8) || 256 % (p.C / 8))) V = 4;
  DMN_REQUIRE(p.C % V == 0 && 256 % (p.C / V) == 0, "gn_finalize: C/vector must divide 256");
  DMN_REQUIRE(p.C % p.groups == 0 && (p.C / p.groups) % V == 0, "gn_finalize: channels-per-group must be a multiple of the vector width");
  DMN_REQUIRE(!p.ostats || (p.ogroups <= 64 && p.C % p.ogroups == 0 && (p.C / p.ogroups) % V == 0), "gn_finalize: ogroups");
  const long items = (long)p.HW * (p.C / V);
  int bpi = (int)((items + 256 * 8 - 1) / (256 * 8));     // ~8 items (2 unrolled iterations) per thread
  if (bpi < 1) bpi = 1;
  if (bpi > 64) bpi = 64;
  dim3 grid(bpi, p.B);
  if (act == ACT_F32) DMN_CUDA_CHECK(launch_pdl(gn_finalize_kernel<float, 4>, grid, dim3(256), 0, st, p));
  else if (V == 8) DMN_CUDA_CHECK(launch_pdl(gn_finalize_kernel<bf16, 8>, grid, dim3(256), 0, st, p));
  else DMN_CUDA_CHECK(launch_pdl(gn_finalize_kernel<bf16, 4>, grid, dim3(256), 0, st, p));
  count_launch();
  DMN_LAUNCH_CHECK("gn_finalize");
  return 0;
}

// =====================================================================================================
// final projection: eps[b][co][pix] = sum_c SiLU(GN(y))[b][pix][c] * w[co][c] + bias[co]      (fp32 NCHW out)
// one thread per pixel (the output is pixel-contiguous per channel => coalesced fp32 stores); GroupNorm coefficients and
// the tiny weight matrix live in shared memory.  HBM-bound: esz*C bytes read + 4*Cout written per pixel.
// =====================================================================================================
template <typename T>
__global__ void __launch_bounds__(128) final_proj_kernel(const FinalProjP p) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float fsm[];
  float* s_sc = fsm;                 // [C] rstd*gamma
  float* s_sh = fsm + p.C;           // [C] beta - mean*rstd*gamma
  float* s_w = fsm + 2 * p.C;        // [Cout][C]
  const int b = blockIdx.y;
  if (!p.plain) {
    const int cpg = p.C / p.groups;
    const float inv = 1.f / (float)(p.HW * cpg);
    for (int c = threadIdx.x; c < p.C; c += blockDim.x) {
      float mean, rstd;
      gn_mean_rstd(p.stats + ((long)b * p.groups + c / cpg) * 2, inv, kGnEps, mean, rstd);
      const float sc = rstd * p.gamma[c];
      s_sc[c] = sc;
      s_sh[c] = p.beta[c] - mean * sc;
    }
  }
  for (int i = threadIdx.x; i < p.Cout * p.C; i += blockDim.x) s_w[i] = p.w[i];
  __syncthreads();
  const int pix = blockIdx.x * blockDim.x + threadIdx.x;
  if (pix >= p.HW) return;
  const T* y = (const T*)p.y + ((long)b * p.HW + pix) * p.C;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  for (int c = 0; c < p.C; c += 4) {
    const float4 t = load4<T>(y + c);
    const float v[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float a = p.plain ? v[e] : silu_f(fmaf(v[e], s_sc[c + e], s_sh[c + e]));
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < p.Cout) acc[j] = fmaf(a, s_w[j * p.C + c + e], acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (j < p.Cout) p.out[((long)b * p.Cout + j) * p.HW + pix] = acc[j] + (p.bias ? p.bias[j] : 0.f);
}


// bf16 fast path: the block's 128 pixel rows are first copied (coalesced 16-byte cp.async) into shared memory with padded rows, then
// one thread per pixel walks its row with conflict-free LDS.128; COUT is a template parameter so the dot products are straight-line.
template <int COUT>
__global__ void __launch_bounds__(128) final_proj_bf16_kernel(const FinalProjP p) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) unsigned char fsmb[];
  const int C = p.C, ld = C * 2 + 16;                       // bytes per staged pixel row
  float* s_sc = reinterpret_cast<float*>(fsmb);             // [C] rstd*gamma
  float* s_sh = s_sc + C;                                   // [C] beta - mean*rstd*gamma
  float* s_w = s_sh + C;                                    // [COUT][C]
  unsigned char* s_tile = fsmb + (size_t)(2 + COUT) * C * 4;
  const int b = blockIdx.y, pix0 = blockIdx.x * 128;
  const int npix = min(128, p.HW - pix0);
  {
    const bf16* y = (const bf16*)p.y + ((long)b * p.HW + pix0) * C;
    const int chunks = C / 8;                               // 16-byte chunks per row
    const uint32_t tile_u = (uint32_t)__cvta_generic_to_shared(s_tile);
    for (int i = threadIdx.x; i < npix * chunks; i += 128) {
      const int r = i / chunks, c16 = i - r * chunks;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(tile_u + (uint32_t)(r * ld + c16 * 16)), "l"(y + (long)r * C + c16 * 8) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  if (!p.plain) {
    const int cpg = C / p.groups;
    const float inv = 1.f / (float)(p.HW * cpg);
    for (int c = threadIdx.x; c < C; c += 128) {
      float mean, rstd;
      gn_mean_rstd(p.stats + ((long)b * p.groups + c / cpg) * 2, inv, kGnEps, mean, rstd);
      const float sc = rstd * p.gamma[c];
      s_sc[c] = sc;
      s_sh[c] = p.beta[c] - mean * sc;
    }
  }
  for (int i = threadIdx.x; i < COUT * C; i += 128) s_w[i] = p.w[i];
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();
  if ((int)threadIdx.x >= npix) return;
  const unsigned char* row = s_tile + (size_t)threadIdx.x * ld;
  float acc[COUT];
#pragma unroll
  for (int j = 0; j < COUT; ++j) acc[j] = 0.f;
  for (int c = 0; c < C; c += 8) {
    float v[8];
    unpack8(*reinterpret_cast<const uint4*>(row + c * 2), v);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float a = p.plain ? v[e] : silu_fast(fmaf(v[e], s_sc[c + e], s_sh[c + e]));
#pragma unroll
      for (int j = 0; j < COUT; ++j) acc[j] = fmaf(a, s_w[j * C + c + e], acc[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < COUT; ++j) p.out[((long)b * COUT + j) * p.HW + pix0 + threadIdx.x] = acc[j] + (p.bias ? p.bias[j] : 0.f);
}

int final_proj(const FinalProjP& p, int act, cudaStream_t st) {
  DMN_REQUIRE(p.Cout <= 8 && p.C % 4 == 0, "final_proj: out_dim > 8 or C % 4 != 0 unsupported");
  const size_t smem = (size_t)(2 + p.Cout) * p.C * sizeof(float);
  DMN_REQUIRE(smem <= 48 * 1024, "final_proj: channel count too large");
  dim3 grid((unsigned)((p.HW + 127) / 128), (unsigned)p.B);
  if (act == ACT_BF16 && p.C % 8 == 0 && (p.Cout == 3 || p.Cout == 6 || p.Cout == 1)) {
    const size_t smem2 = (size_t)(2 + p.Cout) * p.C * sizeof(float) + (size_t)128 * (p.C * 2 + 16);
    if (smem2 <= 200 * 1024) {
      static DeviceOnce attr;
      if (attr.first()) {
        DMN_CUDA_CHECK(cudaFuncSetAttribute(final_proj_bf16_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        DMN_CUDA_CHECK(cudaFuncSetAttribute(final_proj_bf16_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        DMN_CUDA_CHECK(cudaFuncSetAttribute(final_proj_bf16_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      }
      if (p.Cout == 3) DMN_CUDA_CHECK(launch_pdl(final_proj_bf16_kernel<3>, grid, dim3(128), smem2, st, p));
      else if (p.Cout == 6) DMN_CUDA_CHECK(launch_pdl(final_proj_bf16_kernel<6>, grid, dim3(128), smem2, st, p));
      else DMN_CUDA_CHECK(launch_pdl(final_proj_bf16_kernel<1>, grid, dim3(128), smem2, st, p));
      count_launch();
      DMN_LAUNCH_CHECK("final_proj");
      return 0;
    }
  }
  if (act == ACT_F32) DMN_CUDA_CHECK(launch_pdl(final_proj_kernel<float>, grid, dim3(128), smem, st, p));
  else DMN_CUDA_CHECK(launch_pdl(final_proj_kernel<bf16>, grid, dim3(128), smem, st, p));
  count_launch();
  DMN_LAUNCH_CHECK("final_proj");
  return 0;
}

// =====================================================================================================
// LinearAttention core (parts/mha.py:44-58), heads = 4, dim_head = 32.  One block (256 threads) per SAMPLE (all heads):
//   q softmax over d (dim=-2), k softmax over n (dim=-1), q *= scale (after softmax),
//   ctx[h][d][e] = sum_n k[d,n] v[e,n] ; out[e,n] = sum_d ctx[d][e] q[d,n]
// qkv: [B][N][384] (channel = which*128 + head*32 + d);  out: [B][N][128].
// Tokens stream through shared-memory tiles with coalesced 256-byte rows; every reduction has a fixed order (deterministic).
// =====================================================================================================
template <typename T>
__global__ void __launch_bounds__(256) linattn_kernel(const T* __restrict__ qkv, T* __restrict__ out, int N) {
  constexpr int HD = 128, TN = 32, LD = HD + 4;     // row padding keeps float4 rows 16-byte aligned and spreads banks
  extern __shared__ __align__(16) float lsm[];
  float (*tP)[LD] = reinterpret_cast<float (*)[LD]>(lsm);                       // exp(k - max) | q tile rows [0,32)
  float (*tV)[LD] = reinterpret_cast<float (*)[LD]>(lsm + TN * LD);             // v            | q tile rows [32,64)
  float (*ctx)[32][32] = reinterpret_cast<float (*)[32][32]>(lsm + 2 * TN * LD);   // [head][d][e]
  float (*red)[HD] = reinterpret_cast<float (*)[HD]>(lsm + 2 * TN * LD + 4 * 32 * 32);
  float* kmax = lsm + 2 * TN * LD + 4 * 32 * 32 + 2 * HD;
  float* kinv = kmax + HD;
  const int b = blockIdx.x, t = threadIdx.x;
  const T* base = qkv + (long)b * N * 384;

  // phase 1: max over tokens of k, per channel  (thread = (channel, half))
  {
    const int c = t & 127, half = t >> 7;
    float m = -INFINITY;
    for (int n = half; n < N; n += 2) m = fmaxf(m, to_f<T>(base[(long)n * 384 + 128 + c]));
    red[half][c] = m;
    __syncthreads();
    if (t < HD) kmax[t] = fmaxf(red[0][t], red[1][t]);
    __syncthreads();
  }
  // phase 2: ctx accumulation.  thread -> head h = t/64, 4x4 patch (d0, e0) of the 32x32 context
  const int h = t >> 6, pd = ((t & 63) >> 3) * 4, pe = (t & 7) * 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  float ksum = 0.f;                                  // threads 0..127: running sum of exp for channel t
  for (int n0 = 0; n0 < N; n0 += TN) {
    // load tile: TN tokens x (k 128 + v 128) channels, 4 channels per thread-iteration
    for (int i = t; i < TN * 64; i += 256) {
      const int r = i >> 6, q4 = (i & 63) * 4;       // q4 in [0,256): [0,128) -> k, [128,256) -> v
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      const bool ok = n0 + r < N;
      if (ok) v = load4<T>(base + (long)(n0 + r) * 384 + 128 + q4);
      if (q4 < 128) {
        if (ok) {
          v.x = __expf(v.x - kmax[q4]); v.y = __expf(v.y - kmax[q4 + 1]); v.z = __expf(v.z - kmax[q4 + 2]); v.w = __expf(v.w - kmax[q4 + 3]);
        }
        *reinterpret_cast<float4*>(&tP[r][q4]) = v;
      } else {
        *reinterpret_cast<float4*>(&tV[r][q4 - 128]) = v;
      }
    }
    __syncthreads();
    if (t < HD) {
#pragma unroll 8
      for (int r = 0; r < TN; ++r) ksum += tP[r][t];
    }
#pragma unroll 4
    for (int r = 0; r < TN; ++r) {
      const float4 pk = *reinterpret_cast<const float4*>(&tP[r][h * 32 + pd]);
      const float4 vv = *reinterpret_cast<const float4*>(&tV[r][h * 32 + pe]);
      const float pa[4] = {pk.x, pk.y, pk.z, pk.w}, va[4] = {vv.x, vv.y, vv.z, vv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(pa[i], va[j], acc[i][j]);
    }
    __syncthreads();
  }
  if (t < HD) kinv[t] = 1.f / ksum;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) ctx[h][pd + i][pe + j] = acc[i][j] * kinv[h * 32 + pd + i];
  __syncthreads();

  // phase 3: per token softmax of q over d, scale, out[e] = sum_d ctx[d][e] * q[d].  thread = (token r = t%64.., head)
  const float scale = rsqrtf(32.f);
  for (int n0 = 0; n0 < N; n0 += 2 * TN) {
    // q tile of 64 tokens: rows [0,32) in tP, [32,64) in tV
    for (int i = t; i < 2 * TN * 32; i += 256) {
      const int r = i >> 5, q4 = (i & 31) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (n0 + r < N) v = load4<T>(base + (long)(n0 + r) * 384 + q4);
      float* dst = r < TN ? &tP[r][q4] : &tV[r - TN][q4];
      *reinterpret_cast<float4*>(dst) = v;
    }
    __syncthreads();
    {
      const int r = t & 63, hh = t >> 6;
      const float* qrow = (r < TN ? &tP[r][0] : &tV[r - TN][0]) + hh * 32;
      float q[32];
      float qm = -INFINITY;
#pragma unroll
      for (int d = 0; d < 32; d += 4) {
        const float4 v = *reinterpret_cast<const float4*>(qrow + d);
        q[d] = v.x; q[d + 1] = v.y; q[d + 2] = v.z; q[d + 3] = v.w;
        qm = fmaxf(fmaxf(qm, fmaxf(v.x, v.y)), fmaxf(v.z, v.w));
      }
      float qs = 0.f;
#pragma unroll
      for (int d = 0; d < 32; ++d) { q[d] = __expf(q[d] - qm); qs += q[d]; }
      const float qn = scale / qs;
      T* op = out + ((long)b * N + n0 + r) * HD + hh * 32;
#pragma unroll
      for (int eh = 0; eh < 32; eh += 16) {
        float o[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) o[e] = 0.f;
#pragma unroll
        for (int d = 0; d < 32; ++d) {
          const float qd = q[d] * qn;
#pragma unroll
          for (int e = 0; e < 16; e += 4) {
            const float4 cv = *reinterpret_cast<const float4*>(&ctx[hh][d][eh + e]);
            o[e] = fmaf(cv.x, qd, o[e]); o[e + 1] = fmaf(cv.y, qd, o[e + 1]); o[e + 2] = fmaf(cv.z, qd, o[e + 2]); o[e + 3] = fmaf(cv.w, qd, o[e + 3]);
          }
        }
        if (n0 + r < N) {
#pragma unroll
          for (int e = 0; e < 16; e += 4) store4<T>(op + eh + e, make_float4(o[e], o[e + 1], o[e + 2], o[e + 3]));
        }
      }
    }
    __syncthreads();
  }
}

int linattn_core(const void* qkv, void* out, int B, int heads, int dh, int N, int act, cudaStream_t st) {
  DMN_REQUIRE(dh == 32 && heads == 4, "linattn_core: heads must be 4 and dim_head 32");
  if (act == ACT_BF16) return linattn_core_bf16_mma(qkv, out, B, N, st);   // tensor-core kernel (linattn_mma.cu)
  const size_t smem = (size_t)(2 * 32 * 132 + 4 * 32 * 32 + 4 * 128) * sizeof(float);
  static DeviceOnce attr;
  if (attr.first()) {
    DMN_CUDA_CHECK(cudaFuncSetAttribute(linattn_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DMN_CUDA_CHECK(cudaFuncSetAttribute(linattn_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  if (act == ACT_F32) linattn_kernel<float><<<B, 256, smem, st>>>((const float*)qkv, (float*)out, N);
  else linattn_kernel<bf16><<<B, 256, smem, st>>>((const bf16*)qkv, (bf16*)out, N);
  count_launch();
  DMN_LAUNCH_CHECK("linattn_core");
  return 0;
}

// =====================================================================================================
// softmax Attention core (parts/mha.py:16-29), dim_head = 32.  One block per (sample, head), thread per query.
// =====================================================================================================
template <typename T>
__global__ void attn_kernel(const T* __restrict__ qkv, T* __restrict__ out, int heads, int N) {
  pdl_trigger();
  pdl_wait();
  constexpr int D = 32;
  extern __shared__ float kv[];   // k[N][D], v[N][D]
  float* ks = kv;
  float* vs = kv + (long)N * D;
  const int b = blockIdx.x / heads, h = blockIdx.x % heads;
  const int C3 = 3 * heads * D;
  const T* base = qkv + (long)b * N * C3;
  const int qo = h * D, ko = heads * D + h * D, vo = 2 * heads * D + h * D;
  for (int i = threadIdx.x; i < N * D; i += blockDim.x) {
    const int n = i / D, d = i % D;
    ks[i] = to_f<T>(base[(long)n * C3 + ko + d]);
    vs[i] = to_f<T>(base[(long)n * C3 + vo + d]);
  }
  __syncthreads();
  const float scale = rsqrtf((float)D);
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    float q[D], o[D];
#pragma unroll
    for (int d = 0; d < D; ++d) { q[d] = to_f<T>(base[(long)i * C3 + qo + d]) * scale; o[d] = 0.f; }
    float mx = -INFINITY, sum = 0.f;
    for (int j = 0; j < N; ++j) {
      float s = 0.f;
#pragma unroll
      for (int d = 0; d < D; ++d) s = fmaf(q[d], ks[j * D + d], s);
      const float nm = fmaxf(mx, s);
      const float corr = __expf(mx - nm);
      const float pj = __expf(s - nm);
      sum = sum * corr + pj;
#pragma unroll
      for (int d = 0; d < D; ++d) o[d] = fmaf(pj, vs[j * D + d], o[d] * corr);
      mx = nm;
    }
    const float inv = 1.f / sum;
    T* op = out + ((long)b * N + i) * (heads * D) + h * D;
#pragma unroll
    for (int d = 0; d < D; ++d) op[d] = from_f<T>(o[d] * inv);
  }
}

int attn_core(const void* qkv, void* out, int B, int heads, int dh, int N, int act, cudaStream_t st) {
  DMN_REQUIRE(dh == 32, "attn_core: dim_head must be 32");
  const size_t smem = (size_t)2 * N * 32 * sizeof(float);
  DMN_REQUIRE(smem <= 48 * 1024, "attn_core: too many tokens for the bottleneck attention kernel");
  int threads = ((N + 31) / 32) * 32;
  if (threads > 256) threads = 256;
  if (act == ACT_F32) DMN_CUDA_CHECK(launch_pdl(attn_kernel<float>, dim3(B * heads), dim3(threads), smem, st, (const float*)qkv, (float*)out, heads, N));
  else DMN_CUDA_CHECK(launch_pdl(attn_kernel<bf16>, dim3(B * heads), dim3(threads), smem, st, (const bf16*)qkv, (bf16*)out, heads, N));
  count_launch();
  DMN_LAUNCH_CHECK("attn_core");
  return 0;
}

// =====================================================================================================
// time path (fp32 throughout)
// =====================================================================================================
__global__ void sinusoid_kernel(const float* __restrict__ times, const float* __restrict__ freqs, float* __restrict__ out,
                                int rows, int dim, int ld) {
  const int half = dim >> 1;
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)rows * half) return;
  const int r = (int)(i / half), k = (int)(i % half);
  const float a = times[r] * freqs[k];
  out[(long)r * ld + k] = sinf(a);
  out[(long)r * ld + half + k] = cosf(a);
}

// out[r][n] = act_out( sum_k in[r][k] * wT[k][n] + b[n] );  act_out: 0 none, 1 gelu(erf), 2 silu
__global__ void __launch_bounds__(256) rows_linear_kernel(const float* __restrict__ in, int ld_in, int K, const float* __restrict__ wT,
                                                          const float* __restrict__ bias, int N, float* __restrict__ out, int ld_out,
                                                          int act_out) {
  extern __shared__ float row[];
  const int r = blockIdx.y;
  for (int k = threadIdx.x; k < K; k += blockDim.x) row[k] = in[(long)r * ld_in + k];
  __syncthreads();
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float acc = 0.f;
  for (int k = 0; k < K; ++k) acc = fmaf(row[k], wT[(long)k * N + n], acc);
  acc += bias[n];
  if (act_out == 1) acc = 0.5f * acc * (1.0f + erff(acc * 0.70710678118654752440f));
  else if (act_out == 2) acc = acc / (1.0f + expf(-acc));
  out[(long)r * ld_out + n] = acc;
}

int time_table(const TimeP& p, cudaStream_t st) {
  const int td = 4 * p.dim;
  DMN_REQUIRE(p.rows > 0 && p.dim % 2 == 0, "time_table: bad shape");
  float* e0 = p.tmp;                      // [rows][td] (first `dim` columns used)
  float* h1 = p.tmp + (long)p.rows * td;  // [rows][td]
  {
    const long n = (long)p.rows * (p.dim / 2);
    sinusoid_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p.times, p.freqs, e0, p.rows, p.dim, td);
    count_launch();
    DMN_LAUNCH_CHECK("sinusoid");
  }
  dim3 g1((td + 255) / 256, p.rows);
  rows_linear_kernel<<<g1, 256, p.dim * sizeof(float), st>>>(e0, td, p.dim, p.w1t, p.b1, td, h1, td, 1);
  count_launch();
  DMN_LAUNCH_CHECK("time_mlp.1");
  // second Linear, then SiLU (the per-block mlp starts with SiLU, convnext.py:69) stored back into e0
  rows_linear_kernel<<<g1, 256, td * sizeof(float), st>>>(h1, td, td, p.w3t, p.b3, td, e0, td, 2);
  count_launch();
  DMN_LAUNCH_CHECK("time_mlp.3");
  dim3 g2((p.sumC + 255) / 256, p.rows);
  rows_linear_kernel<<<g2, 256, td * sizeof(float), st>>>(e0, td, td, p.wct, p.bc, p.sumC, p.table, p.sumC, 0);
  count_launch();
  DMN_LAUNCH_CHECK("block_mlps");
  return 0;
}

// =====================================================================================================
// FiLM (WaveGradUNet): positional encoding of the noise level, and the modulation x * scale + shift
// =====================================================================================================
// table[r][c] = sin | cos ((5000 * level[r]) * freq[c]) in fp32 with the reference's multiplication order (parts/film.py:21-24)
__global__ void film_pe_kernel(const float* __restrict__ levels, const float* __restrict__ freq, const float* __restrict__ is_cos,
                               float* __restrict__ table, int rows, int sumC) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long)rows * sumC) return;
  const int r = (int)(i / sumC), c = (int)(i - (long)r * sumC);
  const float a = __fmul_rn(__fmul_rn(5000.0f, levels[r]), freq[c]);
  table[i] = is_cos[c] != 0.f ? cosf(a) : sinf(a);
}
int film_pe_table(const float* levels, const float* freq, const float* is_cos, float* table, int rows, int sumC, cudaStream_t st) {
  DMN_REQUIRE(rows > 0 && sumC > 0, "film_pe_table: bad shape");
  const long n = (long)rows * sumC;
  film_pe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(levels, freq, is_cos, table, rows, sumC);
  count_launch();
  DMN_LAUNCH_CHECK("film_pe_table");
  return 0;
}

template <typename T>
__global__ void __launch_bounds__(256) film_modulate_kernel(const T* __restrict__ x, const T* __restrict__ scale, const T* __restrict__ shift,
                                                            T* __restrict__ out, long n4) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 a = load4<T>(x + 4 * i), s = load4<T>(scale + 4 * i), t = load4<T>(shift + 4 * i);
    // reference order: x * scale + shift with a rounding after the product (two torch ops)
    store4<T>(out + 4 * i, make_float4(__fadd_rn(__fmul_rn(a.x, s.x), t.x), __fadd_rn(__fmul_rn(a.y, s.y), t.y),
                                       __fadd_rn(__fmul_rn(a.z, s.z), t.z), __fadd_rn(__fmul_rn(a.w, s.w), t.w)));
  }
}
int film_modulate(const void* x, const void* scale, const void* shift, void* out, long n, int act, cudaStream_t st) {
  DMN_REQUIRE(n > 0 && n % 4 == 0, "film_modulate: element count must be a multiple of 4");
  const long n4 = n / 4;
  long blocks = (n4 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (act == ACT_F32) film_modulate_kernel<float><<<(unsigned)blocks, 256, 0, st>>>((const float*)x, (const float*)scale, (const float*)shift, (float*)out, n4);
  else film_modulate_kernel<bf16><<<(unsigned)blocks, 256, 0, st>>>((const bf16*)x, (const bf16*)scale, (const bf16*)shift, (bf16*)out, n4);
  count_launch();
  DMN_LAUNCH_CHECK("film_modulate");
  return 0;
}

template <typename T>
__global__ void __launch_bounds__(256) class_embed_add_kernel(T* __restrict__ x, const float* __restrict__ cls_w, const int64_t* __restrict__ classes,
                                                              int pad_class, long per_sample4, int C, long n4) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const int b = (int)(i / per_sample4);
    const int c = (int)((i * 4) % C);
    const float* row = cls_w + (long)(classes ? (int)classes[b] : pad_class) * C + c;
    float4 v = load4<T>(x + 4 * i);
    v.x += row[0]; v.y += row[1]; v.z += row[2]; v.w += row[3];
    store4<T>(x + 4 * i, v);
  }
}
int class_embed_add(void* x, const float* cls_w, const int64_t* classes, int pad_class, int B, int HW, int C, int act, cudaStream_t st) {
  DMN_REQUIRE(C % 4 == 0 && cls_w, "class_embed_add: channels must be a multiple of 4");
  const long n4 = (long)B * HW * C / 4, per4 = (long)HW * C / 4;
  long blocks = (n4 + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (act == ACT_F32) class_embed_add_kernel<float><<<(unsigned)blocks, 256, 0, st>>>((float*)x, cls_w, classes, pad_class, per4, C, n4);
  else class_embed_add_kernel<bf16><<<(unsigned)blocks, 256, 0, st>>>((bf16*)x, cls_w, classes, pad_class, per4, C, n4);
  count_launch();
  DMN_LAUNCH_CHECK("class_embed_add");
  return 0;
}

// =====================================================================================================
// layout conversion (public-ABI boundary only; not on the loop's hot path)
// =====================================================================================================
template <typename T>
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ in, T* __restrict__ out, int C, int HW, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int c = (int)(i % C);
  const long bp = i / C;
  const int pix = (int)(bp % HW);
  const long b = bp / HW;
  out[i] = from_f<T>(in[(b * C + c) * HW + pix]);
}
template <typename T>
__global__ void nhwc_to_nchw_kernel(const T* __restrict__ in, float* __restrict__ out, int C, int HW, long total) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int pix = (int)(i % HW);
  const long bc = i / HW;
  const int c = (int)(bc % C);
  const long b = bc / C;
  out[i] = to_f<T>(in[(b * HW + pix) * C + c]);
}
int nchw_to_nhwc(const float* in, void* out, int B, int C, int HW, int act, cudaStream_t st) {
  const long total = (long)B * C * HW;
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (act == ACT_F32) nchw_to_nhwc_kernel<float><<<grid, 256, 0, st>>>(in, (float*)out, C, HW, total);
  else nchw_to_nhwc_kernel<bf16><<<grid, 256, 0, st>>>(in, (bf16*)out, C, HW, total);
  count_launch();
  DMN_LAUNCH_CHECK("nchw_to_nhwc");
  return 0;
}
int nhwc_to_nchw(const void* in, float* out, int B, int C, int HW, int act, cudaStream_t st) {
  const long total = (long)B * C * HW;
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (act == ACT_F32) nhwc_to_nchw_kernel<float><<<grid, 256, 0, st>>>((const float*)in, out, C, HW, total);
  else nhwc_to_nchw_kernel<bf16><<<grid, 256, 0, st>>>((const bf16*)in, out, C, HW, total);
  count_launch();
  DMN_LAUNCH_CHECK("nhwc_to_nchw");
  return 0;
}
__global__ void stats_to_mean_rstd_kernel(const stat_t* __restrict__ stats, float* __restrict__ out, int n, float inv_count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float mean, rstd;
  gn_mean_rstd(stats + 2 * i, inv_count, kGnEps, mean, rstd);
  out[2 * i] = mean;
  out[2 * i + 1] = rstd;
}
int stats_to_mean_rstd(const stat_t* stats, float* out, int n, float inv_count, cudaStream_t st) {
  stats_to_mean_rstd_kernel<<<(n + 127) / 128, 128, 0, st>>>(stats, out, n, inv_count);
  count_launch();
  DMN_LAUNCH_CHECK("stats_to_mean_rstd");
  return 0;
}

}  // namespace dmn

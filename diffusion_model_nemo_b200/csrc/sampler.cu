// sampler.cu -- the per-step posterior / score updates as single vectorised, coalesced elementwise kernels.
//
// Algorithmic traffic per element (fp32): read x, model output, z (parity mode) and write x  = 16 B;
// with in-kernel Philox noise = 12 B.  These kernels are HBM/launch bound (about 2 us at B = 256, 3x32x32).
#include "../../include/dmn_b200.h"
#include "common.cuh"
#include "ops.h"

namespace dmn {

// ---- Philox4x32-10, counter = (quad index lo, quad index hi, step word, stream id), key = seed ----------
struct Philox {
  __device__ static inline uint4 gen(uint64_t seed, uint64_t stream_id, uint32_t step_word, uint64_t quad) {
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint32_t c0 = (uint32_t)quad, c1 = (uint32_t)(quad >> 32), c2 = step_word, c3 = (uint32_t)stream_id ^ (uint32_t)(stream_id >> 32) * 0x9E3779B9u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
      c0 = n0; c1 = n1; c2 = n2; c3 = n3;
      k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
  __device__ static inline float4 normal4(uint64_t seed, uint64_t stream_id, uint32_t step_word, uint64_t quad) {
    const uint4 r = gen(seed, stream_id, step_word, quad);
    // Box-Muller on two pairs; u in (0,1]
    const float u0 = ((float)r.x + 1.0f) * 2.3283064365386963e-10f;
    const float u1 = (float)r.y * 2.3283064365386963e-10f;
    const float u2 = ((float)r.z + 1.0f) * 2.3283064365386963e-10f;
    const float u3 = (float)r.w * 2.3283064365386963e-10f;
    const float ra = sqrtf(-2.0f * __logf(u0)), rb = sqrtf(-2.0f * __logf(u2));
    float s0, c0, s1, c1;
    __sincosf(6.283185307179586f * u1, &s0, &c0);
    __sincosf(6.283185307179586f * u3, &s1, &c1);
    return make_float4(ra * c0, ra * s0, rb * c1, rb * s1);
  }
};

__device__ __forceinline__ const float* coef_row(const float* coef, const int32_t* step_dev, int step) {
  return coef + (long)(step_dev ? *step_dev : step) * DMN_COEF_STRIDE;
}
__device__ __forceinline__ uint32_t step_word(const int32_t* step_dev, int step, int draw) {
  return (uint32_t)((step_dev ? *step_dev : step) + 1) * 8u + (uint32_t)draw;
}
__device__ __forceinline__ dmn_rng pick_rng(const dmn_rng& by_value, const dmn_rng* dev) { return dev ? *dev : by_value; }
__device__ __forceinline__ float clamp1(float v) { return fminf(fmaxf(v, -1.0f), 1.0f); }

// generic 4-wide element loop helpers: n must be a multiple of 4 (C*H*W of images always is here; checked on host)

__global__ void __launch_bounds__(256) ddpm_step_kernel(const float* __restrict__ x, const float* __restrict__ eps,
                                                        const float* __restrict__ z, float* __restrict__ out, long n4,
                                                        const float* __restrict__ coef, const int32_t* step_dev, int step,
                                                        dmn_rng rng_v, const dmn_rng* rng_dev) {
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  const float* c = coef_row(coef, step_dev, step);
  const float c0 = c[0], c1 = c[1], c2 = c[2], c3 = c[3], c4 = c[4];
  const bool pred_x0 = c[5] != 0.f;
  const uint32_t sw = step_word(step_dev, step, 0);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 ev = reinterpret_cast<const float4*>(eps)[i];
    const float4 zv = z ? reinterpret_cast<const float4*>(z)[i] : Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
    float4 o;
#define DMN_DDPM(f)                                                    \
  {                                                                    \
    float x0 = pred_x0 ? ev.f : (c0 * xv.f - c1 * ev.f);               \
    x0 = clamp1(x0);                                                   \
    const float mean = c2 * x0 + c3 * xv.f;                            \
    o.f = mean + c4 * zv.f;                                            \
  }
    DMN_DDPM(x) DMN_DDPM(y) DMN_DDPM(z) DMN_DDPM(w)
#undef DMN_DDPM
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

__global__ void __launch_bounds__(256) learned_step_kernel(const float* __restrict__ x, const float* __restrict__ mo,
                                                           const float* __restrict__ z, float* __restrict__ out, long chw4,
                                                           long n4, const float* __restrict__ coef, const int32_t* step_dev,
                                                           int step, dmn_rng rng_v, const dmn_rng* rng_dev) {
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  const float* c = coef_row(coef, step_dev, step);
  const float c0 = c[0], c1 = c[1], c2 = c[2], c3 = c[3], mask = c[4], min_log = c[5], max_log = c[6];
  const uint32_t sw = step_word(step_dev, step, 0);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const long b = i / chw4, r = i - b * chw4;
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 ev = reinterpret_cast<const float4*>(mo)[b * 2 * chw4 + r];
    const float4 vv = reinterpret_cast<const float4*>(mo)[b * 2 * chw4 + chw4 + r];
    const float4 zv = z ? reinterpret_cast<const float4*>(z)[i] : Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
    float4 o;
#define DMN_LRN(f)                                                     \
  {                                                                    \
    const float frac = (vv.f + 1.0f) * 0.5f;                           \
    const float logvar = frac * max_log + (1.0f - frac) * min_log;     \
    float x0 = clamp1(c0 * xv.f - c1 * ev.f);                          \
    const float mean = c2 * x0 + c3 * xv.f;                            \
    o.f = mean + mask * expf(0.5f * logvar) * zv.f;                    \
  }
    DMN_LRN(x) DMN_LRN(y) DMN_LRN(z) DMN_LRN(w)
#undef DMN_LRN
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

__global__ void __launch_bounds__(256) ddim_step_kernel(const float* __restrict__ x, const float* __restrict__ eps,
                                                        const float* __restrict__ z, float* __restrict__ out, long n4,
                                                        const float* __restrict__ coef, const int32_t* step_dev, int step,
                                                        dmn_rng rng_v, const dmn_rng* rng_dev) {
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  // row: {sqrt(1-a_t), sqrt(a_t), sqrt(a_next), c1, c2, pred_x0}
  const float* c = coef_row(coef, step_dev, step);
  const float s1m = c[0], sa = c[1], san = c[2], k1 = c[3], k2 = c[4];
  const bool pred_x0 = c[5] != 0.f;
  const bool need_z = k1 != 0.f;
  const uint32_t sw = step_word(step_dev, step, 0);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 ev = reinterpret_cast<const float4*>(eps)[i];
    float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (z) zv = reinterpret_cast<const float4*>(z)[i];
    else if (need_z) zv = Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
    float4 o;
#define DMN_DDIM(f)                                                    \
  {                                                                    \
    float x0 = pred_x0 ? ev.f : (xv.f - ev.f * s1m) / sa;              \
    x0 = clamp1(x0);                                                   \
    o.f = san * x0 + k1 * zv.f + k2 * ev.f;                            \
  }
    DMN_DDIM(x) DMN_DDIM(y) DMN_DDIM(z) DMN_DDIM(w)
#undef DMN_DDIM
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

// DPM-Solver++ multistep (Lu et al. 2022): the update is affine in (x, m_i, m_{i-1}, m_{i-2}), m = data prediction.
// row: {c_x, c_0, c_1, c_2, k_x, k_m, slot, mode}.  mode (column 7): 0 = m = clamp(k_x x - k_m mo), 2 = the same without the clamp
// (score-SDE models), any other value = m = clamp(mo) (the output is the data prediction).  hist is a 3-slot ring [3][n]: slot = i mod 3
// receives m_i, (slot+2)%3 holds m_{i-1} and (slot+1)%3 holds m_{i-2}.  A slot whose coefficient is 0 is never read (the ring starts as
// uninitialised scratch).  The model output has `mo_chw4` float4 per sample (C or 2C channels); only the first chw4 of them are used.
// NOISE (SDE-DPM-Solver++): + g z with g = coef2 row[0], z injected or Philox draw 0 of the step word (the x_T draw uses word 0).
template <bool NOISE>
__global__ void __launch_bounds__(256) dpmpp_step_kernel(const float* x, const float* __restrict__ mo, float* __restrict__ hist,
                                                         float* out, long chw4, long mo_chw4, long n4, const float* __restrict__ coef,
                                                         const float* __restrict__ coef2, const float* __restrict__ z,
                                                         const int32_t* step_dev, int step, dmn_rng rng_v, const dmn_rng* rng_dev) {
  const float* c = coef_row(coef, step_dev, step);
  const float cx = c[0], c0 = c[1], c1 = c[2], c2 = c[3], kx = c[4], km = c[5];
  const int slot = (int)c[6];
  const bool pred_x0 = c[7] != 0.f && c[7] != 2.f;
  const bool clamp = c[7] != 2.f;
  float g = 0.f;
  uint32_t sw = 0;
  dmn_rng rng{};
  if (NOISE) {
    g = coef_row(coef2, step_dev, step)[0];
    sw = step_word(step_dev, step, 0);
    rng = pick_rng(rng_v, rng_dev);
  }
  float4* h_cur = reinterpret_cast<float4*>(hist) + (long)slot * n4;
  const float4* h_m1 = reinterpret_cast<const float4*>(hist) + (long)((slot + 2) % 3) * n4;
  const float4* h_m2 = reinterpret_cast<const float4*>(hist) + (long)((slot + 1) % 3) * n4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const long mi = mo_chw4 == chw4 ? i : (i / chw4) * mo_chw4 + i % chw4;
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 ev = reinterpret_cast<const float4*>(mo)[mi];
    float4 m, o;
#define DMN_DPM_M(f)                                         \
  {                                                          \
    const float raw = pred_x0 ? ev.f : (kx * xv.f - km * ev.f); \
    m.f = clamp ? clamp1(raw) : raw;                         \
    o.f = cx * xv.f + c0 * m.f;                              \
  }
    DMN_DPM_M(x) DMN_DPM_M(y) DMN_DPM_M(z) DMN_DPM_M(w)
#undef DMN_DPM_M
    if (c1 != 0.f) {
      const float4 h = h_m1[i];
      o.x += c1 * h.x; o.y += c1 * h.y; o.z += c1 * h.z; o.w += c1 * h.w;
    }
    if (c2 != 0.f) {
      const float4 h = h_m2[i];
      o.x += c2 * h.x; o.y += c2 * h.y; o.z += c2 * h.z; o.w += c2 * h.w;
    }
    if (NOISE) {
      const float4 zv = z ? reinterpret_cast<const float4*>(z)[i] : Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
      o.x += g * zv.x; o.y += g * zv.y; o.z += g * zv.z; o.w += g * zv.w;
    }
    h_cur[i] = m;
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

// RePaint inpainting (Lugmayr et al. 2022), run before the model at every event: the forward jump into this event and the merge of
// the noised known image.  row: {a_j, g_j, a_0, s_0}.
//   y = a_j x + g_j z2 ;  k = a_0 known + s_0 z1 ;  x' = m k + (1 - m) y
// z1 / z2 are draws 1 / 2 of the step word; each is drawn only when its coefficient is nonzero (uniform over the grid), so a row
// {1, 0, 1, 0} draws nothing and returns `known` exactly where m = 1 and x exactly where m = 0.
__global__ void __launch_bounds__(256) inpaint_prepare_kernel(const float* x, const float* __restrict__ known,
                                                              const float* __restrict__ mask, float* out, long n4,
                                                              const float* __restrict__ coef, const int32_t* step_dev, int step,
                                                              dmn_rng rng_v, const dmn_rng* rng_dev) {
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  const float* c = coef_row(coef, step_dev, step);
  const float aj = c[0], gj = c[1], a0 = c[2], s0 = c[3];
  const bool need_z1 = s0 != 0.f, need_z2 = gj != 0.f;
  const uint32_t sw1 = step_word(step_dev, step, 1), sw2 = step_word(step_dev, step, 2);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 kv = reinterpret_cast<const float4*>(known)[i];
    const float4 mv = reinterpret_cast<const float4*>(mask)[i];
    float4 z1 = make_float4(0.f, 0.f, 0.f, 0.f), z2 = z1;
    if (need_z1) z1 = Philox::normal4(rng.seed, rng.stream_id, sw1, (uint64_t)i);
    if (need_z2) z2 = Philox::normal4(rng.seed, rng.stream_id, sw2, (uint64_t)i);
    float4 o;
#define DMN_INP(f)                                                     \
  {                                                                    \
    const float y = aj * xv.f + gj * z2.f;                             \
    const float k = a0 * kv.f + s0 * z1.f;                             \
    o.f = mv.f * k + (1.0f - mv.f) * y;                                \
  }
    DMN_INP(x) DMN_INP(y) DMN_INP(z) DMN_INP(w)
#undef DMN_INP
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

__global__ void __launch_bounds__(256) affine_noise_kernel(const float* __restrict__ x, const float* __restrict__ mo,
                                                           const float* __restrict__ z, float* __restrict__ out,
                                                           float* __restrict__ mean_out, long n4, const float* __restrict__ coef,
                                                           const int32_t* step_dev, int step, int draw, dmn_rng rng_v, const dmn_rng* rng_dev) {
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  const float* c = coef_row(coef, step_dev, step);
  const float a = c[0], b = c[1], g = c[2];
  const uint32_t sw = step_word(step_dev, step, draw);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    const float4 mv = reinterpret_cast<const float4*>(mo)[i];
    const float4 zv = z ? reinterpret_cast<const float4*>(z)[i] : Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
    float4 m, o;
    m.x = a * xv.x + b * mv.x; m.y = a * xv.y + b * mv.y; m.z = a * xv.z + b * mv.z; m.w = a * xv.w + b * mv.w;
    o.x = m.x + g * zv.x; o.y = m.y + g * zv.y; o.z = m.z + g * zv.z; o.w = m.w + g * zv.w;
    if (mean_out) reinterpret_cast<float4*>(mean_out)[i] = m;
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

// Langevin: per-sample sums of squares of g = scale*model_out and z  -> ssq[b][2].  One block per sample adds its partials in a
// fixed order and writes ssq[b] itself (no float atomics), so the step size -- and the whole loop -- is bit-reproducible.
__global__ void __launch_bounds__(256) langevin_sumsq_kernel(const float* __restrict__ mo, const float* __restrict__ z,
                                                             float* __restrict__ ssq, long chw4, const float* __restrict__ coef,
                                                             const int32_t* step_dev, int step, int draw, dmn_rng rng_v, const dmn_rng* rng_dev) {
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  __shared__ float red[2][8];
  const int b = blockIdx.x;
  const float scale = coef_row(coef, step_dev, step)[0];
  const uint32_t sw = step_word(step_dev, step, draw);
  float sg = 0.f, sz = 0.f;
  for (long r = threadIdx.x; r < chw4; r += blockDim.x) {
    const long i = (long)b * chw4 + r;
    float4 g = reinterpret_cast<const float4*>(mo)[i];
    g.x *= scale; g.y *= scale; g.z *= scale; g.w *= scale;
    const float4 zv = z ? reinterpret_cast<const float4*>(z)[i] : Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
    sg += g.x * g.x + g.y * g.y + g.z * g.z + g.w * g.w;
    sz += zv.x * zv.x + zv.y * zv.y + zv.z * zv.z + zv.w * zv.w;
  }
  sg = warp_sum(sg);
  sz = warp_sum(sz);
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][w] = sg; red[1][w] = sz; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float a = 0.f, c = 0.f;
    for (int i = 0; i < 8; ++i) { a += red[0][i]; c += red[1][i]; }
    ssq[2 * b] = a;
    ssq[2 * b + 1] = c;
  }
}
// batch means of the per-sample norms  -> means[0] = mean ||g_b||, means[1] = mean ||z_b||
__global__ void langevin_means_kernel(const float* __restrict__ ssq, float* __restrict__ means, int B) {
  float a = 0.f, c = 0.f;
  for (int b = threadIdx.x; b < B; b += 32) { a += sqrtf(ssq[2 * b]); c += sqrtf(ssq[2 * b + 1]); }
  a = warp_sum(a);
  c = warp_sum(c);
  if (threadIdx.x == 0) { means[0] = a / (float)B; means[1] = c / (float)B; }
}
__global__ void __launch_bounds__(256) langevin_apply_kernel(const float* __restrict__ x, const float* __restrict__ mo,
                                                             const float* __restrict__ z, float* __restrict__ out,
                                                             float* __restrict__ mean_out, long n4, float snr,
                                                             const float* __restrict__ means, const float* __restrict__ coef,
                                                             const int32_t* step_dev, int step, int draw, dmn_rng rng_v, const dmn_rng* rng_dev) {
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  const float* c = coef_row(coef, step_dev, step);
  const float scale = c[0], alpha = c[1];
  const float ratio = snr * means[1] / means[0];
  const float ss = ratio * ratio * 2.0f * alpha;
  const float nz = sqrtf(ss * 2.0f);
  const uint32_t sw = step_word(step_dev, step, draw);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 xv = reinterpret_cast<const float4*>(x)[i];
    float4 g = reinterpret_cast<const float4*>(mo)[i];
    g.x *= scale; g.y *= scale; g.z *= scale; g.w *= scale;
    const float4 zv = z ? reinterpret_cast<const float4*>(z)[i] : Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
    float4 m, o;
    m.x = xv.x + ss * g.x; m.y = xv.y + ss * g.y; m.z = xv.z + ss * g.z; m.w = xv.w + ss * g.w;
    o.x = m.x + nz * zv.x; o.y = m.y + nz * zv.y; o.z = m.z + nz * zv.z; o.w = m.w + nz * zv.w;
    if (mean_out) reinterpret_cast<float4*>(mean_out)[i] = m;
    reinterpret_cast<float4*>(out)[i] = o;
  }
}

__global__ void __launch_bounds__(256) unnormalize_kernel(const float* __restrict__ x, float* __restrict__ out, long n) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    out[i] = (x[i] + 1.0f) * 0.5f;
}
__global__ void __launch_bounds__(256) axpby_kernel(const float* __restrict__ x, const float* __restrict__ y, float a, float b,
                                                    float* __restrict__ out, long n) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x)
    out[i] = a * x[i] + b * y[i];
}
__global__ void __launch_bounds__(256) randn_kernel(float* __restrict__ out, long n4, dmn_rng rng, uint32_t sw) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x)
    reinterpret_cast<float4*>(out)[i] = Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
}
__global__ void advance_counter_kernel(int32_t* c) { *c += 1; }
// loop state: int32 step counter at [0], block ticket of the fused tail at [1], dmn_rng at byte offset 16
__global__ void set_counter_kernel(int32_t* c, int v, dmn_rng rng) {
  c[0] = v;
  c[1] = 0;
  *reinterpret_cast<dmn_rng*>(c + 4) = rng;
}

// =====================================================================================================
// Fused tail of one DDPM step (SURVEY section 8(f) rank 2; reference modules/unet.py:109-116 + gaussian_diffusion.py:118-167):
//   eps = conv1x1(SiLU(GroupNorm(y)))   (final_conv tail)   ->   x0 prediction, clamp, posterior mean, + sigma_t * z   ->   x_{t-1}
// and the step counter of the loop.  The model output never reaches global memory.  One block = 128 pixels of one sample: the
// projection is the staged bf16 path of final_proj_bf16_kernel (kernels_simt.cu), eps goes through shared memory to 3 x 32 threads
// that each update 4 consecutive pixels of one channel with the SAME Philox quads ddpm_step_kernel draws (bit-identical results).
// =====================================================================================================
template <int COUT>
__global__ void __launch_bounds__(128) final_proj_ddpm_kernel(const FinalProjP p, const float* __restrict__ x, const float* __restrict__ z,
                                                              float* __restrict__ xout, const float* __restrict__ coef, const int32_t* step_dev,
                                                              int step, dmn_rng rng_v, const dmn_rng* rng_dev, int32_t* advance) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) unsigned char fsmb[];
  const int C = p.C, ld = C * 2 + 16;                       // bytes per staged pixel row
  float* s_sc = reinterpret_cast<float*>(fsmb);             // [C] rstd*gamma
  float* s_sh = s_sc + C;                                   // [C] beta - mean*rstd*gamma
  float* s_w = s_sh + C;                                    // [COUT][C]
  float* s_eps = s_w + COUT * C;                            // [COUT][128]
  unsigned char* s_tile = fsmb + (size_t)(2 + COUT) * C * 4 + (size_t)COUT * 128 * 4;
  const int b = blockIdx.y, pix0 = blockIdx.x * 128;
  const int npix = min(128, p.HW - pix0);
  {
    const bf16* y = (const bf16*)p.y + ((long)b * p.HW + pix0) * C;
    const int chunks = C / 8;
    const uint32_t tile_u = (uint32_t)__cvta_generic_to_shared(s_tile);
    for (int i = threadIdx.x; i < npix * chunks; i += 128) {
      const int r = i / chunks, c16 = i - r * chunks;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(tile_u + (uint32_t)(r * ld + c16 * 16)), "l"(y + (long)r * C + c16 * 8) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  const float* cr = coef_row(coef, step_dev, step);
  const float c0 = cr[0], c1 = cr[1], c2 = cr[2], c3 = cr[3], c4 = cr[4];
  const bool pred_x0 = cr[5] != 0.f;
  const uint32_t sw = step_word(step_dev, step, 0);
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
  if ((int)threadIdx.x < npix) {
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
    for (int j = 0; j < COUT; ++j) s_eps[j * 128 + threadIdx.x] = acc[j] + (p.bias ? p.bias[j] : 0.f);
  }
  __syncthreads();
  // ---- posterior update: thread u -> channel u / 32, pixels pix0 + 4 * (u % 32) .. + 3 ----
  if ((int)threadIdx.x < COUT * 32) {
    const int j = threadIdx.x >> 5, g4 = threadIdx.x & 31;
    if (4 * g4 < npix) {
      const long e0 = ((long)b * COUT + j) * p.HW + pix0 + 4 * g4;      // first element (HW and pix0 are multiples of 4)
      const long i = e0 >> 2;                                            // the Philox quad ddpm_step_kernel uses for these 4 elements
      const float4 xv = reinterpret_cast<const float4*>(x)[i];
      const float4 ev = *reinterpret_cast<const float4*>(s_eps + j * 128 + 4 * g4);
      const float4 zv = z ? reinterpret_cast<const float4*>(z)[i] : Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
      float4 o;
#define DMN_DDPM(f)                                                    \
  {                                                                    \
    float x0 = pred_x0 ? ev.f : (c0 * xv.f - c1 * ev.f);               \
    x0 = clamp1(x0);                                                   \
    const float mean = c2 * x0 + c3 * xv.f;                            \
    o.f = mean + c4 * zv.f;                                            \
  }
      DMN_DDPM(x) DMN_DDPM(y) DMN_DDPM(z) DMN_DDPM(w)
#undef DMN_DDPM
      reinterpret_cast<float4*>(xout)[i] = o;
    }
  }
  // ---- step counter: the last block to finish advances it (every block has read the step index above) ----
  if (advance) {
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      const int total = (int)(gridDim.x * gridDim.y);
      if (atomicAdd(advance + 1, 1) == total - 1) {
        advance[1] = 0;
        advance[0] += 1;
      }
    }
  }
}
// copy every `every`-th step's state into the trajectory buffer (device-side decision => graph friendly)
__global__ void __launch_bounds__(256) traj_kernel(const float* __restrict__ x, float* __restrict__ traj, long n4,
                                                   const int32_t* step_dev, int every, int n_steps) {
  const int s = *step_dev;
  if (((s + 1) % every) != 0 || s >= n_steps) return;
  const long slot = (long)((s + 1) / every - 1);
  float4* dst = reinterpret_cast<float4*>(traj) + slot * n4;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x)
    dst[i] = reinterpret_cast<const float4*>(x)[i];
}

// classifier-free guidance helpers (doubled batch): x2 = [x ; x],  eps = eps_u + w (eps_c - eps_u) with mo2 = [eps_c ; eps_u]
__global__ void __launch_bounds__(256) cfg_dup_kernel(const float* __restrict__ x, float* __restrict__ x2, long n4) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    reinterpret_cast<float4*>(x2)[i] = v;
    reinterpret_cast<float4*>(x2)[n4 + i] = v;
  }
}
// per sample the first `guided4` float4 (the eps channels) are mixed; the rest (learned-variance channels) are the conditional branch's
__global__ void __launch_bounds__(256) cfg_combine_kernel(const float* __restrict__ mo2, float* __restrict__ mo, long n4, long per4, long guided4,
                                                          float w) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 c = reinterpret_cast<const float4*>(mo2)[i];
    float4 o = c;
    if (i % per4 < guided4) {
      const float4 u = reinterpret_cast<const float4*>(mo2)[n4 + i];
      o.x = u.x + w * (c.x - u.x); o.y = u.y + w * (c.y - u.y); o.z = u.z + w * (c.z - u.z); o.w = u.w + w * (c.w - u.w);
    }
    reinterpret_cast<float4*>(mo)[i] = o;
  }
}

// ---- bits-per-dimension evaluation (models/abstract_diffusion_model.py:137-197) ------------------------------------------
// q_sample (gaussian_diffusion.py:104-116): x_t = sqrt_ac[t] * x0 + sqrt_1m_ac[t] * z.  coef row columns 6 / 7.
__global__ void __launch_bounds__(256) bpd_qsample_kernel(const float* __restrict__ x0, const float* __restrict__ z, float* __restrict__ xt,
                                                          long n4, const float* __restrict__ coef, const int32_t* step_dev, int step,
                                                          dmn_rng rng_v, const dmn_rng* rng_dev) {
  const dmn_rng rng = pick_rng(rng_v, rng_dev);
  const float* c = coef_row(coef, step_dev, step);
  const float a = c[6], b = c[7];
  const uint32_t sw = step_word(step_dev, step, 0);
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long)gridDim.x * blockDim.x) {
    const float4 xv = reinterpret_cast<const float4*>(x0)[i];
    const float4 zv = z ? reinterpret_cast<const float4*>(z)[i] : Philox::normal4(rng.seed, rng.stream_id, sw, (uint64_t)i);
    reinterpret_cast<float4*>(xt)[i] = make_float4(a * xv.x + b * zv.x, a * xv.y + b * zv.y, a * xv.z + b * zv.z, a * xv.w + b * zv.w);
  }
}

__device__ __forceinline__ float approx_std_normal_cdf(float x) {      // utils.py:37-38
  return 0.5f * (1.0f + tanhf(0.7978845608028654f * (x + 0.044715f * (x * x * x))));
}
// One variational-bound term per sample (loss/variational_bound_loss.py:31-52 on top of q_posterior / p_mean_variance,
// gaussian_diffusion.py:91-101,125-154; learned variance: learned_gaussian_diffusion.py:27-53):
//   t > 0 : mean_chw KL( q(x_{t-1} | x_t, x_0) || p(x_{t-1} | x_t) ) / ln 2        t == 0 : mean_chw decoder NLL / ln 2
// One block per sample, fixed reduction order (deterministic).  coef row = {sqrt_recip_ac, sqrt_recipm1_ac, post_coef1, post_coef2,
// post_logvar_clipped, pred_x0 flag, sqrt_ac, sqrt_1m_ac}; coef2 row = {log beta_t (learned max log variance), t, is_t0}.
// mode 1 = prior term: mean_chw KL( q(x_T | x_0) || N(0, 1) ) / ln 2 with coef2 row = {log(1 - ac_T)}, coef column 6 = sqrt_ac_T.
__global__ void __launch_bounds__(256) bpd_term_kernel(const float* __restrict__ x0, const float* __restrict__ xt, const float* __restrict__ mo,
                                                       float* __restrict__ terms, long chw, int learned, int n_cols, int mode,
                                                       const float* __restrict__ coef, const float* __restrict__ coef2,
                                                       const int32_t* step_dev, int step) {
  const int b = blockIdx.x;
  const float* c = coef_row(coef, step_dev, step);
  const float* c2 = coef2 + (long)(step_dev ? *step_dev : step) * DMN_COEF_STRIDE;
  const float c0 = c[0], c1 = c[1], p1 = c[2], p2 = c[3], lv_true = c[4];
  const bool pred_x0 = c[5] != 0.f;
  const float max_log = c2[0];
  const int col = (int)c2[1];
  const bool t0 = c2[2] != 0.f;
  const float* xs = x0 + (long)b * chw;
  float acc = 0.f;
  if (mode == 1) {
    const float a = c[6], lv1 = c2[0];
    for (long i = threadIdx.x; i < chw; i += blockDim.x) {
      const float m1 = xs[i] * a;
      acc += 0.5f * (-1.0f + 0.0f - lv1 + expf(lv1 - 0.0f) + (m1 * m1) * expf(-0.0f));
    }
  } else {
    const float* xts = xt + (long)b * chw;
    const float* eps = mo + (long)b * chw * (learned ? 2 : 1);
    for (long i = threadIdx.x; i < chw; i += blockDim.x) {
      const float xv = xs[i], xtv = xts[i], ev = eps[i];
      float lv = lv_true;
      if (learned) {
        const float frac = (eps[chw + i] + 1.0f) * 0.5f;
        lv = frac * max_log + (1.0f - frac) * lv_true;
      }
      float x0p = pred_x0 ? ev : (c0 * xtv - c1 * ev);
      x0p = clamp1(x0p);
      const float mm = p1 * x0p + p2 * xtv;      // model mean
      const float tm = p1 * xv + p2 * xtv;       // true posterior mean
      float v;
      if (!t0) {
        const float d = tm - mm;
        v = 0.5f * (-1.0f + lv - lv_true + expf(lv_true - lv) + (d * d) * expf(-lv));      // utils.normal_kl
      } else {                                                                                // utils.discretized_gaussian_log_likelihood
        const float centered = xv - mm, inv_stdv = expf(-0.5f * lv);
        const float cdf_plus = approx_std_normal_cdf(inv_stdv * (centered + 1.0f / 255.0f));
        const float cdf_min = approx_std_normal_cdf(inv_stdv * (centered - 1.0f / 255.0f));
        const float lp = xv < -0.999f ? logf(fmaxf(cdf_plus, 1e-12f))
                                      : (xv > 0.999f ? logf(fmaxf(1.0f - cdf_min, 1e-12f)) : logf(fmaxf(cdf_plus - cdf_min, 1e-12f)));
        v = -lp;
      }
      acc += v;
    }
  }
  __shared__ float red[8];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    const float val = t / (float)chw * 1.4426950408889634f;       // mean over C*H*W, in bits
    if (mode == 1) terms[b] = val;
    else terms[(long)b * n_cols + col] = val;
  }
}

static inline unsigned grid_for(long n, int per_block = 256, int cap = 148 * 8) {
  long g = (n + per_block - 1) / per_block;
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (unsigned)g;
}

int launch_advance_counter(int32_t* c, cudaStream_t st) {
  advance_counter_kernel<<<1, 1, 0, st>>>(c);
  count_launch();
  DMN_LAUNCH_CHECK("advance_counter");
  return 0;
}
int launch_set_counter(int32_t* c, int v, dmn_rng rng, cudaStream_t st) {
  set_counter_kernel<<<1, 1, 0, st>>>(c, v, rng);
  count_launch();
  DMN_LAUNCH_CHECK("set_counter");
  return 0;
}
int launch_cfg_dup(const float* x, float* x2, long n, cudaStream_t st) {
  cfg_dup_kernel<<<grid_for(n / 4), 256, 0, st>>>(x, x2, n / 4);
  count_launch();
  DMN_LAUNCH_CHECK("cfg_dup");
  return 0;
}
int launch_cfg_combine(const float* mo2, float* mo, long n, long per_sample, long guided, float w, cudaStream_t st) {
  DMN_REQUIRE(per_sample % 4 == 0 && guided % 4 == 0, "cfg_combine: per-sample sizes must be multiples of 4");
  cfg_combine_kernel<<<grid_for(n / 4), 256, 0, st>>>(mo2, mo, n / 4, per_sample / 4, guided / 4, w);
  count_launch();
  DMN_LAUNCH_CHECK("cfg_combine");
  return 0;
}
int launch_traj(const float* x, float* traj, long n, const int32_t* step_dev, int every, int n_steps, cudaStream_t st) {
  traj_kernel<<<grid_for(n / 4), 256, 0, st>>>(x, traj, n / 4, step_dev, every, n_steps);
  count_launch();
  DMN_LAUNCH_CHECK("traj");
  return 0;
}
int launch_langevin(const float* x, const float* mo, const float* z, float* out, float* mean_out, int batch, long chw,
                    float snr, const float* coef, const int32_t* step_dev, int step, int draw, float* scratch, dmn_rng rng,
                    const dmn_rng* rng_dev, cudaStream_t st) {
  DMN_REQUIRE(chw % 4 == 0, "langevin: C*H*W must be a multiple of 4");
  float* ssq = scratch;                 // [batch][2]
  float* means = scratch + 2 * batch;   // [2]
  langevin_sumsq_kernel<<<batch, 256, 0, st>>>(mo, z, ssq, chw / 4, coef, step_dev, step, draw, rng, rng_dev);
  count_launch();
  DMN_LAUNCH_CHECK("langevin_sumsq");
  langevin_means_kernel<<<1, 32, 0, st>>>(ssq, means, batch);
  count_launch();
  DMN_LAUNCH_CHECK("langevin_means");
  const long n4 = (long)batch * chw / 4;
  langevin_apply_kernel<<<grid_for(n4), 256, 0, st>>>(x, mo, z, out, mean_out, n4, snr, means, coef, step_dev, step, draw, rng,
                                                      rng_dev);
  count_launch();
  DMN_LAUNCH_CHECK("langevin_apply");
  return 0;
}
int launch_affine_noise(const float* x, const float* mo, const float* z, float* out, float* mean_out, long n, const float* coef,
                        const int32_t* step_dev, int step, int draw, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st) {
  DMN_REQUIRE(n % 4 == 0, "affine_noise: element count must be a multiple of 4");
  affine_noise_kernel<<<grid_for(n / 4), 256, 0, st>>>(x, mo, z, out, mean_out, n / 4, coef, step_dev, step, draw, rng, rng_dev);
  count_launch();
  DMN_LAUNCH_CHECK("affine_noise");
  return 0;
}

int launch_ddpm(const float* x, const float* eps, const float* z, float* out, long n, const float* coef, const int32_t* step_dev,
                int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st) {
  DMN_REQUIRE(n % 4 == 0 && n > 0, "ddpm_step: element count must be a positive multiple of 4");
  ddpm_step_kernel<<<grid_for(n / 4), 256, 0, st>>>(x, eps, z, out, n / 4, coef, step_dev, step, rng, rng_dev);
  count_launch();
  DMN_LAUNCH_CHECK("ddpm_step");
  return 0;
}
bool fused_tail_supported(const FinalProjP& p, int act) {
  const size_t smem = (size_t)(2 + p.Cout) * p.C * 4 + (size_t)p.Cout * 128 * 4 + (size_t)128 * (p.C * 2 + 16);
  return act == ACT_BF16 && p.C % 8 == 0 && (p.Cout == 3 || p.Cout == 1) && p.HW % 4 == 0 && smem <= 200 * 1024;
}
// eps = final_conv tail (never stored) + DDPM update + (optionally) the loop's step counter, one launch
int launch_final_proj_ddpm(const FinalProjP& p, const float* x, const float* z, float* out, const float* coef, const int32_t* step_dev,
                           int step, dmn_rng rng, const dmn_rng* rng_dev, int32_t* advance, cudaStream_t st) {
  const size_t smem = (size_t)(2 + p.Cout) * p.C * 4 + (size_t)p.Cout * 128 * 4 + (size_t)128 * (p.C * 2 + 16);
  static DeviceOnce attr;
  if (attr.first()) {
    DMN_CUDA_CHECK(cudaFuncSetAttribute(final_proj_ddpm_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    DMN_CUDA_CHECK(cudaFuncSetAttribute(final_proj_ddpm_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  dim3 grid((unsigned)((p.HW + 127) / 128), (unsigned)p.B);
  if (p.Cout == 3) DMN_CUDA_CHECK(launch_pdl(final_proj_ddpm_kernel<3>, grid, dim3(128), smem, st, p, x, z, out, coef, step_dev, step, rng, rng_dev, advance));
  else DMN_CUDA_CHECK(launch_pdl(final_proj_ddpm_kernel<1>, grid, dim3(128), smem, st, p, x, z, out, coef, step_dev, step, rng, rng_dev, advance));
  count_launch();
  DMN_LAUNCH_CHECK("final_proj_ddpm");
  return 0;
}

int launch_learned(const float* x, const float* mo, const float* z, float* out, int batch, long chw, const float* coef,
                   const int32_t* step_dev, int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st) {
  DMN_REQUIRE(chw % 4 == 0 && chw > 0 && batch > 0, "learned_step: C*H*W must be a positive multiple of 4");
  const long n4 = (long)batch * chw / 4;
  learned_step_kernel<<<grid_for(n4), 256, 0, st>>>(x, mo, z, out, chw / 4, n4, coef, step_dev, step, rng, rng_dev);
  count_launch();
  DMN_LAUNCH_CHECK("learned_step");
  return 0;
}
int launch_bpd_qsample(const float* x0, const float* z, float* xt, long n, const float* coef, const int32_t* step_dev, int step,
                       dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st) {
  DMN_REQUIRE(n % 4 == 0 && n > 0, "bpd_qsample: element count must be a positive multiple of 4");
  bpd_qsample_kernel<<<grid_for(n / 4), 256, 0, st>>>(x0, z, xt, n / 4, coef, step_dev, step, rng, rng_dev);
  count_launch();
  DMN_LAUNCH_CHECK("bpd_qsample");
  return 0;
}
int launch_bpd_term(const float* x0, const float* xt, const float* mo, float* terms, int batch, long chw, int learned, int n_cols,
                    int mode, const float* coef, const float* coef2, const int32_t* step_dev, int step, cudaStream_t st) {
  DMN_REQUIRE(batch > 0 && chw > 0 && coef && coef2 && terms && x0, "bpd_term: bad arguments");
  bpd_term_kernel<<<batch, 256, 0, st>>>(x0, xt, mo, terms, chw, learned, n_cols, mode, coef, coef2, step_dev, step);
  count_launch();
  DMN_LAUNCH_CHECK("bpd_term");
  return 0;
}
int launch_ddim(const float* x, const float* eps, const float* z, float* out, long n, const float* coef, const int32_t* step_dev,
                int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st) {
  DMN_REQUIRE(n % 4 == 0 && n > 0, "ddim_step: element count must be a positive multiple of 4");
  ddim_step_kernel<<<grid_for(n / 4), 256, 0, st>>>(x, eps, z, out, n / 4, coef, step_dev, step, rng, rng_dev);
  count_launch();
  DMN_LAUNCH_CHECK("ddim_step");
  return 0;
}
int launch_dpmpp(const float* x, const float* mo, float* hist, float* out, int batch, long chw, long mo_chw, const float* coef,
                 const float* coef2, const float* z, const int32_t* step_dev, int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st) {
  DMN_REQUIRE(batch > 0 && chw > 0 && chw % 4 == 0 && mo_chw >= chw && mo_chw % 4 == 0,
              "dpmpp_step: C*H*W must be a positive multiple of 4 and the model output at least C*H*W per sample");
  DMN_REQUIRE(x && mo && hist && out && coef, "dpmpp_step: null pointer");
  const long n4 = (long)batch * chw / 4;
  if (coef2)
    dpmpp_step_kernel<true><<<grid_for(n4), 256, 0, st>>>(x, mo, hist, out, chw / 4, mo_chw / 4, n4, coef, coef2, z, step_dev, step, rng,
                                                          rng_dev);
  else
    dpmpp_step_kernel<false><<<grid_for(n4), 256, 0, st>>>(x, mo, hist, out, chw / 4, mo_chw / 4, n4, coef, nullptr, nullptr, step_dev,
                                                           step, rng, nullptr);
  count_launch();
  DMN_LAUNCH_CHECK("dpmpp_step");
  return 0;
}
int launch_inpaint_prepare(const float* x, const float* known, const float* mask, float* out, long n, const float* coef,
                           const int32_t* step_dev, int step, dmn_rng rng, const dmn_rng* rng_dev, cudaStream_t st) {
  DMN_REQUIRE(n % 4 == 0 && n > 0, "inpaint_prepare: element count must be a positive multiple of 4");
  DMN_REQUIRE(x && known && mask && out && coef, "inpaint_prepare: null pointer");
  inpaint_prepare_kernel<<<grid_for(n / 4), 256, 0, st>>>(x, known, mask, out, n / 4, coef, step_dev, step, rng, rng_dev);
  count_launch();
  DMN_LAUNCH_CHECK("inpaint_prepare");
  return 0;
}

}  // namespace dmn

using namespace dmn;

extern "C" {

int dmn_ddpm_step(const float* x, const float* eps, const float* z_dev, float* x_out, int64_t n, const float* coef_dev,
                  const int32_t* step_dev, int step, dmn_rng rng, void* stream) {
  return launch_ddpm(x, eps, z_dev, x_out, n, coef_dev, step_dev, step, rng, nullptr, (cudaStream_t)stream);
}

int dmn_learned_step(const float* x, const float* model_out, const float* z_dev, float* x_out, int batch, int64_t chw,
                     const float* coef_dev, const int32_t* step_dev, int step, dmn_rng rng, void* stream) {
  return launch_learned(x, model_out, z_dev, x_out, batch, chw, coef_dev, step_dev, step, rng, nullptr, (cudaStream_t)stream);
}

int dmn_ddim_step(const float* x, const float* eps, const float* z_dev, float* x_out, int64_t n, const float* coef_dev,
                  const int32_t* step_dev, int step, dmn_rng rng, void* stream) {
  return launch_ddim(x, eps, z_dev, x_out, n, coef_dev, step_dev, step, rng, nullptr, (cudaStream_t)stream);
}

int dmn_dpmpp_step(const float* x, const float* model_out, float* hist, float* x_out, int batch, int64_t chw, int64_t mo_chw,
                   const float* coef_dev, const int32_t* step_dev, int step, void* stream) {
  return launch_dpmpp(x, model_out, hist, x_out, batch, chw, mo_chw, coef_dev, nullptr, nullptr, step_dev, step, dmn_rng{}, nullptr,
                      (cudaStream_t)stream);
}

int dmn_dpmpp_sde_step(const float* x, const float* model_out, const float* z_dev, float* hist, float* x_out, int batch, int64_t chw,
                       int64_t mo_chw, const float* coef_dev, const float* coef2_dev, const int32_t* step_dev, int step, dmn_rng rng,
                       void* stream) {
  DMN_REQUIRE(coef2_dev, "dpmpp_sde_step: null noise-weight table");
  return launch_dpmpp(x, model_out, hist, x_out, batch, chw, mo_chw, coef_dev, coef2_dev, z_dev, step_dev, step, rng, nullptr,
                      (cudaStream_t)stream);
}

int dmn_inpaint_prepare(const float* x, const float* known, const float* mask, float* x_out, int64_t n, const float* coef_dev,
                        const int32_t* step_dev, int step, dmn_rng rng, void* stream) {
  return launch_inpaint_prepare(x, known, mask, x_out, n, coef_dev, step_dev, step, rng, nullptr, (cudaStream_t)stream);
}

int dmn_affine_noise_step(const float* x, const float* model_out, const float* z_dev, float* x_out, float* x_mean_out, int64_t n,
                          const float* coef_dev, const int32_t* step_dev, int step, dmn_rng rng, void* stream) {
  return launch_affine_noise(x, model_out, z_dev, x_out, x_mean_out, n, coef_dev, step_dev, step, 7, rng, nullptr,
                             (cudaStream_t)stream);
}

int dmn_langevin_step(const float* x, const float* model_out, const float* z_dev, float* x_out, float* x_mean_out, int batch,
                      int64_t chw, float snr, const float* coef_dev, const int32_t* step_dev, int step, float* scratch_dev,
                      dmn_rng rng, void* stream) {
  return launch_langevin(x, model_out, z_dev, x_out, x_mean_out, batch, chw, snr, coef_dev, step_dev, step, 0, scratch_dev, rng,
                         nullptr, (cudaStream_t)stream);
}

int dmn_bpd_qsample(const float* x0, const float* z_dev, float* x_t, int64_t n, const float* coef_dev, const int32_t* step_dev, int step,
                    dmn_rng rng, void* stream) {
  return launch_bpd_qsample(x0, z_dev, x_t, n, coef_dev, step_dev, step, rng, nullptr, (cudaStream_t)stream);
}
int dmn_bpd_term(const float* x0, const float* x_t, const float* model_out, float* terms, int batch, int64_t chw, int learned, int n_cols,
                 int mode, const float* coef_dev, const float* coef2_dev, const int32_t* step_dev, int step, void* stream) {
  return launch_bpd_term(x0, x_t, model_out, terms, batch, chw, learned, n_cols, mode, coef_dev, coef2_dev, step_dev, step,
                         (cudaStream_t)stream);
}

int dmn_unnormalize(const float* x, float* out, int64_t n, void* stream) {
  unnormalize_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(x, out, n);
  count_launch();
  DMN_LAUNCH_CHECK("unnormalize");
  return 0;
}

int dmn_randn(float* out, int64_t n, dmn_rng rng, int step, void* stream) {
  DMN_REQUIRE(n % 4 == 0 && n > 0, "randn: element count must be a positive multiple of 4");
  randn_kernel<<<grid_for(n / 4), 256, 0, (cudaStream_t)stream>>>(out, n / 4, rng, (uint32_t)(step + 1) * 8u);
  count_launch();
  DMN_LAUNCH_CHECK("randn");
  return 0;
}

int dmn_axpby(const float* x, const float* y, float a, float b, float* out, int64_t n, void* stream) {
  axpby_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(x, y, a, b, out, n);
  count_launch();
  DMN_LAUNCH_CHECK("axpby");
  return 0;
}

}  // extern "C"

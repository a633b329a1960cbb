// ode.cu -- probability-flow ODE sampling: scipy.integrate.RK45 (Dormand-Prince 5(4), FSAL) with the whole step control on the
// device, so a solve runs as one CUDA graph (init phase + a WHILE conditional node over attempts) without host round trips.
//
// What is reproduced (scipy/integrate/_ivp/rk.py, common.py, base.py):
//   select_initial_step (d0 / d1 / d2, h0, h1), rk_step (stages, y_new, f_new), the error norm RMS(h * K^T E / scale) with
//   scale = atol + max(|y|, |y_new|) * rtol, SAFETY 0.9 / MIN_FACTOR 0.2 / MAX_FACTOR 10 / exponent -1/5, the growth cap after a
//   rejection, min_step = 10 * |nextafter(t, direction * inf) - t| (TOO_SMALL_STEP) and the clip of the last step onto t_bound.
// y / y_new are fp64; the stage rows K hold fp32 drifts (scipy's K rows are float64 but only ever hold fp32 drifts, so fp32
// storage is lossless).  The drift is the reference's reverse-SDE algebra with probability_flow=True in its fp32 op order
// (score_sde sde_lib.py reverse(); VP: f = -0.5 beta(t) x, score = -model / std(t); VE: f = 0, score = model):
//   drift = f(x, t) - (g(t)^2 * score) * 0.5
// written with explicit round-to-nearest intrinsics so no FMA contraction changes it.
//
// Launches of one attempt: stage 0 (input of stage 1), dmn_time_table (6 rows), then 6 x (U-Net, stage s), then the controller.
// Reductions (error norm, select_initial_step norms) are fixed-order: per-block fp64 partials over a grid that depends only on the
// element count, summed by one block in a fixed order, so a solve is bit-reproducible run to run and graph == plain launches.
#include "../../include/dmn_b200.h"
#include "common.cuh"
#include "ops.h"

namespace dmn {
namespace ode {

// RK45 tableau, the same double literals as scipy's rk.py
__constant__ double kA[6][5] = {
    {0, 0, 0, 0, 0},
    {1.0 / 5, 0, 0, 0, 0},
    {3.0 / 40, 9.0 / 40, 0, 0, 0},
    {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
    {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
    {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};
__constant__ double kB[6] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
__constant__ double kE[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};
__constant__ double kC[7] = {0, 1.0 / 5, 3.0 / 10, 4.0 / 5, 8.0 / 9, 1.0, 1.0};

constexpr int kThreads = 256;

// fp32 scalars of one evaluation at time t, in the reference's torch op order (vec_t = ones(B) * t is fp32)
__device__ void stage_scalars(const OdeParams& P, double t, float& label, float& fx, float& sc, float& g2) {
  const float vt = __double2float_rn(t);
  if (P.sde_kind == DMN_SDE_VP) {
    const float bt = __fadd_rn(__fmul_rn(vt, (float)(P.beta_1 - P.beta_0)), (float)P.beta_0);   // beta_0 + t * (beta_1 - beta_0)
    const float g = __fsqrt_rn(bt);
    fx = __fmul_rn(-0.5f, bt);
    g2 = __fmul_rn(g, g);
    const float lmc = __fsub_rn(__fmul_rn(__fmul_rn(-0.25f, __fmul_rn(vt, vt)), (float)(P.beta_1 - P.beta_0)),
                                __fmul_rn(__fmul_rn(0.5f, vt), (float)P.beta_0));
    sc = __fsqrt_rn(__fsub_rn(1.0f, expf(__fmul_rn(2.0f, lmc))));      // std(t); score = -model / std
    label = __fmul_rn(vt, (float)(P.N - 1));
  } else {
    const float sigma = __fmul_rn((float)P.sigma_min, powf((float)(P.sigma_max / P.sigma_min), vt));
    const float g = __fmul_rn(sigma, __fsqrt_rn((float)(2.0 * (log(P.sigma_max) - log(P.sigma_min)))));
    fx = 0.f;
    g2 = __fmul_rn(g, g);
    sc = 1.f;
    label = sigma;
  }
}

__device__ __forceinline__ float drift(int kind, float x, float m, float fx, float sc, float g2) {
  if (kind == DMN_SDE_VP) return __fsub_rn(__fmul_rn(fx, x), __fmul_rn(__fmul_rn(g2, __fdiv_rn(-m, sc)), 0.5f));
  return __fsub_rn(0.0f, __fmul_rn(__fmul_rn(g2, m), 0.5f));
}

__device__ void set_stage(OdeRec& r, const OdeParams& P, int i, double t) {
  stage_scalars(P, t, r.labels[i], r.fx[i], r.sc[i], r.g2[i]);
}

__device__ void publish(const OdeRec& r, dmn_ode_result* res) {
  res->status = r.status;
  res->nfev = r.nfev;
  res->n_accepted = r.n_acc;
  res->n_rejected = r.n_rej;
  res->t_final = r.t;
}

// start of an attempt (RK45._step_impl): step bounds, termination checks, clip onto t_bound, the 6 stage times
__device__ void begin_attempt(OdeRec& r, const OdeParams& P, bool new_step) {
  const double dir = P.t1 > P.t0 ? 1.0 : -1.0;
  if (new_step) {
    r.min_step = 10.0 * fabs(nextafter(r.t, dir * INFINITY) - r.t);
    if (r.h_abs < r.min_step) r.h_abs = r.min_step;
  }
  if (r.h_abs < r.min_step) { r.status = DMN_ODE_TOO_SMALL_STEP; return; }
  if (r.nfev + 6 > P.max_nfe) { r.status = DMN_ODE_LIMIT; return; }
  double t_new = r.t + r.h_abs * dir;
  if (dir * (t_new - P.t1) > 0) t_new = P.t1;
  const double h = t_new - r.t;
  r.h = h;
  r.h_abs = fabs(h);
  r.t_new = t_new;
  for (int s = 1; s <= 5; ++s) set_stage(r, P, s - 1, r.t + kC[s] * h);
  set_stage(r, P, 5, r.t + h);
}

// fixed-order block sum of the per-block partial pairs -> tot[0], tot[1] (valid in every thread after the call)
__device__ void reduce_partials(const double* part, int nblk, double tot[2]) {
  __shared__ double red[2][kThreads];
  double a = 0.0, b = 0.0;
  for (int i = threadIdx.x; i < nblk; i += kThreads) { a += part[2 * i]; b += part[2 * i + 1]; }
  red[0][threadIdx.x] = a;
  red[1][threadIdx.x] = b;
  __syncthreads();
  for (int w = kThreads / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) { red[0][threadIdx.x] += red[0][threadIdx.x + w]; red[1][threadIdx.x] += red[1][threadIdx.x + w]; }
    __syncthreads();
  }
  tot[0] = red[0][0];
  tot[1] = red[1][0];
}

// fixed-order block reduction of two per-thread sums into part[2 * blockIdx.x + {0, 1}]
__device__ void block_partials(double a, double b, double* part) {
  __shared__ double red[2][kThreads];
  red[0][threadIdx.x] = a;
  red[1][threadIdx.x] = b;
  __syncthreads();
  for (int w = kThreads / 2; w > 0; w >>= 1) {
    if ((int)threadIdx.x < w) { red[0][threadIdx.x] += red[0][threadIdx.x + w]; red[1][threadIdx.x] += red[1][threadIdx.x + w]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { part[2 * blockIdx.x] = red[0][0]; part[2 * blockIdx.x + 1] = red[1][0]; }
}

__device__ __forceinline__ void set_cond(cudaGraphConditionalHandle h, int use, bool v) {
  if (use) cudaGraphSetConditional(h, v ? 1u : 0u);
}

// ---- init phase -------------------------------------------------------------------------------------------------------------
// phase 0 (1 thread): fresh record, stage row 0 = t0
__global__ void ode_init_kernel(OdeWork w, OdeParams P) {
  OdeRec& r = *w.rec;
  r = OdeRec{};
  r.t = P.t0;
  r.status = DMN_ODE_RUNNING;
  r.k0 = 0;
  r.k6 = 6;
  for (int s = 0; s < 6; ++s) { w.rows[s] = s; set_stage(r, P, s, P.t0); }
  publish(r, w.result);
}

// elementwise init passes.  mode 0: y0 = (double)state, U-Net input = state.
//   mode 1: f0 = drift -> K0; partials {sum (y0/scale)^2, sum (f0/scale)^2}, scale = atol + |y0| rtol.
//   mode 2: U-Net input = (float)(y0 + (h0 * direction) * f0).      mode 3: f1 = drift; partials {sum ((f1 - f0)/scale)^2, 0}.
__global__ void __launch_bounds__(kThreads) ode_init_elem_kernel(OdeWork w, OdeParams P, const float* __restrict__ state, int mode) {
  const OdeRec& r = *w.rec;
  const long n = w.n;
  double* y = w.y;
  float* K0 = w.K;
  const float fx = r.fx[0], sc = r.sc[0], g2 = r.g2[0];
  const double dir = P.t1 > P.t0 ? 1.0 : -1.0;
  const double hd = r.h0 * dir;
  double a = 0.0, b = 0.0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    if (mode == 0) {
      y[i] = i < w.nx ? (double)state[i] : 0.0;
      if (i < w.nx) w.x32[i] = state[i];
    } else if (mode == 2) {
      if (i < w.nx) w.x32[i] = __double2float_rn(y[i] + hd * (double)K0[i]);
    } else {
      const float f = i < w.nx ? drift(P.sde_kind, w.x32[i], w.mo[i], fx, sc, g2) : w.mo[i];
      const double s = P.atol + fabs(y[i]) * P.rtol;
      if (mode == 1) {
        K0[i] = f;
        const double u = y[i] / s, v = (double)f / s;
        a += u * u;
        b += v * v;
      } else {
        const double u = ((double)f - (double)K0[i]) / s;
        a += u * u;
      }
    }
  }
  if (mode == 1 || mode == 3) block_partials(a, b, w.partials);
}

// one block: select_initial_step.  mode 0: d0, d1 -> h0 and the stage row of t0 + h0 * direction.
//   mode 1: d2 -> h1 -> h_abs, then the first attempt.
__global__ void __launch_bounds__(kThreads) ode_init_step_kernel(OdeWork w, OdeParams P, int nblk, int mode, cudaGraphConditionalHandle hnd,
                                                                 int use_cond) {
  double tot[2];
  reduce_partials(w.partials, nblk, tot);
  if (threadIdx.x != 0) return;
  OdeRec& r = *w.rec;
  const double rootn = sqrt((double)w.n);
  const double dir = P.t1 > P.t0 ? 1.0 : -1.0;
  const double interval = fabs(P.t1 - P.t0);
  if (mode == 0) {
    const double d0 = sqrt(tot[0]) / rootn, d1 = sqrt(tot[1]) / rootn;
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = fmin(h0, interval);
    r.h0 = h0;
    r.d1 = d1;
    r.nfev = 1;
    set_stage(r, P, 0, P.t0 + h0 * dir);
  } else {
    const double d1 = r.d1, h0 = r.h0;
    const double d2 = sqrt(tot[0]) / rootn / h0;
    const double h1 = (d1 <= 1e-15 && d2 <= 1e-15) ? fmax(1e-6, h0 * 1e-3) : pow(0.01 / fmax(d1, d2), 1.0 / 5);
    r.h_abs = fmin(fmin(100 * h0, h1), interval);
    r.nfev = 2;
    begin_attempt(r, P, true);
    set_cond(hnd, use_cond, r.status == DMN_ODE_RUNNING);
  }
  publish(r, w.result);
}

// ---- one attempt ------------------------------------------------------------------------------------------------------------
// Stage S after the U-Net evaluation of stage S (S = 0: no evaluation, only the input of stage 1):
//   K_S = drift(x_S, model_out)                                                        (S >= 1)
//   S <= 4: next U-Net input x_{S+1} = (float)(y + (sum_{j<=S} a_{S+1,j} K_j) * h)
//   S == 5: y_new = y + h * sum_j b_j K_j (fp64, kept) and the U-Net input (float)y_new
//   S == 6: per-block partial sums of (h * sum_j e_j K_j / scale)^2
template <int S>
__global__ void __launch_bounds__(kThreads) ode_stage_kernel(OdeWork w, OdeParams P) {
  const OdeRec& r = *w.rec;
  const long n = w.n;
  const double h = r.h;
  const double* y = w.y + (long)r.cur * n;
  double* yn = w.y + (long)(r.cur ^ 1) * n;
  const float* Kj[7];
#pragma unroll
  for (int j = 0; j < 7; ++j) Kj[j] = w.K + (long)(j == 0 ? r.k0 : j == 6 ? r.k6 : j) * n;
  float* Ks = const_cast<float*>(Kj[S]);
  float fx = 0.f, sc = 1.f, g2 = 0.f;
  if (S >= 1) { fx = r.fx[S - 1]; sc = r.sc[S - 1]; g2 = r.g2[S - 1]; }
  const double rtol = P.rtol, atol = P.atol;
  double part = 0.0;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) {
    float k = 0.f;
    if (S >= 1) {
      k = i < w.nx ? drift(P.sde_kind, w.x32[i], w.mo[i], fx, sc, g2) : w.mo[i];
      Ks[i] = k;
    }
    if (S <= 4) {
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j <= S; ++j) acc = __dadd_rn(acc, __dmul_rn((double)(S >= 1 && j == S ? k : Kj[j][i]), kA[S + 1][j]));
      if (i < w.nx) w.x32[i] = __double2float_rn(__dadd_rn(y[i], __dmul_rn(acc, h)));
    } else if (S == 5) {
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j <= 5; ++j) acc = __dadd_rn(acc, __dmul_rn((double)(j == 5 ? k : Kj[j][i]), kB[j]));
      const double v = __dadd_rn(y[i], __dmul_rn(h, acc));
      yn[i] = v;
      if (i < w.nx) w.x32[i] = __double2float_rn(v);
    } else {
      double acc = 0.0;
#pragma unroll
      for (int j = 0; j <= 6; ++j) acc = __dadd_rn(acc, __dmul_rn((double)(j == 6 ? k : Kj[j][i]), kE[j]));
      const double s = __dadd_rn(atol, __dmul_rn(fmax(fabs(y[i]), fabs(yn[i])), rtol));
      const double q = __dmul_rn(acc, h) / s;
      part = __fma_rn(q, q, part);
    }
  }
  if (S == 6) block_partials(part, 0.0, w.partials);
}

// one block: error norm, accept / reject, step-size update, rotation of y / y_new and K0 / K6 by index, counters, the next
// attempt's stage rows, and the WHILE condition
__global__ void __launch_bounds__(kThreads) ode_control_kernel(OdeWork w, OdeParams P, int nblk, cudaGraphConditionalHandle hnd, int use_cond) {
  double tot[2];
  reduce_partials(w.partials, nblk, tot);
  if (threadIdx.x != 0) return;
  OdeRec& r = *w.rec;
  if (r.status != DMN_ODE_RUNNING) {     // plain launches never get here in a finished state; keep the record unchanged if they do
    set_cond(hnd, use_cond, false);
    return;
  }
  r.nfev += 6;
  const double err = sqrt(tot[0]) / sqrt((double)w.n);
  const double dir = P.t1 > P.t0 ? 1.0 : -1.0;
  bool accepted = false;
  if (err < 1.0) {
    double factor = err == 0.0 ? 10.0 : fmin(10.0, 0.9 * pow(err, -0.2));
    if (r.rejected) factor = fmin(1.0, factor);
    r.h_abs *= factor;
    r.t = r.t_new;
    r.cur ^= 1;
    const int k = r.k0;
    r.k0 = r.k6;
    r.k6 = k;
    r.rejected = 0;
    r.n_acc += 1;
    accepted = true;
    if (dir * (r.t - P.t1) >= 0) r.status = DMN_ODE_DONE;
  } else {
    r.h_abs *= fmax(0.2, 0.9 * pow(err, -0.2));
    r.rejected = 1;
    r.n_rej += 1;
  }
  if (r.status == DMN_ODE_RUNNING) begin_attempt(r, P, accepted);
  set_cond(hnd, use_cond, r.status == DMN_ODE_RUNNING);
  publish(r, w.result);
}

// ---- likelihood (augmented state [x ; delta_logp]) ----------------------------------------------------------------------------
// Hutchinson divergence of the drift at the evaluation of stage row `row`: mo[nx + b] = sum_i eps_i * drift(eps_i, dmo_i) over
// sample b, where dmo is the U-Net JVP in direction eps (drift is linear in (x, model output), so drift(eps, dmo) is its tangent).
// One block per sample, fp64 per-thread sums in a fixed order, then a fixed-order block reduction.
__global__ void __launch_bounds__(kThreads) ode_div_kernel(OdeWork w, OdeParams P, int row, long chw) {
  __shared__ double red[kThreads];
  const OdeRec& r = *w.rec;
  const float fx = r.fx[row], sc = r.sc[row], g2 = r.g2[row];
  const long base = (long)blockIdx.x * chw;
  double a = 0.0;
  for (long i = threadIdx.x; i < chw; i += kThreads) {
    const float e = w.eps[base + i];
    a += (double)e * (double)drift(P.sde_kind, e, w.dmo[base + i], fx, sc, g2);
  }
  red[threadIdx.x] = a;
  __syncthreads();
  for (int s = kThreads / 2; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) red[threadIdx.x] += red[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) w.mo[w.nx + blockIdx.x] = __double2float_rn(red[0]);
}

// Rademacher noise from a Gaussian draw: +1 where the draw is >= 0, -1 elsewhere
__global__ void __launch_bounds__(kThreads) ode_rademacher_kernel(float* __restrict__ e, long n) {
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long)gridDim.x * blockDim.x) e[i] = e[i] >= 0.f ? 1.f : -1.f;
}

// solution.y[:, -1] cast to fp32 (the last accepted state)
__global__ void __launch_bounds__(kThreads) ode_finish_kernel(OdeWork w, float* __restrict__ state) {
  const double* y = w.y + (long)w.rec->cur * w.n;
  for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < w.n; i += (long)gridDim.x * blockDim.x) state[i] = __double2float_rn(y[i]);
}

}  // namespace ode
using namespace ode;

int ode_grid(long n) {
  long g = (n + kThreads - 1) / kThreads;
  if (g > 148 * 4) g = 148 * 4;
  return (int)(g < 1 ? 1 : g);
}

size_t ode_work_layout(long n, char* base, OdeWork* w) {
  auto up = [](size_t v) { return (v + 255) / 256 * 256; };
  size_t off = 0;
  const size_t o_rec = off;  off += up(sizeof(OdeRec) + 8 * sizeof(int32_t));
  const size_t o_y = off;    off += up((size_t)2 * n * sizeof(double));
  const size_t o_k = off;    off += up((size_t)7 * n * sizeof(float));
  const size_t o_x = off;    off += up((size_t)n * sizeof(float));
  const size_t o_mo = off;   off += up((size_t)n * sizeof(float));
  const size_t o_p = off;    off += up((size_t)2 * ode_grid(n) * sizeof(double));
  if (w) {
    w->n = n;
    w->nx = n;
    w->rec = (OdeRec*)(base + o_rec);
    w->rows = (int32_t*)(base + o_rec + sizeof(OdeRec));
    w->y = (double*)(base + o_y);
    w->K = (float*)(base + o_k);
    w->x32 = (float*)(base + o_x);
    w->mo = (float*)(base + o_mo);
    w->partials = (double*)(base + o_p);
  }
  return off;
}

int launch_ode_init(const OdeWork& w, const OdeParams& P, cudaStream_t st) {
  ode_init_kernel<<<1, 1, 0, st>>>(w, P);
  count_launch();
  DMN_LAUNCH_CHECK("ode_init");
  return 0;
}
int launch_ode_init_elem(const OdeWork& w, const OdeParams& P, const float* state, int mode, cudaStream_t st) {
  ode_init_elem_kernel<<<ode_grid(w.n), kThreads, 0, st>>>(w, P, state, mode);
  count_launch();
  DMN_LAUNCH_CHECK("ode_init_elem");
  return 0;
}
int launch_ode_init_step(const OdeWork& w, const OdeParams& P, int mode, cudaGraphConditionalHandle hnd, int use_cond, cudaStream_t st) {
  ode_init_step_kernel<<<1, kThreads, 0, st>>>(w, P, ode_grid(w.n), mode, hnd, use_cond);
  count_launch();
  DMN_LAUNCH_CHECK("ode_init_step");
  return 0;
}
int launch_ode_stage(const OdeWork& w, const OdeParams& P, int s, cudaStream_t st) {
  const int g = ode_grid(w.n);
  switch (s) {
    case 0: ode_stage_kernel<0><<<g, kThreads, 0, st>>>(w, P); break;
    case 1: ode_stage_kernel<1><<<g, kThreads, 0, st>>>(w, P); break;
    case 2: ode_stage_kernel<2><<<g, kThreads, 0, st>>>(w, P); break;
    case 3: ode_stage_kernel<3><<<g, kThreads, 0, st>>>(w, P); break;
    case 4: ode_stage_kernel<4><<<g, kThreads, 0, st>>>(w, P); break;
    case 5: ode_stage_kernel<5><<<g, kThreads, 0, st>>>(w, P); break;
    default: ode_stage_kernel<6><<<g, kThreads, 0, st>>>(w, P); break;
  }
  count_launch();
  DMN_LAUNCH_CHECK("ode_stage");
  return 0;
}
int launch_ode_control(const OdeWork& w, const OdeParams& P, cudaGraphConditionalHandle hnd, int use_cond, cudaStream_t st) {
  ode_control_kernel<<<1, kThreads, 0, st>>>(w, P, ode_grid(w.n), hnd, use_cond);
  count_launch();
  DMN_LAUNCH_CHECK("ode_control");
  return 0;
}
int launch_ode_div(const OdeWork& w, const OdeParams& P, int row, int batch, cudaStream_t st) {
  ode_div_kernel<<<batch, kThreads, 0, st>>>(w, P, row, w.nx / batch);
  count_launch();
  DMN_LAUNCH_CHECK("ode_div");
  return 0;
}
int launch_ode_rademacher(float* e, long n, cudaStream_t st) {
  ode_rademacher_kernel<<<ode_grid(n), kThreads, 0, st>>>(e, n);
  count_launch();
  DMN_LAUNCH_CHECK("ode_rademacher");
  return 0;
}
int launch_ode_finish(const OdeWork& w, float* state, cudaStream_t st) {
  ode_finish_kernel<<<ode_grid(w.n), kThreads, 0, st>>>(w, state);
  count_launch();
  DMN_LAUNCH_CHECK("ode_finish");
  return 0;
}

}  // namespace dmn

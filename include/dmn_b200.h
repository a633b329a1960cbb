/*
 * dmn_b200.h -- C ABI of libdmn_b200.so: the B200 (sm_100a) reverse-diffusion sampling hot path.
 *
 * The reference (titu1994/diffusion_model_nemo) is pure Python and has no FFI of its own; its plugin
 * surface is Python duck typing selected by Hydra `_target_` strings (SURVEY.md section 8b).  This header is
 * the boundary the Python drop-in classes (diffusion_model_nemo_b200/modules/ *.py) bind with ctypes; every
 * entry point names the reference function(s) it replaces (paths relative to
 * /root/reference/diffusion_model_nemo/).  INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch types.  All `*_dev` pointers are device pointers owned by the
 *     CALLER (PyTorch allocates them); the library never allocates device memory.
 *   - every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns without syncing,
 *     except dmn_plan_load_param (host repack + async copy) and dmn_loop_* (documented below).
 *   - return value: 0 = ok, <0 = error (DMN_E*); dmn_last_error() returns a thread-local message.
 *   - there is NO CPU fallback: unsupported shapes / missing GPU give an error code, never a slow path.
 */
#ifndef DMN_B200_H
#define DMN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DMN_OK        0
#define DMN_EINVAL   -1   /* bad argument / unsupported configuration */
#define DMN_ENOTSUP  -2   /* valid request, but this build has no kernel for it */
#define DMN_ECUDA    -3   /* CUDA runtime error (message holds cudaGetErrorString) */
#define DMN_ESTATE   -4   /* call order violated (e.g. forward before bind / load) */

#define DMN_ABI_VERSION 1

/* activation storage / arithmetic mode of a plan */
#define DMN_ACT_F32   0   /* fp32 activations, fp32 CUDA-core convolutions (parity mode, 1e-4) */
#define DMN_ACT_BF16  1   /* bf16 activations, fp32 accumulation (throughput mode, 2e-2) */

/* convolution engine */
#define DMN_CONV_SIMT     0   /* CUDA-core implicit GEMM (any shape; used by DMN_ACT_F32) */
#define DMN_CONV_TCGEN05  1   /* tcgen05/TMEM implicit GEMM, bf16 operands (DMN_ACT_BF16 only) */

const char* dmn_last_error(void);
int dmn_abi_version(void);

/* ------------------------------------------------------------------------------------------------------
 * U-Net plan.  Replaces Unet.__init__ / Unet.forward (modules/unet.py:14-168) and everything below it:
 * ResnetBlock/Block (parts/convnext.py:8-86), LinearAttention/Attention (parts/mha.py:8-59),
 * SinusoidalPositionEmbeddings (parts/positional_encoding.py:6-18), Residual/PreNorm/Upsample/Downsample
 * (utils.py:68-93), and WaveGradUNet.forward + FeatureWiseLinearModulation / PositionalEncoding (unet.py:171-266,
 * parts/film.py:11-61) when cfg.film = 1.  use_convnext=True is DMN_ENOTSUP (no shipped config uses it).
 * ---------------------------------------------------------------------------------------------------- */
typedef struct dmn_plan dmn_plan;

typedef struct dmn_unet_cfg {
  int32_t dim;             /* Unet(dim=)                         unet.py:18 */
  int32_t n_mults;         /* len(dim_mults), 1..8               unet.py:20 */
  int32_t dim_mults[8];
  int32_t channels;        /* image channels                     unet.py:21 */
  int32_t out_dim;         /* channels * (2 if learned_variance) unet.py:109-110 */
  int32_t groups;          /* resnet_block_groups                unet.py:22 */
  int32_t with_time_emb;   /* 1 = time_mlp present               unet.py:59-69 */
  int32_t num_classes;     /* -1 = unconditional; else class_embed has num_classes+1 rows, unet.py:118-120 */
  int32_t image_size;      /* H == W of the input                */
  int32_t max_batch;       /* workspace is sized for this batch  */
  int32_t act_dtype;       /* DMN_ACT_*                          */
  int32_t conv_engine;     /* DMN_CONV_*                         */
  int32_t max_time_rows;   /* rows of the time-embedding table (>= max_batch and >= loop steps) */
  int32_t film;            /* 1 = WaveGradUNet (unet.py:171-266): requires with_time_emb = 0; FeatureWiseLinearModulation
                              layers films.0 .. films.{n_mults-1} (parts/film.py:29-61) driven by a continuous noise level */
  int32_t plain_tail;      /* 1 = resnet_block_order 'conv_bn_act': final_conv = [ResnetBlock, Conv2d(dim, out_dim, 1)] without the
                              GroupNorm + SiLU in front of the 1x1 (unet.py:112-116); the 1x1 is then final_conv.1 */
  int32_t reserved[1];
} dmn_unet_cfg;

int    dmn_plan_create(const dmn_unet_cfg* cfg, dmn_plan** out);
void   dmn_plan_destroy(dmn_plan* p);
size_t dmn_plan_weights_bytes(const dmn_plan* p);      /* packed-parameter arena */
size_t dmn_plan_workspace_bytes(const dmn_plan* p);    /* activations + statistics + time table */
int    dmn_plan_bind(dmn_plan* p, void* weights_dev, size_t weights_bytes, void* workspace_dev, size_t workspace_bytes);

/* Parameter table: names and shapes are those of the reference state_dict (SURVEY.md section 5). */
int         dmn_plan_num_params(const dmn_plan* p);
const char* dmn_plan_param_name(const dmn_plan* p, int i);
int         dmn_plan_param_shape(const dmn_plan* p, int i, int64_t shape_out[4]);   /* returns ndim */
/* host fp32 data in PyTorch layout; repacked (OIHW -> engine layout, bf16 rounding) and copied on `stream`. */
int dmn_plan_load_param(dmn_plan* p, const char* name, const float* host_data, int64_t numel, void* stream);
/* host fp32 [dim/2] sinusoid frequencies, computed by the host with the reference's torch ops
 * (positional_encoding.py:13-15) so the table is bit-exact. */
int dmn_plan_load_freqs(dmn_plan* p, const float* host_freqs, int n, void* stream);
int dmn_plan_ready(const dmn_plan* p);                 /* 1 when every parameter has been loaded */
/* film plans: channels of every evaluated FiLM layer in table-column order (returns the count).  dmn_plan_load_freqs then takes
 * sum(channels) values: for each layer its [exponents | exponents], exponents = 1e-4 ** (arange(C/2) / (C/2)) computed by the
 * host with the reference's torch ops (PositionalEncoding.forward, parts/film.py:19-21). */
int dmn_plan_film_layout(const dmn_plan* p, int32_t* channels_out, int cap);

/* time_mlp + the 16 per-block `mlp` projections for `rows` time values -> table rows [row0, row0+rows).
 * Replaces Unet.time_mlp (unet.py:61-66) and ResnetBlock.mlp (convnext.py:68-72,81-83).  At most 65535 rows per call
 * (DMN_EINVAL otherwise, before anything is enqueued). */
int dmn_time_table(dmn_plan* p, const float* times_dev, int row0, int rows, void* stream);
/* Read-only view of the table (validation aid): row r, column c is the fp32 at workspace + *ws_offset + (r * *sum_c + c) * 4 for
 * r < *max_rows.  DMN_EINVAL for a plan with neither time embedding nor FiLM.  Any output pointer may be NULL. */
int dmn_plan_time_table_info(const dmn_plan* p, size_t* ws_offset, int32_t* sum_c, int32_t* max_rows);
/* First table column of parameter i: a ResnetBlock's `mlp.1.weight` / `mlp.1.bias` fill columns [col, col + Cout); -1 for any
 * other parameter or a bad index. */
int dmn_plan_param_time_col(const dmn_plan* p, int i);
/* film plans: first table column of FiLM layer `layer` (dmn_plan_film_layout order; it fills [col, col + channels)); -1 otherwise. */
int dmn_plan_film_col(const dmn_plan* p, int layer);
/* film plans: `times_dev` holds continuous noise levels and the table rows are the FiLM positional encodings
 * sin | cos (5000 * level * exponents) of every FiLM layer (parts/film.py:17-26); dmn_unet_forward then evaluates
 * WaveGradUNet.forward(x, noise_level) (unet.py:212-266).  Plans with neither time embedding nor FiLM ignore the call. */

/* eps = Unet.forward(x, time, classes)  (unet.py:131-168).
 *   x_dev    fp32 NCHW [batch, channels, S, S]         out_dev  fp32 NCHW [batch, out_dim, S, S]
 *   time row: if row_dev == NULL sample b uses table row b (call dmn_time_table(times, 0, batch) first);
 *             else every sample uses row *row_dev (device int32; CUDA-graph friendly).
 *   classes_dev: int64 [batch] or NULL (NULL + num_classes>=0 means the padding row, unet.py:135-137). */
int dmn_unet_forward(dmn_plan* p, const float* x_dev, const int32_t* row_dev, const int64_t* classes_dev,
                     float* out_dev, int batch, void* stream);
/* number of kernel launches one dmn_unet_forward enqueues (for bench.py's gpu_launches). */
int dmn_plan_launches_per_forward(const dmn_plan* p);

/* Forward-mode JVP: out = u(x, t) and out_tangent = (du/dx) . v, for fp32 plans on the SIMT engine (DMN_ENOTSUP for bf16 /
 * tcgen05 plans and for FiLM plans).  x_dev, v_dev, out_dev, out_tangent_dev and the time / class arguments as in
 * dmn_unet_forward; out_dev is bit-identical to what dmn_unet_forward writes.  The time and class embeddings do not depend on x.
 * work_dev: caller-owned, 256-byte aligned, >= dmn_unet_jvp_work_bytes(p, batch) bytes (the tangents of the workspace buffers
 * and the operand of the tangent convolutions).  No device allocation; graph-capturable. */
int dmn_unet_jvp(dmn_plan* p, const float* x_dev, const float* v_dev, const int32_t* row_dev, const int64_t* classes_dev,
                 float* out_dev, float* out_tangent_dev, void* work_dev, size_t work_bytes, int batch, void* stream);
size_t dmn_unet_jvp_work_bytes(const dmn_plan* p, int batch);

/* Measurement aids for bench.py's roofline (no reference counterpart).
 * dmn_plan_num_ops / dmn_plan_op_info: static description of launch i of the forward program -- name, kind
 *   (0 memset, 1 init_conv, 2 conv, 3 gn_finalize, 4 linattn, 5 attn, 6 final_proj, 7 film_modulate, 8 class_embed_add), engine (0 CUDA cores, 1 tcgen05),
 *   algorithmic FLOPs (2*MAC) and algorithmic bytes (operands read once + result written once) PER SAMPLE.
 * dmn_plan_profile_forward: one forward with a CUDA event pair around every launch on `stream`; writes per-launch
 *   milliseconds to ms_out[0..num_ops) and synchronises the stream (not graph-capturable). */
int dmn_plan_num_ops(const dmn_plan* p);
int dmn_plan_op_info(const dmn_plan* p, int i, char* name_out, int name_cap, int32_t* kind, int32_t* engine,
                     double* flops_per_sample, double* bytes_per_sample);
int dmn_plan_profile_forward(dmn_plan* p, const float* x_dev, const int32_t* row_dev, const int64_t* classes_dev,
                             float* out_dev, int batch, void* stream, float* ms_out, int max_ops);
/* the same per-launch times measured INSIDE one CUDA graph (event-record nodes between the launches): the kernels run back to back
 * as in the sampling loop, without the launch latency plain stream launches expose between dependent kernels. */
int dmn_plan_profile_forward_graph(dmn_plan* p, const float* x_dev, const int32_t* row_dev, const int64_t* classes_dev,
                                   float* out_dev, int batch, void* stream, float* ms_out, int max_ops);

/* ------------------------------------------------------------------------------------------------------
 * Sampler updates: ONE fused elementwise kernel per step.  Coefficients live in a device table
 * coef_dev[step][DMN_COEF_STRIDE] (fp32) built by the host from the bit-exact schedule tables; the row is
 * selected by *step_dev (device int32) or by `step` when step_dev is NULL.  z_dev is the injected N(0,1)
 * tensor for this step (parity mode) or NULL to draw in-kernel with Philox4x32-10 keyed (seed, stream_id),
 * counter (step, element).  All tensors fp32 NCHW, n = batch*C*H*W elements, x_out may alias x.
 * ---------------------------------------------------------------------------------------------------- */
#define DMN_COEF_STRIDE 8

typedef struct dmn_rng { uint64_t seed; uint64_t stream_id; } dmn_rng;

/* GaussianDiffusion.p_mean_variance + p_sample (gaussian_diffusion.py:118-167).
 * coef row: {sqrt_recip_ac, sqrt_recipm1_ac, post_coef1, post_coef2, mask*exp(0.5*post_logvar), pred_x0?1:0} */
int dmn_ddpm_step(const float* x, const float* eps, const float* z_dev, float* x_out, int64_t n,
                  const float* coef_dev, const int32_t* step_dev, int step, dmn_rng rng, void* stream);
/* LearnedGaussianDiffusion.p_mean_variance (learned_gaussian_diffusion.py:27-53) + p_sample.
 * model_out is [batch, 2C, H, W]; chw = C*H*W.  coef row: {.., .., .., .., mask, min_log, max_log} */
int dmn_learned_step(const float* x, const float* model_out, const float* z_dev, float* x_out, int batch,
                     int64_t chw, const float* coef_dev, const int32_t* step_dev, int step, dmn_rng rng, void* stream);
/* GeneralizedGaussianDiffusion.p_sample (generalized_gaussian_diffusion.py:42-45,75-95).
 * coef row: {sqrt(1-a_t), 1/sqrt(a_t)... see modules/generalized_gaussian_diffusion.py in the package} */
int dmn_ddim_step(const float* x, const float* eps, const float* z_dev, float* x_out, int64_t n,
                  const float* coef_dev, const int32_t* step_dev, int step, dmn_rng rng, void* stream);
/* DPM-Solver++ multistep update, orders 1-3 (Lu et al. 2022, "DPM-Solver++", Algorithm 2 and its third-order extension; not in
 * the reference: modules/dpm_solver_diffusion.py in the package builds the rows).  Deterministic: draws no noise.
 *   m  = clamp(pred_x0 ? model_out : k_x * x - k_m * model_out, -1, 1)      (data prediction; first C channels of each sample)
 *   x' = c_x * x + c_0 * m + c_1 * hist[(slot+2)%3] + c_2 * hist[(slot+1)%3] ;  hist[slot] = m
 * coef row: {c_x, c_0, c_1, c_2, k_x, k_m, slot, pred_x0 ? 1 : 0}.  hist_dev is a ring of 3 slots [3][batch*chw] fp32 holding the
 * previous steps' m (slot = step mod 3); a slot whose coefficient is 0 is not read, so the ring needs no initialisation.
 * model_out is [batch, mo_chw] with mo_chw = C*H*W or 2*C*H*W (learned variance: the variance channels are ignored).
 * x_out may alias x. */
int dmn_dpmpp_step(const float* x, const float* model_out, float* hist_dev, float* x_out, int batch, int64_t chw, int64_t mo_chw,
                   const float* coef_dev, const int32_t* step_dev, int step, void* stream);
/* ReverseDiffusionPredictor / EulerMaruyamaPredictor with the score wrapper folded in
 * (reverse_diffusion_predictor.py:11-16, euler_maruyama_predictor.py:11-17, sde_lib.py:91-105,
 *  score_function_loss.py:47-91):  x_mean = a*x + b*model_out ; x = x_mean + g*z.  coef row: {a, b, g} */
int dmn_affine_noise_step(const float* x, const float* model_out, const float* z_dev, float* x_out, float* x_mean_out,
                          int64_t n, const float* coef_dev, const int32_t* step_dev, int step, dmn_rng rng, void* stream);
/* LangevinCorrector.update_fn (langevin_corrector.py:15-35), two kernels:
 *   norms: per-sample ||g_b||, ||z_b|| -> batch means (scratch_dev: 2*batch + 2 floats; one block per sample, fixed summation
 *          order, so the result is bit-reproducible)
 *   apply: step = (snr*mean||z|| / mean||g||)^2 * 2*alpha ; x_mean = x + step*g ; x = x_mean + sqrt(2 step) z
 * where g = score_scale * model_out (VP: -1/std(t), VE: 1).  coef row: {score_scale, alpha}.
 * z_dev == NULL draws z in-kernel (the same Philox counters in both kernels). */
int dmn_langevin_step(const float* x, const float* model_out, const float* z_dev, float* x_out, float* x_mean_out,
                      int batch, int64_t chw, float snr, const float* coef_dev, const int32_t* step_dev, int step,
                      float* scratch_dev, dmn_rng rng, void* stream);
/* Bits-per-dimension evaluation pieces (models/abstract_diffusion_model.py:137-197).
 * dmn_bpd_qsample: x_t = sqrt_ac[t] * x_0 + sqrt_1m_ac[t] * z  (GaussianDiffusion.q_sample, gaussian_diffusion.py:104-116); coef row
 *   columns 6 / 7; z_dev == NULL draws z in-kernel.
 * dmn_bpd_term: one block per sample reduces, in a fixed order, mean_chw of KL(q(x_{t-1}|x_t,x_0) || p(x_{t-1}|x_t)) (t > 0) or of the
 *   discretised-Gaussian decoder NLL (t == 0), in bits (VariationalBoundLoss.compute_variation_loss_terms,
 *   loss/variational_bound_loss.py:31-52; utils.normal_kl / discretized_gaussian_log_likelihood, utils.py:28-56), with the posterior of
 *   q_posterior / p_mean_variance (gaussian_diffusion.py:91-101,125-154) or the learned variance interpolation
 *   (learned_gaussian_diffusion.py:27-53; model_out is [batch, 2C, H, W] when `learned`).  Writes terms[b * n_cols + col].
 *   coef row  = {sqrt_recip_ac, sqrt_recipm1_ac, post_coef1, post_coef2, post_logvar_clipped, pred_x0 ? 1 : 0, sqrt_ac, sqrt_1m_ac}
 *   coef2 row = {log beta_t, col (= t), t == 0 ? 1 : 0}
 *   mode 1 = prior term mean_chw KL(q(x_T|x_0) || N(0,1)) / ln 2 -> terms[b]; coef column 6 = sqrt_ac[T-1], coef2 row = {log(1 - ac[T-1])}. */
int dmn_bpd_qsample(const float* x0, const float* z_dev, float* x_t, int64_t n, const float* coef_dev, const int32_t* step_dev, int step,
                    dmn_rng rng, void* stream);
int dmn_bpd_term(const float* x0, const float* x_t, const float* model_out, float* terms, int batch, int64_t chw, int learned, int n_cols,
                 int mode, const float* coef_dev, const float* coef2_dev, const int32_t* step_dev, int step, void* stream);
/* x0 -> [0,1] image: (x + 1) * 0.5  (gaussian_diffusion.py:187) */
int dmn_unnormalize(const float* x, float* out, int64_t n, void* stream);
/* standard normal fill (the x_T draw, gaussian_diffusion.py:177) with the same Philox stream layout (step = -1). */
int dmn_randn(float* out, int64_t n, dmn_rng rng, int step, void* stream);
/* q_sample (gaussian_diffusion.py:104-116): out = a*x0 + b*noise */
int dmn_axpby(const float* x, const float* y, float a, float b, float* out, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Whole-loop driver: captures ONE step (U-Net + update) as a CUDA graph whose kernels read the step index
 * from a device counter, then replays it n_steps times.  Replaces p_sample_loop
 * (gaussian_diffusion.py:171-189, generalized_gaussian_diffusion.py:99-131) and
 * PredictorCorrectorSampler.forward (sde_samplers/predictor_corrector_sampler.py:58-120).
 * ---------------------------------------------------------------------------------------------------- */
#define DMN_LOOP_DDPM     0
#define DMN_LOOP_LEARNED  1
#define DMN_LOOP_DDIM     2
#define DMN_LOOP_PC       3   /* [langevin corrector x n_corr] + affine-noise predictor */
#define DMN_LOOP_BPD      4   /* bits-per-dimension evaluation: per step q_sample(x_0) -> U-Net -> one variational-bound term per sample
                                 (AbstractDiffusionModel.calculate_bits_per_dimension, models/abstract_diffusion_model.py:137-197).
                                 state_dev = x_0 (read only), aux_dev = terms [batch][n_steps] (column = coef2 row[1]),
                                 coef_dev / coef2_dev rows as documented at dmn_bpd_term; noise_dev injects the q_sample draws */
#define DMN_LOOP_DPMPP    5   /* DPM-Solver++ multistep: per step U-Net (or the guidance path) -> dmn_dpmpp_step; rows as documented
                                 there, one per (t_i, t_{i+1}) pair.  out_dim = C or 2C.  Draws nothing: noise_dev, if given, only
                                 selects plain launches with the host step index.  The history ring lives in scratch_dev. */

typedef struct dmn_loop_desc {
  int32_t kind;            /* DMN_LOOP_* */
  int32_t n_steps;         /* loop length; time table rows [0, n_steps) must be filled */
  int32_t batch;
  int32_t n_corr;          /* PC: corrector steps per iteration (0 = none) */
  float   snr;             /* PC: Langevin target snr */
  int32_t denoise;         /* PC: 1 = report x_mean of the last step */
  int32_t use_graph;       /* 1 = CUDA graph replay, 0 = plain launches (debug) */
  int32_t corr_kind;       /* PC corrector: 0 = Langevin (batch-mean norms), 1 = affine-noise rows {a,b,g} in coef2 (ALD) */
  const float*   coef_dev;       /* [n_steps][DMN_COEF_STRIDE]  update coefficients (predictor for PC) */
  const float*   coef2_dev;      /* PC: [n_steps][DMN_COEF_STRIDE] corrector coefficients */
  const int64_t* classes_dev;    /* optional class labels */
  const float*   noise_dev;      /* parity mode: [n_steps * draws_per_step][batch*C*H*W] in draw order, else NULL */
  dmn_rng        rng;            /* throughput mode */
  float*         state_dev;      /* in: x_T (fp32 NCHW); out: final state in [-1,1] space */
  float*         aux_dev;        /* PC: x_mean of the last step when denoise */
  float*         scratch_dev;    /* at least dmn_loop_scratch_bytes() bytes: model output, x_mean, the guidance buffers and
                                    the DPM-Solver++ history ring */
  size_t         scratch_bytes;
  float*         traj_dev;       /* optional [n_traj][batch*C*H*W] trajectory capture, every traj_every steps */
  int32_t        traj_every;
  float          cfg_scale;      /* guidance weight w, used when cfg_on != 0 (w = 0 is a valid weight: eps = eps_u).
                                    Classifier-free guidance (not in the reference: SURVEY.md section 8 config 5a).  Every step
                                    evaluates the U-Net on the doubled batch [x ; x] with classes_dev[0..batch) = labels and
                                    classes_dev[batch..2*batch) = num_classes (the null / padding row, unet.py:118-120) and uses
                                    eps = eps_u + cfg_scale * (eps_c - eps_u).  Needs max_batch >= 2*batch and the larger
                                    scratch dmn_loop_scratch_bytes() reports with cfg_on set.  DDPM / learned / DDIM /
                                    DPM-Solver++ loops only.
                                    With a learned-variance U-Net only the eps half is guided; the variance channels are the
                                    conditional branch's. */
  int32_t        cfg_on;         /* 1 = classifier-free guidance with weight cfg_scale, 0 = off */
  int64_t        state_elems;    /* number of floats behind state_dev; must equal batch * cfg.channels * image_size^2 (0 = unchecked) */
} dmn_loop_desc;

/* Runs the whole loop on `stream`; returns after enqueueing (no host sync unless use_graph needs capture,
 * which happens on first use of a given (plan, kind, batch) and is cached in the plan). */
int dmn_sample_loop(dmn_plan* p, const dmn_loop_desc* d, void* stream);
/* bytes of scratch_dev the descriptor needs on this plan; reads kind, batch and cfg_on only.  0 for a NULL argument, an unknown
 * kind or batch < 1. */
size_t dmn_loop_scratch_bytes(const dmn_plan* p, const dmn_loop_desc* d);
/* kernels launched per loop step for the given descriptor (bench.py's gpu_launches). */
int dmn_loop_launches_per_step(const dmn_plan* p, const dmn_loop_desc* d);

/* RePaint inpainting (Lugmayr et al. 2022, "RePaint: Inpainting using Denoising Diffusion Probabilistic Models"; not in the
 * reference: modules/gaussian_diffusion.py in the package builds the rows).  One elementwise step before the model of every event:
 *   y  = a_j * x + g_j * z2             (forward jump into this event; a_j = 1, g_j = 0 when there is none)
 *   k  = a_0 * known + s_0 * z1         (q_sample of the known image at this event's time: a_0 = sqrt(abar_t), s_0 = sqrt(1 - abar_t))
 *   x' = mask * k + (1 - mask) * y
 * coef row: {a_j, g_j, a_0, s_0}.  z1 / z2 are Philox draws 1 / 2 of step word (step + 1) * 8 + draw, keyed by element index; a draw
 * whose coefficient is 0 is not made.  known, mask: [n] fp32 (mask in [0, 1], 1 = keep).  x_out may alias x.  16 B per element. */
int dmn_inpaint_prepare(const float* x, const float* known, const float* mask, float* x_out, int64_t n, const float* coef_dev,
                        const int32_t* step_dev, int step, dmn_rng rng, void* stream);

typedef struct dmn_inpaint_desc {
  const float* known_dev;        /* [batch*C*H*W] fp32 known image in [-1, 1] */
  const float* mask_dev;         /* [batch*C*H*W] fp32 mask in [0, 1], 1 = keep */
  const float* prep_coef_dev;    /* [n_steps + 1][DMN_COEF_STRIDE] dmn_inpaint_prepare rows; row n_steps = the final composite */
} dmn_inpaint_desc;

/* dmn_sample_loop with dmn_inpaint_prepare in front of every step ("event": one model evaluation and the sampler's own update, rows
 * coef_dev[e] and time table row e), then the final composite (prepare with row n_steps, host step n_steps) after the last event.
 * Graph mode replays one captured event; the graph cache key adds the three pointers.  DMN_LOOP_DDPM / LEARNED / DDIM only (others:
 * DMN_EINVAL); noise_dev must be NULL (there is no injected-noise mode).  Kernels per event: dmn_loop_launches_per_step + 1. */
int dmn_sample_loop_inpaint(dmn_plan* p, const dmn_loop_desc* d, const dmn_inpaint_desc* ip, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Probability-flow ODE sampler.  Replaces ProbabilityFlowSampler.forward (sde_samplers/probability_flow_sampler.py:46-100,
 * score_sde's get_ode_sampler): solve_ivp(ode_func, (t0, t1), x_T, rtol, atol, method='RK45') where ode_func is the drift of
 * the reverse SDE with probability_flow=True, f(x,t) - 0.5 g(t)^2 score(x,t), over this plan's U-Net (score wrapper of
 * score_function_loss.py:47-91: VP labels t*(N-1) and score = -model/std(t); VE labels sigma(t) and score = model).
 * Every model evaluation, the error norm, the accept / reject decision and the step-size update run on the device with
 * scipy.integrate.RK45's rules (Dormand-Prince 5(4), FSAL, select_initial_step, SAFETY 0.9, factors 0.2..10, exponent -1/5).
 * use_graph = 1: one cached CUDA graph per (plan, descriptor): init phase, then a WHILE conditional node over attempts; the
 * call enqueues and returns.  use_graph = 0: the same kernels with a host read of the status after every attempt (syncs).
 * The solve stops at t1 (DMN_ODE_DONE), at a step below scipy's min_step (DMN_ODE_TOO_SMALL_STEP: the last accepted state is
 * returned, as solve_ivp does) or before an attempt that would exceed max_nfe evaluations (DMN_ODE_LIMIT).
 * The plan needs max_time_rows >= 6 (the 6 stage rows of an attempt), out_dim == channels and no FiLM.
 * ---------------------------------------------------------------------------------------------------- */
#define DMN_SDE_VP 0
#define DMN_SDE_VE 1

#define DMN_ODE_RUNNING         0
#define DMN_ODE_DONE            1
#define DMN_ODE_TOO_SMALL_STEP -1
#define DMN_ODE_LIMIT          -2

typedef struct dmn_ode_result {
  int32_t status;          /* DMN_ODE_* */
  int32_t nfev;            /* model evaluations (solution.nfev) */
  int32_t n_accepted;
  int32_t n_rejected;
  double  t_final;         /* time of the returned state */
} dmn_ode_result;

typedef struct dmn_ode_desc {
  int32_t sde_kind;        /* DMN_SDE_VP / DMN_SDE_VE */
  int32_t N;               /* VP: label = t * (N - 1) */
  double  beta_0, beta_1;  /* VP */
  double  sigma_min, sigma_max;   /* VE */
  double  t0, t1;          /* integration interval (sde.T -> eps); t0 != t1 */
  double  rtol, atol;      /* scalar tolerances: rtol > 0 (raised to 100 * DBL_EPSILON like scipy), atol >= 0 */
  int32_t max_nfe;         /* evaluation budget, >= 2 */
  int32_t batch;
  int32_t use_graph;
  int32_t reserved;
  const int64_t* classes_dev;     /* optional class labels [batch] */
  float*   state_dev;      /* in: x_T (fp32 NCHW); out: the final state (fp32) */
  int64_t  state_elems;    /* floats behind state_dev: batch * channels * image_size^2 */
  void*    work_dev;       /* caller-owned, 256-byte aligned, >= dmn_ode_work_bytes(plan, batch) */
  size_t   work_bytes;
  dmn_ode_result* result_dev;     /* device record, valid once the stream has run the solve */
} dmn_ode_desc;

int    dmn_ode_sample(dmn_plan* p, const dmn_ode_desc* d, void* stream);
size_t dmn_ode_work_bytes(const dmn_plan* p, int batch);

/* Probability-flow ODE log-likelihood (score_sde's get_likelihood_fn; reference modules/sde_lib/likelihood.py): the same device
 * RK45 over the augmented state [x ; delta_logp] (batch * channels * image_size^2 + batch elements) from t0 = eps to t1 = sde.T.
 * The drift of x is the probability-flow drift above; the drift of delta_logp[b] is the Hutchinson divergence
 * sum_i eps_i * (d drift / dx . eps)_i over sample b, from one dmn_unet_jvp pass in direction eps per evaluation (which also
 * gives the model output).  The error norm runs over all elements, as scipy's does over the concatenated vector.  eps is
 * noise_dev (injected, fp32 [batch, C, S, S]) or, when NULL, drawn once per solve with Philox4x32-10 keyed rng
 * (Rademacher: the sign of the Gaussian draw).  Needs an fp32 SIMT plan (DMN_ENOTSUP otherwise) with the dmn_ode_sample
 * requirements.  use_graph as in dmn_ode_sample (one cached graph per plan and descriptor). */
#define DMN_HUTCH_RADEMACHER 0
#define DMN_HUTCH_GAUSSIAN   1

typedef struct dmn_ode_likelihood_desc {
  int32_t sde_kind;        /* DMN_SDE_VP / DMN_SDE_VE */
  int32_t N;               /* VP: label = t * (N - 1) */
  double  beta_0, beta_1;  /* VP */
  double  sigma_min, sigma_max;   /* VE */
  double  t0, t1;          /* integration interval (eps -> sde.T); t0 != t1 */
  double  rtol, atol;      /* as in dmn_ode_desc */
  int32_t max_nfe;         /* evaluation budget, >= 2 */
  int32_t batch;
  int32_t use_graph;
  int32_t hutchinson;      /* DMN_HUTCH_RADEMACHER / DMN_HUTCH_GAUSSIAN (ignored when noise_dev is given) */
  dmn_rng rng;             /* Philox key of the Hutchinson draw when noise_dev == NULL */
  const float* noise_dev;  /* injected Hutchinson noise [batch * channels * image_size^2] or NULL */
  const int64_t* classes_dev;     /* optional class labels [batch] */
  float*   state_dev;      /* in: data in the first batch * channels * image_size^2 floats; out: z, then delta_logp[batch] */
  int64_t  state_elems;    /* floats behind state_dev: batch * (channels * image_size^2 + 1) */
  void*    work_dev;       /* caller-owned, 256-byte aligned, >= dmn_ode_likelihood_work_bytes(plan, batch) */
  size_t   work_bytes;
  dmn_ode_result* result_dev;     /* device record, valid once the stream has run the solve */
} dmn_ode_likelihood_desc;

int    dmn_ode_likelihood(dmn_plan* p, const dmn_ode_likelihood_desc* d, void* stream);
size_t dmn_ode_likelihood_work_bytes(const dmn_plan* p, int batch);

/* ------------------------------------------------------------------------------------------------------
 * Layer-level entry points (unit tests and INTEGRATION.md's per-module swap).  Activations are fp32 NCHW at
 * this boundary; the call converts to the plan-independent engine layout (NHWC) internally, so they are for
 * validation, not speed.  `engine`/`act` as in the plan.
 * ---------------------------------------------------------------------------------------------------- */
/* Block.forward_conv_bn_relu input side: y_raw = conv2d(prologue(x)) + bias, and GroupNorm statistics of y_raw.
 *   mode 0: k x k stride-1 same-padding (k = 1, 3)   [Block.proj convnext.py:11,34; 1x1s mha.py:13-14,39-42]
 *   mode 1: Downsample k4 s2 p1                       [utils.py:81-82]
 *   mode 2: Upsample ConvTranspose2d k4 s2 p1         [utils.py:77-78]
 * prologue: gn_groups > 0 applies GroupNorm(gn_groups) with gamma/beta (+ SiLU if silu) (+ temb[b][c] if given)
 * to x before the convolution (convnext.py:35-41,81-83).  Weights fp32 in PyTorch layout (device). */
typedef struct dmn_conv_args {
  int32_t mode, ksize, batch, cin, cout, hin, win;
  int32_t gn_groups, silu;
  int32_t out_groups;      /* >0: also return GroupNorm stats of the output, [batch][out_groups][2] = {mean, rstd} */
  int32_t act, engine;
  const float* x;  const float* w;  const float* bias;
  const float* gn_gamma; const float* gn_beta; const float* temb;   /* temb: [batch][cin] or NULL */
  float* y;  float* out_stats;
  void* scratch_dev; size_t scratch_bytes;
} dmn_conv_args;
int dmn_conv_forward(const dmn_conv_args* a, void* stream);
size_t dmn_conv_scratch_bytes(const dmn_conv_args* a);
/* The same convolution over the channel concatenation cat(x, x2) [ResnetBlock of the up path, unet.py cat((x, h.pop()), dim=1)]:
 * a->cin = C1 + C2 is the total, a->x holds the first C1 = cin - cin2 channels ([batch][C1][hin][win]), x2 the other cin2
 * ([batch][cin2][hin][win]), a->w is the concat weight [cout][cin][k][k].  Plain operand only: a->gn_groups must be 0 (DMN_EINVAL
 * otherwise).  Scratch as for dmn_conv_forward (dmn_conv_scratch_bytes(a)). */
int dmn_conv_forward_cat(const dmn_conv_args* a, const float* x2, int32_t cin2, void* stream);

/* LinearAttention core (mha.py:44-58, between to_qkv and to_out) / Attention core (mha.py:16-29).
 * qkv fp32 NCHW [batch, 3*heads*dim_head, H, W] -> out fp32 NCHW [batch, heads*dim_head, H, W]. */
int dmn_linear_attention_core(const float* qkv, float* out, int batch, int heads, int dim_head, int n_tokens,
                              int act, void* scratch_dev, size_t scratch_bytes, void* stream);
int dmn_attention_core(const float* qkv, float* out, int batch, int heads, int dim_head, int n_tokens,
                       int act, void* scratch_dev, size_t scratch_bytes, void* stream);

/* Self-test of the tcgen05/TMEM/bulk-copy plumbing on a plain GEMM D[M,N] = A[M,K] * B[N,K]^T (bf16 in,
 * fp32 out; all device pointers).  Used by tests to pin the UMMA descriptor encodings. */
int dmn_selftest_umma_gemm(const void* a_bf16, const void* b_bf16, float* d, int M, int N, int K, void* stream);

/* Self-test of the TMA tensor copies (cp.async.bulk.tensor.2d, 128-byte swizzle) + SWIZZLE_128B UMMA descriptors used by the fused
 * attention kernel: D[M,N] = A[M,K] * B[N,K]^T, row-major bf16 in, fp32 out, K a multiple of 64 (all device pointers). */
int dmn_selftest_tma_sw128_gemm(const void* a_bf16, const void* b_bf16, float* d, int M, int N, int K, void* stream);

/* Residual(PreNorm(dim, LinearAttention(dim))) (utils.py:68-93, parts/mha.py:33-59) through the fused tcgen05 kernel:
 *   y = GroupNorm(1)(to_out(linear_attention(to_qkv(GroupNorm(1)(x))))) + x,   heads = 4, dim_head = 32.
 * x / y fp32 NCHW [batch, dim, H, W] with H*W a multiple of 128 and dim in {128, 256}; parameters fp32 in PyTorch layout (device):
 * norm_w / norm_b [dim] (PreNorm), w_qkv [384, dim], w_out [dim, 128], b_out [dim], out_norm_w / out_norm_b [dim].
 * scratch_dev >= dmn_linear_attention_block_scratch_bytes().  Validation path (host repack, sync copies). */
typedef struct dmn_attn_block_args {
  int32_t batch, dim, n_tokens;
  int32_t softmax;         /* 0: LinearAttention block (above).  1: Residual(PreNorm(Attention)) (parts/mha.py:8-30, the bottleneck softmax
                              attention): y = to_out(softmax attention) + x, at most 64 tokens; w_out / b_out are to_out.weight / .bias,
                              out_norm_w / out_norm_b are unused */
  const float* x;
  const float* norm_w; const float* norm_b;
  const float* w_qkv;
  const float* w_out; const float* b_out;
  const float* out_norm_w; const float* out_norm_b;
  float* y;
  void* scratch_dev; size_t scratch_bytes;
} dmn_attn_block_args;
int dmn_linear_attention_block(const dmn_attn_block_args* a, void* stream);
size_t dmn_linear_attention_block_scratch_bytes(const dmn_attn_block_args* a);

/* Unet.init_conv (unet.py:41, 7x7 pad 3) with the class embedding of unet.py:133-137 added in its epilogue:
 *   y[b] = conv7x7(x[b]) + bias + cls_w[classes ? classes[b] : pad_class]       (cls_w NULL: no class term)
 * x fp32 NCHW [batch][cin][size][size] (the sampler state), w [cout][cin][7][7], bias [cout], cls_w [rows][cout], classes int64
 * [batch]; y fp32 NCHW [batch][cout][size][size] holding the act-typed values the engine stores.  Dispatch as the plan's:
 * engine DMN_CONV_TCGEN05 and a shape the tensor-core stem supports -> tensor-core stem (bf16 out), otherwise the CUDA-core stem
 * in `act`.  scratch_dev >= dmn_init_conv_scratch_bytes().  Validation path (host repack, sync copies). */
typedef struct dmn_init_conv_args {
  int32_t batch, cin, size, cout;
  int32_t act, engine;
  int32_t pad_class;
  const float* x; const float* w; const float* bias;
  const float* cls_w; const int64_t* classes;
  float* y;
  void* scratch_dev; size_t scratch_bytes;
} dmn_init_conv_args;
int dmn_init_conv_forward(const dmn_init_conv_args* a, void* stream);
size_t dmn_init_conv_scratch_bytes(const dmn_init_conv_args* a);

/* The ResnetBlock / attention-block epilogue (parts/convnext.py:35-45,86; utils.py:68-93):
 *   y = act(GroupNorm(groups)(raw) * gamma + beta) + res        act = SiLU if silu, else identity; res optional (NULL)
 * raw / res / y fp32 NCHW [batch][channels][hw] (y holds the act-typed values the engine stores).  The input statistics are the
 * engine's fixed-point sums stats[batch][groups][2] = {round(sum * 2^24), round(sum of squares * 2^20)} (int64, device); with
 * ogroups > 0 the call also returns the engine's fixed-point sums of y over ogroups groups in out_stats[batch][ogroups][2]
 * (zeroed by the call, then accumulated by the kernel).  scratch_dev >= dmn_gn_finalize_scratch_bytes(). */
typedef struct dmn_gn_finalize_args {
  int32_t batch, channels, hw, groups, ogroups, silu, act;
  const float* raw; const float* res;
  const int64_t* stats;
  const float* gamma; const float* beta;
  float* y;
  int64_t* out_stats;
  void* scratch_dev; size_t scratch_bytes;
} dmn_gn_finalize_args;
int dmn_gn_finalize_forward(const dmn_gn_finalize_args* a, void* stream);
size_t dmn_gn_finalize_scratch_bytes(const dmn_gn_finalize_args* a);

/* The final_conv tail (unet.py:109-116): eps = conv1x1(SiLU(GroupNorm(groups)(y) * gamma + beta)) + bias, or with `plain`
 * ('conv_bn_act' tail) eps = conv1x1(y) + bias (stats / gamma / beta unused).  y fp32 NCHW [batch][channels][hw], stats as for
 * dmn_gn_finalize_forward, w [cout][channels], bias [cout]; eps fp32 NCHW [batch][cout][hw].
 * With x != NULL the call runs the DDPM sampling loop's fused tail instead: the same projection followed by dmn_ddpm_step's update
 * with coef row `step`, injected noise z (or, z NULL, the Philox draws of `rng` at loop step `step`), x_out = x_{t-1}
 * [batch][cout][hw]; eps is then not written.  DMN_ENOTSUP where the plan would not fuse the tail.
 * scratch_dev >= dmn_final_proj_scratch_bytes(). */
typedef struct dmn_final_proj_args {
  int32_t batch, channels, hw, cout, groups, plain, act;
  const float* y;
  const int64_t* stats;
  const float* gamma; const float* beta;
  const float* w; const float* bias;
  float* eps;
  const float* x; const float* coef; const float* z;
  int32_t step;
  dmn_rng rng;
  float* x_out;
  void* scratch_dev; size_t scratch_bytes;
} dmn_final_proj_args;
int dmn_final_proj_forward(const dmn_final_proj_args* a, void* stream);
size_t dmn_final_proj_scratch_bytes(const dmn_final_proj_args* a);

#ifdef __cplusplus
}
#endif
#endif /* DMN_B200_H */

"""WaveGrad-style continuous-noise-level sampler: drop-in for reference modules/wavegrad_diffusion.py::WaveGradDiffusion.

The reference class only overrides the tables, `q_sample`, `predict_start_from_noise` and `p_mean_variance`; sampling runs
through the p_sample / p_sample_loop it inherits from GaussianDiffusion (its own overrides are commented out,
wavegrad_diffusion.py:219-226).  Differences from DDPM on the hot path:
  * the denoiser is called with the CONTINUOUS noise level sqrt_alphas_cumprod_prev[t + 1] as a [B,1,1,1] float tensor instead
    of the integer timestep (wavegrad_diffusion.py:169-172);
  * x0 = sqrt_recip_alphas_cumprod * x - sqrt_alphas_cumprod_m1 * eps with sqrt_alphas_cumprod_m1 = sqrt(1 - acp) * sqrt(1 / acp)
    (:106,150-158) -- same value as DDPM's sqrt(1/acp - 1) in exact arithmetic, different fp32 rounding, so the table is built
    with the reference's op order and fed to the SAME fused update kernel (dmn_ddpm_step) as a coefficient column.
The denoiser is this package's WaveGradUNet (reference modules/unet.py:171-266) -- then the whole loop runs natively: the FiLM
positional encodings of all T noise levels are tabulated once, and ONE CUDA graph (U-Net + fused update) is replayed T times --
or any other callable (x, noise_level) -> eps, which is called per step while the update stays the fused kernel.
"""
import copy
from typing import Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import _runtime as R
from .gaussian_diffusion import GaussianDiffusion
from .unet import WaveGradUNet


class WaveGradDiffusion(GaussianDiffusion):
    def __init__(self, timesteps: int, schedule_name: str, schedule_cfg=None, objective: str = "pred_noise"):
        super().__init__(timesteps=timesteps, schedule_name=schedule_name, schedule_cfg=schedule_cfg, objective=objective)
        self.original_timesteps = timesteps
        self.original_schedule_name = schedule_name
        self.original_schedule_cfg = copy.deepcopy(schedule_cfg)
        self.compute_constants(self.timesteps)

    def calculate_bits_per_dimension(self, *args, **kwargs):
        """Not built: the inherited evaluation feeds integer timesteps to the denoiser and uses the DDPM x0 coefficients, both wrong for
        the continuous-noise-level WaveGrad parameterisation (reference wavegrad_diffusion.py:150-189)."""
        raise NotImplementedError("bits-per-dimension evaluation is not defined for WaveGradDiffusion in this package")

    # ---- tables (reference wavegrad_diffusion.py:101-106) -------------------------------------------------
    def compute_constants(self, timesteps, verbose: bool = True):
        super().compute_constants(timesteps)
        self.sqrt_alphas_cumprod_prev = torch.sqrt(F.pad(self.alphas_cumprod, (1, 0), value=1.0))
        self.sqrt_alphas_cumprod_m1 = torch.sqrt(1.0 - self.alphas_cumprod) * self.sqrt_recip_alphas_cumprod

    def change_noise_schedule(self, schedule_name: str = None, schedule_cfg: dict = None, reset_cfg: bool = False, verbose: bool = True):
        """reference wavegrad_diffusion.py:35-55 (bookkeeping only; call compute_constants afterwards as the reference does)."""
        if reset_cfg:
            self.schedule_name = self.original_schedule_name
            self.schedule_cfg = copy.deepcopy(self.original_schedule_cfg)
        self.schedule_name = self.schedule_name if schedule_name is None else schedule_name
        self.schedule_cfg = self.schedule_cfg if schedule_cfg is None else schedule_cfg

    def sample_continuous_noise_level(self, batch_size: int, device):
        """reference wavegrad_diffusion.py:120-131 (training-time helper; numpy RNG as in the reference)."""
        s = np.random.randint(1, self.timesteps + 1, size=batch_size)
        lv = torch.tensor(np.random.uniform(self.sqrt_alphas_cumprod_prev[s - 1], self.sqrt_alphas_cumprod_prev[s], size=batch_size),
                          dtype=torch.float32).to(device)
        return lv.view(-1, 1, 1, 1)

    def q_sample(self, x_start, continuous_sqrt_alpha_cumprod=None, noise=None):
        """reference wavegrad_diffusion.py:133-148."""
        lv = (self.sample_continuous_noise_level(x_start.size(0), device=x_start.device).to(x_start)
              if noise is None else continuous_sqrt_alpha_cumprod)
        if noise is None:
            noise = torch.randn_like(x_start)
        return lv * x_start + (1.0 - lv ** 2).sqrt() * noise

    def predict_start_from_noise(self, x_t, t, noise):
        a = self.extract(self.sqrt_recip_alphas_cumprod, t, x_t.shape)
        b = self.extract(self.sqrt_alphas_cumprod_m1, t, noise.shape)
        return a * x_t - b * noise

    def noise_level(self, t: torch.Tensor, shape) -> torch.Tensor:
        return self.extract(self.sqrt_alphas_cumprod_prev, t + 1, shape)

    def p_mean_variance(self, model, x, t, model_output=None, noise_level=None, return_pred_x_start: bool = False):
        """reference wavegrad_diffusion.py:160-189 (torch semantics; note the reference always re-evaluates the model)."""
        if noise_level is None:
            noise_level = self.noise_level(t, x.shape)
        model_output = model(x, noise_level)
        x_recon = self.predict_start_from_noise(x, t, model_output) if self.objective == "pred_noise" else model_output
        x_recon = x_recon.clamp(-1.0, 1.0)
        mean, logvar = self.q_posterior(x_start=x_recon, x=x, t=t)
        return (mean, None, logvar, x_recon) if return_pred_x_start else (mean, None, logvar)

    # ---- hot path: fused update kernel with the WaveGrad x0 coefficient --------------------------------------
    def _step_rows(self, ts: torch.Tensor):
        rows = super()._step_rows(ts)
        rows[1] = self.sqrt_alphas_cumprod_m1[ts]
        return rows

    def _loop_tables(self, ts: torch.Tensor, device):
        """Coefficient rows + the denoiser's per-step argument: the continuous noise level sqrt_alphas_cumprod_prev[t + 1]
        (reference wavegrad_diffusion.py:169-172) instead of the integer timestep."""
        coef, _ = super()._loop_tables(ts, device)
        key = ("levels", str(device), tuple(ts[:: max(1, len(ts) // 5)].tolist()), len(ts))
        lv = self._coef_cache.get(key)
        if lv is None:
            lv = self.sqrt_alphas_cumprod_prev[ts + 1].to(torch.float32).to(device)
            self._coef_cache[key] = lv
        return coef, lv

    def _model_arg(self, ti: int, b: int, device):
        lv = self.sqrt_alphas_cumprod_prev[ti + 1]
        return torch.full((b, 1, 1, 1), float(lv), dtype=torch.float32, device=device)

    @torch.no_grad()
    def p_sample(self, model, x, t, noise=None):
        ti = self._uniform_t(t)
        return self._fused_step(x, model(x, self._model_arg(ti, x.shape[0], x.device)), torch.tensor([ti], dtype=torch.long), noise=noise)

    @torch.no_grad()
    def p_sample_loop(self, model, shape, device=None, use_tqdm=True, noise=None, img=None, start: Optional[int] = None):
        unet, _ = R.resolve_model(model)
        if unet is not None and not isinstance(unet, WaveGradUNet):
            raise NotImplementedError("WaveGradDiffusion drives a (x, noise_level) denoiser; the native Unet takes timesteps. "
                                      "Pass this package's WaveGradUNet (native loop) or any other (x, noise_level) callable")
        return super().p_sample_loop(model, shape, device=device, use_tqdm=use_tqdm, noise=noise, img=img, start=start)

    def inpaint(self, model, x_known, mask, device=None, noise=None, jump_length: int = 1, jump_n_sample: int = 1):
        raise NotImplementedError("WaveGradDiffusion has no inpaint(): use GaussianDiffusion, LearnedGaussianDiffusion or "
                                  "GeneralizedGaussianDiffusion")

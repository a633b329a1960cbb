"""Improved-DDPM learned-variance sampler: drop-in for reference modules/learned_gaussian_diffusion.py."""
import torch

from .. import _lib as L
from .gaussian_diffusion import GaussianDiffusion, _default


class LearnedGaussianDiffusion(GaussianDiffusion):
    """The U-Net emits 2C channels (eps, v); log-variance = v-interpolation between log(beta_t) and the clipped
    posterior log-variance, per pixel (reference learned_gaussian_diffusion.py:36-43)."""

    _loop_kind = L.LOOP_LEARNED
    _out_widths = (2,)

    def __init__(self, timesteps: int, schedule_name: str, schedule_cfg=None, objective: str = "pred_noise"):
        super().__init__(timesteps=timesteps, schedule_name=schedule_name, schedule_cfg=schedule_cfg, objective=objective)

    def _step_rows(self, ts):
        mask = 1 - (ts == 0).float()
        return [self.sqrt_recip_alphas_cumprod[ts], self.sqrt_recipm1_alphas_cumprod[ts], self.posterior_mean_coef1[ts],
                self.posterior_mean_coef2[ts], mask, self.posterior_log_variance_clipped[ts], torch.log(self.betas)[ts]]

    def p_mean_variance(self, model, x, t, model_output=None, return_pred_x_start: bool = False):
        model_output = _default(model_output, lambda: model(x, t))
        eps, v = model_output.chunk(2, dim=1)
        lo = self.extract(self.posterior_log_variance_clipped, t, x.shape)
        hi = self.extract(torch.log(self.betas), t, x.shape)
        frac = (v + 1) * 0.5
        logvar = frac * hi + (1 - frac) * lo
        x0 = self.predict_start_from_noise(x_t=x, t=t, noise=eps).clamp(-1.0, 1.0)
        mean, _ = self.q_posterior(x0, x, t)
        return (mean, logvar.exp(), logvar, x0) if return_pred_x_start else (mean, logvar.exp(), logvar)

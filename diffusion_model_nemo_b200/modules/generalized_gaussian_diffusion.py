"""DDIM (eta in [0,1]) strided sampler: drop-in for reference modules/generalized_gaussian_diffusion.py."""
from typing import Optional

import torch

from .. import _lib as L
from . import _runtime as R
from .gaussian_diffusion import GaussianDiffusion, _default


def strided_pairs(timesteps: int, steps: int):
    """[(t, t_next)] in visiting order (reference :110-112,119): stride = timesteps // steps, the last t_next is -1."""
    stride = timesteps // steps
    seq = list(range(0, timesteps, stride))
    return list(zip(reversed(seq), reversed([-1] + seq[:-1])))


class GeneralizedGaussianDiffusion(GaussianDiffusion):
    _loop_kind = L.LOOP_DDIM

    def __init__(self, timesteps: int, schedule_name: str, schedule_cfg=None, objective: str = "pred_noise", eta: float = 0.0,
                 ddim_timesteps: int = -1):
        super().__init__(timesteps=timesteps, schedule_name=schedule_name, schedule_cfg=schedule_cfg, objective=objective)
        if not (0.0 <= eta <= 1.0):
            raise ValueError("`eta` must be a value in [0, 1]. 0 = DDIM and 1 = DDPM mode")
        self.eta = eta
        self.ddim_timesteps = ddim_timesteps if ddim_timesteps > 0 else self.timesteps
        self.compute_constants(self.timesteps)

    def compute_constants(self, timesteps):
        super().compute_constants(timesteps)
        # abar with a leading 1: index t+1 == abar_t, index 0 == 1 (reference generalized_gaussian_diffusion.py:106-108)
        self.betas_extended = torch.cat([torch.zeros(1), self.betas], dim=0)
        self.alphas_extended = 1.0 - self.betas_extended
        self.alphas_extended_cumprod = self.alphas_extended.cumprod(dim=0)

    def timestep_pairs(self):
        """[(t, t_next)] in visiting order (reference :110-112,119): stride = T // ddim_timesteps."""
        return strided_pairs(self.timesteps, self.ddim_timesteps)

    def _pair_rows(self, t: torch.Tensor, t_next: torch.Tensor):
        at = self.alphas_extended_cumprod[t + 1]
        an = self.alphas_extended_cumprod[t_next + 1]
        c1 = self.eta * torch.sqrt((1.0 - at / an) * (1.0 - an) / (1.0 - at))
        c2 = torch.sqrt((1.0 - an) - c1 ** 2)
        flag = torch.full_like(at, 1.0 if self.objective == "pred_x0" else 0.0)
        return [(1.0 - at).sqrt(), at.sqrt(), an.sqrt(), c1, c2, flag]

    def generalized_predict_start_from_noise(self, x_t, t, noise):
        assert x_t.shape == noise.shape, f"{x_t.shape} != {noise.shape}"
        a = self.extract(self.alphas_extended_cumprod, t + 1, x_t.shape)
        return (x_t - noise * (1.0 - a).sqrt()) / a.sqrt()

    def p_mean_variance(self, model, x, t, model_output=None, return_pred_x_start: bool = False):
        model_output = _default(model_output, lambda: model(x, t))
        x0 = self.generalized_predict_start_from_noise(x, t, model_output) if self.objective == "pred_noise" else model_output
        x0 = x0.clamp(-1.0, 1.0)
        mean, logvar = self.q_posterior(x_start=x0, x=x, t=t)
        return (mean, None, logvar, x0) if return_pred_x_start else (mean, None, logvar)

    @torch.no_grad()
    def p_sample(self, model, x, t, t_next, noise=None):
        """(x_next, x0) for one DDIM transition (reference :75-95)."""
        ti, tn = self._uniform_t(t), self._uniform_t(t_next)
        R.require_cuda(x.device)
        mo = model(x, t).float().contiguous()
        coef = R.coef_rows(self._pair_rows(torch.tensor([ti]), torch.tensor([tn])), x.device)
        out = torch.empty_like(x, dtype=torch.float32)
        with torch.cuda.device(x.device):
            R.launch_step(L.LOOP_DDIM, x.float().contiguous(), mo, None if noise is None else noise.float().contiguous(), out, coef, 0,
                          L.Rng(R.draw_seed(), R.rank_stream_id()), L.stream_ptr(x.device))
        x0 = self.generalized_predict_start_from_noise(x, t, mo).clamp(-1.0, 1.0) if self.objective == "pred_noise" else mo.clamp(-1, 1)
        return out, x0

    def _loop_tables(self, ts, device):
        pairs = self.timestep_pairs()
        key = (str(device), self.eta, self.ddim_timesteps, self.timesteps, self.objective)
        hit = self._coef_cache.get(key)
        if hit is None:
            t = torch.tensor([p[0] for p in pairs], dtype=torch.long)
            tn = torch.tensor([p[1] for p in pairs], dtype=torch.long)
            hit = (R.coef_rows(self._pair_rows(t, tn), device), t.to(torch.float32).to(device))
            self._coef_cache[key] = hit
        return hit

    def _visit_order(self, start=None):
        return torch.tensor([p[0] for p in self.timestep_pairs()], dtype=torch.long)

    @torch.no_grad()
    def p_sample_loop(self, model, shape, use_tqdm=True, img=None, device=None, noise=None):
        return super().p_sample_loop(model, shape, device=device, use_tqdm=use_tqdm, noise=noise, img=img)

    @torch.no_grad()
    def sample(self, model, shape, device=None, noise=None):
        return self.p_sample_loop(model, shape=shape, device=device, noise=noise)

    @torch.no_grad()
    def interpolate(self, model, x, t: Optional[int] = None, noise=None):
        """Deterministic decode of a given latent x (reference :139-140)."""
        return self.p_sample_loop(model, x.shape, img=x, device=x.device, noise=noise)

"""Score-SDE predictor-corrector sampling: drop-in for the reference's
modules/sde_lib/{sde_lib,vp_sde,ve_sde}.py, modules/sde_predictors/*, modules/sde_correctors/*,
modules/sde_samplers/predictor_corrector_sampler.py and loss/sde_loss/score_function_loss.py::resolve_score_function.

Every built-in predictor / corrector update is affine in (x, model output, z) once the time step is fixed, so the
host folds the SDE algebra (discretisation, score wrapper `-model/std`, step sizes) into per-step coefficient rows
computed with the reference's torch CPU ops, and the device runs ONE fused kernel per update
(dmn_affine_noise_step / dmn_langevin_step).  With this package's Unet the whole N-step loop is a CUDA graph.

ProbabilityFlowSampler (modules/sde_samplers/probability_flow_sampler.py) solves the probability-flow ODE with scipy's RK45
rules on the device (dmn_ode_sample): the step control runs in device code, so the adaptive solve is one CUDA graph.
LikelihoodEstimate (score_sde's get_likelihood_fn) runs the same solver over [x ; delta_logp] with a forward-mode JVP of the fp32
Unet per evaluation for the Hutchinson divergence (dmn_ode_likelihood).
DPMSolverSampler (not in the reference) is few-step DPM-Solver++ / SDE-DPM-Solver++ sampling of VP and VE score models on the
DPM-Solver++ loop of DPMSolverDiffusion (dmn_dpmpp_step / dmn_dpmpp_sde_step, DMN_LOOP_DPMPP).
"""
import abc
import ctypes as C
import math
import warnings
from typing import List, Optional

import numpy as np
import torch

from .. import _lib as L
from . import _runtime as R
from .dpm_solver_diffusion import multistep_coefs

# ------------------------------------------------------------------------------------------------------
# SDEs (tables are CPU fp32, reference op order => bit-exact)
# ------------------------------------------------------------------------------------------------------


class SDE(abc.ABC):
    sampling_epsilon: float = None

    def __init__(self, N):
        super().__init__()
        self.N = N
        if self.sampling_epsilon is None:
            raise ValueError("Sampling epsilon cannot be None ! Must be set as a class variable !")

    @property
    @abc.abstractmethod
    def T(self):
        pass

    @abc.abstractmethod
    def sde(self, x, t):
        pass

    @abc.abstractmethod
    def marginal_prob(self, x, t):
        pass

    @abc.abstractmethod
    def prior_sampling(self, shape):
        pass

    def discretize(self, x, t):
        """Euler-Maruyama default (reference sde_lib.py:53-67)."""
        dt = 1 / self.N
        drift, diffusion = self.sde(x, t)
        return drift * dt, diffusion * torch.sqrt(torch.tensor(dt, device=t.device))


class VPSDE(SDE):
    sampling_epsilon = 1e-3

    def __init__(self, beta_min=0.1, beta_max=20, N=1000):
        super().__init__(N)
        self.beta_0, self.beta_1, self.N = beta_min, beta_max, N
        self.compute_constants(N)

    def compute_constants(self, timesteps):
        self.betas = torch.linspace(self.beta_0 / timesteps, self.beta_1 / timesteps, timesteps)
        self.alphas = 1.0 - self.betas
        self.alphas_cumprod = torch.cumprod(self.alphas, dim=0)
        self.sqrt_alphas_cumprod = torch.sqrt(self.alphas_cumprod)
        self.sqrt_1m_alphas_cumprod = torch.sqrt(1.0 - self.alphas_cumprod)

    @property
    def T(self):
        return 1

    def sde(self, x, t):
        beta_t = self.beta_0 + t * (self.beta_1 - self.beta_0)
        return -0.5 * beta_t[:, None, None, None] * x, torch.sqrt(beta_t)

    def marginal_prob(self, x, t):
        lmc, std = _vp_log_mean_std(self, t)
        return torch.exp(lmc[:, None, None, None]) * x, std

    def prior_sampling(self, shape):
        return torch.randn(*shape)

    def prior_logp(self, z):
        n = np.prod(z.shape[1:])
        return -n / 2.0 * np.log(2 * np.pi) - torch.sum(z ** 2, dim=(1, 2, 3)) / 2.0

    def discretize(self, x, t):
        ts = (t * (self.N - 1) / self.T).long()
        beta = self.betas.to(x.device)[ts]
        alpha = self.alphas.to(x.device)[ts]
        return torch.sqrt(alpha)[:, None, None, None] * x - x, torch.sqrt(beta)


def _vp_log_mean_std(sde: VPSDE, t):
    """(log mean coefficient, std) of the VP marginal p(x_t | x_0) at the times t, in the reference's op order (vp_sde.py
    marginal_prob), so that every table built from it is bit-identical to the reference's."""
    lmc = -0.25 * t ** 2 * (sde.beta_1 - sde.beta_0) - 0.5 * t * sde.beta_0
    return lmc, torch.sqrt(1.0 - torch.exp(2.0 * lmc))


class VESDE(SDE):
    sampling_epsilon = 1e-5

    def __init__(self, sigma_min=0.01, sigma_max=50, N=1000):
        super().__init__(N)
        self.sigma_min, self.sigma_max, self.N = sigma_min, sigma_max, N
        self.discrete_sigmas = torch.exp(torch.linspace(np.log(self.sigma_min), np.log(self.sigma_max), N))

    @property
    def T(self):
        return 1

    def sde(self, x, t):
        sigma = self.sigma_min * (self.sigma_max / self.sigma_min) ** t
        g = sigma * torch.sqrt(torch.tensor(2 * (np.log(self.sigma_max) - np.log(self.sigma_min)), device=t.device))
        return torch.zeros_like(x), g

    def marginal_prob(self, x, t):
        return x, self.sigma_min * (self.sigma_max / self.sigma_min) ** t

    def prior_sampling(self, shape):
        return torch.randn(*shape) * self.sigma_max

    def prior_logp(self, z):
        n = np.prod(z.shape[1:])
        return -n / 2.0 * np.log(2 * np.pi * self.sigma_max ** 2) - torch.sum(z ** 2, dim=(1, 2, 3)) / (2 * self.sigma_max ** 2)

    def discretize(self, x, t):
        ts = (t * (self.N - 1) / self.T).long()
        sig = self.discrete_sigmas.to(t.device)[ts]
        adj = torch.where(ts == 0, torch.zeros_like(t), self.discrete_sigmas.to(t.device)[ts - 1])
        return torch.zeros_like(x), torch.sqrt(sig ** 2 - adj ** 2)


def init_scale(sde: SDE) -> float:
    """Factor from an N(0, I) draw to x_T: the prior of a VE SDE has std sigma_max, a VP prior is N(0, I)."""
    return float(sde.sigma_max) if isinstance(sde, VESDE) else 1.0


def _checked_sde(sde: Optional[SDE], call: str = "forward()") -> SDE:
    """The SDE a sampler was given with update_sde; the native samplers are built for VP and VE."""
    if sde is None:
        raise ValueError(f"Must explicitly set `update_sde(sde)` for this module prior to calling {call}")
    if not isinstance(sde, (VPSDE, VESDE)):
        raise NotImplementedError(f"SDE class {sde.__class__.__name__} not yet supported.")
    return sde


# ------------------------------------------------------------------------------------------------------
# score wrapper (reference loss/sde_loss/score_function_loss.py:47-91, continuous=True)
# ------------------------------------------------------------------------------------------------------


class ScoreFunction:
    """score(x, t) = scale(t) * model(x, labels(t));  VP: labels = t*(N-1), scale = -1/std(t);  VE: labels = sigma(t), scale = 1."""

    def __init__(self, model, sde, continuous=True):
        if not isinstance(sde, (VPSDE, VESDE)):
            raise NotImplementedError(f"SDE class {sde.__class__.__name__} not yet supported.")
        if not continuous:
            raise NotImplementedError("continuous=False score models are outside the built sampling path")
        self.model, self.sde = model, sde

    def labels(self, t):
        if isinstance(self.sde, VPSDE):
            return t * (self.sde.N - 1)
        return self.sde.marginal_prob(None, t)[1]

    def scale(self, t):
        if isinstance(self.sde, VPSDE):
            return -1.0 / _vp_log_mean_std(self.sde, t)[1]
        return torch.ones_like(t)

    def raw(self, x, t):
        return self.model(x, self.labels(t))

    def __call__(self, x, t):
        return self.raw(x, t) * self.scale(t)[:, None, None, None]


def resolve_score_function(model, sde, continuous=True):
    return ScoreFunction(model, sde, continuous)


# ------------------------------------------------------------------------------------------------------
# per-step coefficient algebra (host, fp32 torch CPU ops in the reference's order)
# ------------------------------------------------------------------------------------------------------


def _ts_index(sde, t):
    return (t * (sde.N - 1) / sde.T).long()


def _alpha(sde, t):
    if isinstance(sde, VPSDE):
        return sde.alphas[_ts_index(sde, t)]
    return torch.ones_like(t)


def predictor_rows(name: Optional[str], sde, sf: ScoreFunction, t: torch.Tensor, probability_flow: bool = False):
    """x_mean = a*x + b*model_out ; x = x_mean + g*z   -> columns (a, b, g) for the time vector t (CPU fp32).
    probability_flow=True is the reference's RSDE with the halved score term and no diffusion (sde_lib.py:91-105): g = 0, but the
    update still takes its z, so the draw order is unchanged."""
    scale = sf.scale(t)
    if name in (None, "none", "null"):
        return [torch.ones_like(t), torch.zeros_like(t), torch.zeros_like(t)]
    if name == "reverse_diffusion":         # reverse_diffusion_predictor.py:11-16 + sde_lib.py:100-105
        ts = _ts_index(sde, t)
        if isinstance(sde, VPSDE):
            G = torch.sqrt(sde.betas[ts])
            a = 2.0 - torch.sqrt(sde.alphas[ts])        # x - (sqrt(alpha) x - x)
        else:
            sig = sde.discrete_sigmas[ts]
            adj = torch.where(ts == 0, torch.zeros_like(t), sde.discrete_sigmas[ts - 1])
            G = torch.sqrt(sig ** 2 - adj ** 2)
            a = torch.ones_like(t)
        if probability_flow:
            return [a, G ** 2 * scale * 0.5, torch.zeros_like(t)]
        return [a, G ** 2 * scale, G]
    if name == "euler_maruyama":            # euler_maruyama_predictor.py:11-17 + sde_lib.py:91-98
        dt = -1.0 / sde.N
        if isinstance(sde, VPSDE):
            beta_t = sde.beta_0 + t * (sde.beta_1 - sde.beta_0)
            diff = torch.sqrt(beta_t)
            a = 1.0 + (-0.5 * beta_t) * dt
        else:
            sigma = sde.sigma_min * (sde.sigma_max / sde.sigma_min) ** t
            diff = sigma * torch.sqrt(torch.tensor(2 * (np.log(sde.sigma_max) - np.log(sde.sigma_min))))
            a = torch.ones_like(t)
        if probability_flow:
            return [a, -(diff ** 2) * scale * 0.5 * dt, torch.zeros_like(t)]
        return [a, -(diff ** 2) * scale * dt, diff * np.sqrt(-dt)]
    raise NotImplementedError(f"predictor `{name}` has no native update (built: reverse_diffusion, euler_maruyama, none)")


def corrector_rows(name: Optional[str], sde, sf: ScoreFunction, t: torch.Tensor, snr: float):
    """langevin -> (kind 0, columns (score_scale, alpha));  ald -> (kind 1, affine columns (1, step*scale, sqrt(2 step)))."""
    scale = sf.scale(t)
    alpha = _alpha(sde, t)
    if name == "langevin":                  # langevin_corrector.py:15-35 (step size needs the batch-mean norms: on device)
        return 0, [scale, alpha]
    if name == "ald":                       # annealed_langevin_dynamics_corrector.py:21-41
        std = sde.marginal_prob(None, t)[1] if isinstance(sde, VESDE) else _vp_log_mean_std(sde, t)[1]
        step = (snr * std) ** 2 * 2 * alpha
        return 1, [torch.ones_like(t), step * scale, torch.sqrt(step * 2)]
    raise NotImplementedError(f"corrector `{name}` has no native update (built: langevin, ald, none)")


# ------------------------------------------------------------------------------------------------------
# predictor / corrector plugin classes and registries (reference base_predictor.py, base_corrector.py)
# ------------------------------------------------------------------------------------------------------

PREDICTOR_REGISTRY = {}
CORRECTOR_REGISTRY = {}


def register_predictor(cls, name=None):
    name = name or cls.__name__
    if name in PREDICTOR_REGISTRY:
        raise ValueError(f"Predictor {name} has already been registered !")
    PREDICTOR_REGISTRY[name] = cls


def get_predictor(name: str):
    return PREDICTOR_REGISTRY.get(name)


def register_corrector(cls, name=None):
    name = name or cls.__name__
    if name in CORRECTOR_REGISTRY:
        raise ValueError(f"Corrector {name} has already been registered !")
    CORRECTOR_REGISTRY[name] = cls


def get_corrector(name: str):
    return CORRECTOR_REGISTRY.get(name)


def _uniform(t):
    tc = t.detach().float().cpu()
    if not bool((tc == tc[0]).all()):
        raise NotImplementedError("fused updates take one time value per call (all entries of t equal)")
    return tc[:1]


def _affine_update(x, mo, rows, noise=None):
    R.require_cuda(x.device)
    coef = R.coef_rows(rows, x.device)
    out, mean = torch.empty_like(x), torch.empty_like(x)
    with torch.cuda.device(x.device):
        L.check(L.lib().dmn_affine_noise_step(L.ptr(x.contiguous()), L.ptr(mo.float().contiguous()),
                                              L.ptr(None if noise is None else noise.float().contiguous()), L.ptr(out), L.ptr(mean),
                                              x.numel(), L.ptr(coef), None, 0, L.Rng(R.draw_seed(), R.rank_stream_id()),
                                              L.stream_ptr(x.device)), "dmn_affine_noise_step")
    return out, mean


class Predictor(abc.ABC):
    native_name: Optional[str] = None

    def __init__(self, sde, score_fn, probability_flow=False):
        super().__init__()
        self.sde, self.score_fn, self.probability_flow = sde, score_fn, probability_flow

    def update_fn(self, x, t, noise=None):
        """(x, x_mean) after one predictor step; one model call + one fused kernel."""
        tc = _uniform(t)
        rows = predictor_rows(self.native_name, self.sde, self.score_fn, tc, self.probability_flow)
        return _affine_update(x.float(), self.score_fn.raw(x, t), rows, noise)

    @classmethod
    def register_predictor(cls, name=None):
        name = name or cls.__name__
        if get_predictor(name) is None:
            register_predictor(cls, name=name)


class NonePredictor(Predictor):
    def __init__(self, sde=None, score_fn=None, probability_flow=False):
        pass

    def update_fn(self, x, t, noise=None):
        return x, x


class ReverseDiffusionPredictor(Predictor):
    native_name = "reverse_diffusion"


class EulerMaruyamaPredictor(Predictor):
    native_name = "euler_maruyama"


class AncestralSamplingPredictor(Predictor):
    def __init__(self, sde, score_fn, probability_flow=False):
        raise NotImplementedError("ancestral_sampling: the reference's VP path raises AttributeError (discrete_betas) and the VE "
                                  "path is CPU-only; out of scope (SURVEY.md section 2, row 7)")


NonePredictor.register_predictor("none")
NonePredictor.register_predictor("null")
ReverseDiffusionPredictor.register_predictor("reverse_diffusion")
EulerMaruyamaPredictor.register_predictor("euler_maruyama")
AncestralSamplingPredictor.register_predictor("ancestral_sampling")


class Corrector(abc.ABC):
    native_name: Optional[str] = None

    def __init__(self, sde, score_fn, snr, n_steps):
        super().__init__()
        if not isinstance(sde, (VPSDE, VESDE)):
            raise NotImplementedError(f"SDE class {sde.__class__.__name__} not yet supported.")
        self.sde, self.score_fn, self.snr, self.n_steps = sde, score_fn, snr, n_steps

    def update_fn(self, x, t, noise=None):
        tc = _uniform(t)
        kind, rows = corrector_rows(self.native_name, self.sde, self.score_fn, tc, self.snr)
        x = x.float()
        x_mean = x
        for i in range(self.n_steps):
            z = None if noise is None else noise[i]
            mo = self.score_fn.raw(x, t)
            if kind == 1:
                x, x_mean = _affine_update(x, mo, rows, z)
            else:
                R.require_cuda(x.device)
                coef = R.coef_rows(rows, x.device)
                out, mean = torch.empty_like(x), torch.empty_like(x)
                scratch = torch.empty(2 * x.shape[0] + 8, dtype=torch.float32, device=x.device)
                with torch.cuda.device(x.device):
                    L.check(L.lib().dmn_langevin_step(L.ptr(x.contiguous()), L.ptr(mo.float().contiguous()),
                                                      L.ptr(None if z is None else z.float().contiguous()), L.ptr(out), L.ptr(mean),
                                                      x.shape[0], x.numel() // x.shape[0], float(self.snr), L.ptr(coef), None, 0,
                                                      L.ptr(scratch), L.Rng(R.draw_seed(), R.rank_stream_id()),
                                                      L.stream_ptr(x.device)), "dmn_langevin_step")
                x, x_mean = out, mean
        return x, x_mean

    @classmethod
    def register_corector(cls, name: str = None):      # [sic] the reference spells it this way (base_corrector.py:54)
        name = name or cls.__name__
        if get_corrector(name) is None:
            register_corrector(cls, name=name)

    register_corrector_cls = register_corector


class NoneCorrector(Corrector):
    def __init__(self, sde=None, score_fn=None, snr=None, n_steps=None):
        pass

    def update_fn(self, x, t, noise=None):
        return x, x


class LangevinCorrector(Corrector):
    native_name = "langevin"


class AnnealedLangevinDynamics(Corrector):
    native_name = "ald"


NoneCorrector.register_corector("none")
NoneCorrector.register_corector("null")
LangevinCorrector.register_corector("langevin")
AnnealedLangevinDynamics.register_corector("ald")

# ------------------------------------------------------------------------------------------------------
# the PC sampler
# ------------------------------------------------------------------------------------------------------

_NATIVE_PREDICTORS = {None: None, "none": None, "null": None, "reverse_diffusion": "reverse_diffusion",
                      "euler_maruyama": "euler_maruyama"}
_NATIVE_CORRECTORS = {None: None, "none": None, "null": None, "langevin": "langevin", "ald": "ald"}


class PredictorCorrectorSampler(torch.nn.Module):
    def __init__(self, predictor: str, corrector: str, snr: float, n_steps: int = 1, probability_flow: bool = False,
                 continuous: bool = True, denoise: bool = True, eps: float = None):
        super().__init__()
        self.predictor, self.corrector, self.snr, self.n_steps = predictor, corrector, snr, n_steps
        self.probability_flow, self.continuous, self.denoise, self.eps = probability_flow, continuous, denoise, eps
        self.sde: Optional[SDE] = None
        self.seed: Optional[int] = None
        self.trajectory_every = 0
        self.use_cuda_graph = True
        self._cache = {}

    def update_sde(self, sde: SDE):
        self.sde = sde
        self._cache = {}

    def timesteps(self):
        eps = self.sde.sampling_epsilon if self.eps is None else self.eps
        return torch.linspace(self.sde.T, eps, self.sde.N)

    def _native_ok(self):
        pred_cls, corr_cls = get_predictor(self.predictor) if self.predictor else None, get_corrector(self.corrector) if self.corrector else None
        builtin_p = self.predictor in _NATIVE_PREDICTORS and (pred_cls is None or pred_cls.__module__ == __name__)
        builtin_c = self.corrector in _NATIVE_CORRECTORS and (corr_cls is None or corr_cls.__module__ == __name__)
        return builtin_p and builtin_c and isinstance(self.sde, (VPSDE, VESDE))

    def forward(self, model, shape: List[int], device, return_nfe: bool = True, use_tqdm: bool = True, noise=None):
        sde = _checked_sde(self.sde)
        R.require_cuda(device)
        ts = self.timesteps()
        sf = ScoreFunction(model, sde, self.continuous)
        unet, classes = R.resolve_model(model)
        n_corr = self.n_steps if _NATIVE_CORRECTORS.get(self.corrector) else 0
        scale = init_scale(sde)
        if unet is not None and self._native_ok():
            key = (str(device), self.predictor, self.corrector, float(self.snr), sde.N, self.eps, bool(self.probability_flow))
            hit = self._cache.get(key)
            if hit is None:
                coef = R.coef_rows(predictor_rows(_NATIVE_PREDICTORS[self.predictor], sde, sf, ts, bool(self.probability_flow)), device)
                kind, coef2 = 0, None
                if n_corr:
                    kind, rows = corrector_rows(_NATIVE_CORRECTORS[self.corrector], sde, sf, ts, self.snr)
                    coef2 = R.coef_rows(rows, device)
                hit = (coef, coef2, kind, sf.labels(ts).to(torch.float32).to(device))
                self._cache[key] = hit
            coef, coef2, kind, labels = hit
            res = R.run_native_loop(unet, kind=L.LOOP_PC, shape=shape, device=device, times=labels, coef=coef, coef2=coef2,
                                    noise=noise, classes=classes, n_corr=n_corr, corr_kind=kind, snr=float(self.snr),
                                    denoise=self.denoise, seed=self.seed, traj_every=self.trajectory_every,
                                    use_graph=self.use_cuda_graph, init_scale=scale)
            final = res.aux if self.denoise else res.final
            imgs = R.to_image_list(final, res.traj)
        else:
            # plugin path: user-registered predictor/corrector classes or a foreign model -> per-step update_fn calls
            pred = (get_predictor(self.predictor) if self.predictor else NonePredictor)(sde, sf, self.probability_flow)
            corr = (get_corrector(self.corrector) if self.corrector else NoneCorrector)(sde, sf, self.snr, self.n_steps)
            k = 0
            if noise is not None:
                x = noise[0].to(device, torch.float32) * scale
                k = 1
            else:
                x = sde.prior_sampling(shape).to(device)
            x_mean = x
            for i in range(sde.N):
                vec_t = torch.ones(shape[0], device=device) * ts[i]
                zc = None if noise is None else noise[k:k + n_corr].to(device)
                zp = None if noise is None else noise[k + n_corr].to(device)
                k += (n_corr + 1) if noise is not None else 0
                x, x_mean = corr.update_fn(x, vec_t, noise=zc) if n_corr else corr.update_fn(x, vec_t)
                x, x_mean = pred.update_fn(x, vec_t, noise=zp)
            imgs = R.to_image_list((x_mean if self.denoise else x).float().contiguous(), None)
        nfe = sde.N * (self.n_steps + 1)
        return (imgs, nfe) if return_nfe else imgs

    def sample(self, model, shape: List[int], device=None, return_nfe: bool = False, noise=None):
        if device is None:
            device = next(model.parameters()).device
        return self.forward(model=model, shape=shape, device=device, return_nfe=return_nfe, noise=noise)


# ------------------------------------------------------------------------------------------------------
# the probability-flow ODE sampler (reference modules/sde_samplers/probability_flow_sampler.py, score_sde get_ode_sampler)
# ------------------------------------------------------------------------------------------------------


def _check_solver_args(method, max_nfe, **scalars):
    """Constructor arguments of the RK45 solvers: every scalar (rtol, atol, eps) finite, > 0 except atol (>= 0)."""
    if method != "RK45":
        raise NotImplementedError(f"method={method!r}: only the RK45 solver is built")
    for name, v in scalars.items():
        if isinstance(v, bool) or not isinstance(v, (int, float, np.floating, np.integer)):
            raise ValueError(f"{name} must be a scalar number (per-component values are not supported), got {type(v).__name__}")
        if not np.isfinite(v) or v < 0 or (name != "atol" and v == 0):
            raise ValueError(f"{name} must be finite and {'>= 0' if name == 'atol' else '> 0'}, got {v}")
    if isinstance(max_nfe, bool) or not isinstance(max_nfe, (int, np.integer)) or max_nfe < 2:
        raise ValueError(f"max_nfe must be an integer >= 2, got {max_nfe!r}")


def _check_ode_unet(unet, shape):
    b, c, h, w = (int(v) for v in shape)
    if c != unet.channels or h != w:
        raise ValueError(f"shape {list(shape)} does not fit the U-Net ({unet.channels} channels, square images)")
    if unet.out_dim != unet.channels:
        raise ValueError("the probability-flow drift needs a U-Net whose output has as many channels as its input")


# per solve: descriptor, work-size query, entry point, plan attribute of its buffers (one set per solve: each has its own graph
# cache), how its errors name it and its end time
_ODE_SOLVES = {
    "sample": (L.OdeDesc, "dmn_ode_work_bytes", "dmn_ode_sample", "_ode_bufs", "probability-flow", "eps"),
    "likelihood": (L.OdeLikelihoodDesc, "dmn_ode_likelihood_work_bytes", "dmn_ode_likelihood", "_lik_bufs", "likelihood", "T"),
}


def _ode_solve(solver, kind: str, unet, classes, x: torch.Tensor, t0: float, t1: float, noise: Optional[torch.Tensor] = None,
               **fields) -> torch.Tensor:
    """One adaptive RK45 solve of solver.sde's probability-flow ODE from t0 to t1 with this package's Unet, on x's device: the
    "sample" solve integrates x, the "likelihood" solve [x ; delta_logp] from delta_logp = 0 with `noise` (optional, x's shape)
    as its Hutchinson noise.  `fields` sets the remaining descriptor fields.  Records solver.last_stats and returns the final
    state (flat, a copy); a solve stopped by max_nfe raises RuntimeError."""
    desc_t, work_bytes, entry, bufs_name, what, end = _ODE_SOLVES[kind]
    sde, lib, device = solver.sde, L.lib(), x.device
    b, h, n = x.shape[0], x.shape[2], x.numel()
    plan = unet.plan(h, b, device, time_rows=6)
    with torch.cuda.device(device):
        st = L.stream_ptr(device)
        # buffers live with the plan so the addresses baked into the cached graph stay valid
        bufs = plan.__dict__.setdefault(bufs_name, {})
        if b not in bufs:
            nbytes = int(getattr(lib, work_bytes)(plan.h, b))
            bufs[b] = {"state": torch.empty(n + (b if kind == "likelihood" else 0), dtype=torch.float32, device=device),
                       "work": torch.empty(nbytes + 256, dtype=torch.uint8, device=device),
                       "result": torch.zeros(3, dtype=torch.float64, device=device)}
        buf = bufs[b]
        state, work, result = buf["state"], buf["work"], buf["result"]
        state[:n].copy_(x.reshape(-1))
        state[n:].zero_()
        d = desc_t()
        if classes is not None:
            d.classes_dev = R.stable_copy(buf, "classes", classes.to(device, torch.int64).reshape(-1)).data_ptr()
        if noise is not None:
            d.noise_dev = R.stable_copy(buf, "noise", noise.to(device, torch.float32).reshape(-1)).data_ptr()
        wp = (work.data_ptr() + 255) // 256 * 256
        if isinstance(sde, VPSDE):
            d.sde_kind, d.N, d.beta_0, d.beta_1 = L.SDE_VP, int(sde.N), float(sde.beta_0), float(sde.beta_1)
        else:
            d.sde_kind, d.N, d.sigma_min, d.sigma_max = L.SDE_VE, int(sde.N), float(sde.sigma_min), float(sde.sigma_max)
        d.t0, d.t1, d.rtol, d.atol = t0, t1, solver.rtol, solver.atol
        d.max_nfe, d.batch, d.use_graph = solver.max_nfe, b, int(bool(solver.use_cuda_graph))
        for k, v in fields.items():
            setattr(d, k, v)
        d.state_dev, d.state_elems = state.data_ptr(), state.numel()
        d.work_dev, d.work_bytes = wp, work.numel() - (wp - work.data_ptr())
        d.result_dev = result.data_ptr()
        L.check(getattr(lib, entry)(plan.h, C.byref(d), st), entry)
        plan.time_rows_key = None            # the solve rewrote rows 0..5 of the time table
        raw = result.cpu().numpy().tobytes()
        out = state.clone()
    res = L.OdeResult.from_buffer_copy(raw)
    solver.last_stats = {"status": int(res.status), "nfev": int(res.nfev), "n_accepted": int(res.n_accepted),
                         "n_rejected": int(res.n_rejected), "t_final": float(res.t_final)}
    if res.status == L.ODE_LIMIT:
        raise RuntimeError(f"{what} ODE: stopped at {res.nfev} model evaluations (max_nfe={solver.max_nfe}) at "
                           f"t={res.t_final:.6g}, before reaching {end}={t1:g}")
    if res.status == L.ODE_TOO_SMALL_STEP:
        warnings.warn(f"{what} ODE: required step size became too small at t={res.t_final:.6g} (scipy status -1); "
                      "returning the last accepted state, as solve_ivp does")
    return out


class ProbabilityFlowSampler(torch.nn.Module):
    """Deterministic sampler of a score-SDE model: integrates the probability-flow ODE dx/dt = f(x,t) - 0.5 g(t)^2 score(x,t) from
    sde.T down to eps with scipy's adaptive RK45 rules (solve_ivp(..., method='RK45')), entirely on the GPU: every model
    evaluation, the error norm, the accept / reject decision and the step-size update run in device code, and with
    `use_cuda_graph` (default) the whole solve is one CUDA graph replay.  Needs this package's Unet (or a
    functools.partial of it with `classes`); any other model callable raises NotImplementedError (there is no host solver).

    Differences to the reference: eps=None uses sde.sampling_epsilon (the reference fails inside solve_ivp); a solve that would
    need more than `max_nfe` model evaluations stops and raises RuntimeError; `last_stats` holds the solver counters of the last
    call.  Step sizes are chosen per process: under torchrun every rank solves its own batch with its own steps."""

    def __init__(self, denoise: bool = False, rtol: float = 1e-5, atol: float = 1e-5, method: str = "RK45", eps: float = None,
                 max_nfe: int = 100_000):
        super().__init__()
        _check_solver_args(method, max_nfe, rtol=rtol, atol=atol)
        self.denoise, self.rtol, self.atol, self.method, self.eps = denoise, float(rtol), float(atol), method, eps
        self.max_nfe = int(max_nfe)
        self.sde: Optional[SDE] = None
        self.use_cuda_graph = True
        self.last_stats: Optional[dict] = None

    def update_sde(self, sde: SDE):
        self.sde = sde

    def forward(self, model, shape: List[int], device, return_nfe: bool = True, use_tqdm: bool = True, noise=None):
        sde = _checked_sde(self.sde)
        R.require_cuda(device)
        device = torch.device(device)
        unet, classes = R.resolve_model(model)
        if unet is None:
            raise NotImplementedError("ProbabilityFlowSampler runs this package's Unet natively; other model callables have no "
                                      "host solver path")
        b, c, h, w = (int(v) for v in shape)
        _check_ode_unet(unet, shape)
        eps = sde.sampling_epsilon if self.eps is None else float(self.eps)
        x = noise[0] * init_scale(sde) if noise is not None else sde.prior_sampling(shape)
        if tuple(x.shape) != (b, c, h, w):
            raise ValueError(f"x_T has shape {tuple(x.shape)}; expected {(b, c, h, w)}")
        x = _ode_solve(self, "sample", unet, classes, x.to(device, torch.float32), float(sde.T), eps).view(b, c, h, w)
        if self.denoise:      # one reverse-diffusion predictor step at eps, probability_flow=False, keeping x_mean
            vec_eps = torch.ones(b, device=device) * eps
            pred = ReverseDiffusionPredictor(sde, ScoreFunction(model, sde), probability_flow=False)
            _, x = pred.update_fn(x, vec_eps)
        imgs = R.to_image_list(x.float().contiguous(), None)
        return (imgs, self.last_stats["nfev"]) if return_nfe else imgs

    def sample(self, model, shape: List[int], device=None, return_nfe: bool = False, noise=None):
        if device is None:
            device = next(model.parameters()).device
        return self.forward(model=model, shape=shape, device=device, return_nfe=return_nfe, noise=noise)


class LikelihoodEstimate(torch.nn.Module):
    """Exact log-likelihood of a score-SDE model under its probability-flow ODE, in bits/dim (score_sde's get_likelihood_fn; the
    reference's modules/sde_lib/likelihood.py): the augmented state [x ; delta_logp] is integrated from eps to sde.T with scipy's
    RK45 rules, where d delta_logp / dt is the Hutchinson estimate eps^T (d drift / dx) eps of the drift's divergence.  Everything
    runs on the GPU: one forward-mode JVP pass of this package's fp32 Unet per evaluation gives both the model output and the
    directional derivative, and with `use_cuda_graph` (default) the whole adaptive solve is one CUDA graph replay.

    likelihood(model, data, noise=None) -> (bpd [B], z [B, C, H, W], nfe).  data is in the model's [-1, 1] space, already
    dequantised; bpd = -(prior_logp(z) + delta_logp) / ln 2 / D + 7 (score_sde's offset 7 - inverse_scaler(-1) for centred
    data).  `noise` injects the Hutchinson noise; otherwise it is drawn once per call by the in-kernel Philox generator keyed by
    (`seed` or a draw from torch's CPU generator, data-parallel rank).  Needs this package's Unet in fp32 (compute_dtype='fp32')."""

    def __init__(self, hutchinson_type: str = "Rademacher", rtol: float = 1e-5, atol: float = 1e-5, method: str = "RK45",
                 eps: float = 1e-5, max_nfe: int = 100_000):
        super().__init__()
        if hutchinson_type not in ("Rademacher", "Gaussian"):
            raise NotImplementedError(f"Hutchinson type {hutchinson_type} unknown.")
        _check_solver_args(method, max_nfe, rtol=rtol, atol=atol, eps=eps)
        self.hutchinson_type, self.rtol, self.atol, self.method = hutchinson_type, float(rtol), float(atol), method
        self.eps, self.max_nfe = float(eps), int(max_nfe)
        self.sde: Optional[SDE] = None
        self.seed: Optional[int] = None
        self.use_cuda_graph = True
        self.last_stats: Optional[dict] = None

    def update_sde(self, sde: SDE):
        self.sde = sde

    def likelihood(self, model, data: torch.Tensor, noise: Optional[torch.Tensor] = None):
        sde = _checked_sde(self.sde, "likelihood()")
        unet, classes = R.resolve_model(model)
        if unet is None or unet._film:
            raise NotImplementedError("LikelihoodEstimate runs this package's Unet natively (its forward-mode JVP); other model "
                                      "callables have no host path")
        if unet.compute_dtype not in ("fp32", "float32"):
            raise ValueError("LikelihoodEstimate needs the Unet in fp32 (compute_dtype='fp32'): likelihoods are an fp32 metric")
        if data.dim() != 4:
            raise ValueError(f"data must be [B, C, H, W], got shape {tuple(data.shape)}")
        b, c, h, w = (int(v) for v in data.shape)
        _check_ode_unet(unet, data.shape)
        if noise is not None and tuple(noise.shape) != tuple(data.shape):
            raise ValueError(f"noise has shape {tuple(noise.shape)}; expected {tuple(data.shape)}")
        R.require_cuda(data.device)
        # the state is [x ; delta_logp]: delta_logp starts at 0
        state = _ode_solve(self, "likelihood", unet, classes, data.to(torch.float32), self.eps, float(sde.T), noise=noise,
                           hutchinson=L.HUTCH_RADEMACHER if self.hutchinson_type == "Rademacher" else L.HUTCH_GAUSSIAN,
                           rng=L.Rng(self.seed if self.seed is not None else R.draw_seed(), R.rank_stream_id()))
        n = b * c * h * w
        z, delta_logp = state[:n].view(b, c, h, w), state[n:]
        bpd = likelihood_bpd(sde, z, delta_logp)
        return bpd, z, self.last_stats["nfev"]


def likelihood_bpd(sde: SDE, z: torch.Tensor, delta_logp: torch.Tensor) -> torch.Tensor:
    """score_sde likelihood_fn's tail: bpd = -(prior_logp(z) + delta_logp) / ln 2 / D + (7 - inverse_scaler(-1)) for centred data."""
    bpd = -(sde.prior_logp(z) + delta_logp) / np.log(2)
    return bpd / np.prod(z.shape[1:]) + 7.0


# ------------------------------------------------------------------------------------------------------
# few-step DPM-Solver++ / SDE-DPM-Solver++ (Lu et al. 2022) for VP and VE score models; not in the reference
# ------------------------------------------------------------------------------------------------------


def score_sde_schedule(sde, t: float):
    """(alpha_t, sigma_t, lambda_t) of a VP or VE SDE at time t, in fp64.  VP: log alpha = -t^2 (b1 - b0) / 4 - t b0 / 2 and
    sigma = sqrt(1 - alpha^2) (ScoreFunction.scale's std); VE: alpha = 1, sigma = sigma_min (sigma_max / sigma_min)^t."""
    if isinstance(sde, VPSDE):
        la = -0.25 * t * t * (sde.beta_1 - sde.beta_0) - 0.5 * t * sde.beta_0
        sigma = math.sqrt(-math.expm1(2.0 * la))
        return math.exp(la), sigma, la - math.log(sigma)
    ls = math.log(sde.sigma_min) + t * math.log(sde.sigma_max / sde.sigma_min)
    return 1.0, math.exp(ls), -ls


def score_sde_inverse_lambda(sde, lam: float) -> float:
    """The time t whose lambda_t is `lam` (score_sde_schedule's inverse)."""
    if isinstance(sde, VPSDE):
        L_ = 0.5 * np.logaddexp(0.0, -2.0 * lam)          # -log alpha
        b0, db = sde.beta_0, sde.beta_1 - sde.beta_0
        return float(2.0 * L_ / (0.5 * b0 + math.sqrt(0.25 * b0 * b0 + db * L_)))
    return math.log(math.exp(-lam) / sde.sigma_min) / math.log(sde.sigma_max / sde.sigma_min)


def score_sde_grid(sde, steps: int, eps: float, skip_type: str) -> List[float]:
    """steps + 1 fp64 times from sde.T down to eps (both exact): uniform in t ("time_uniform") or in lambda ("logSNR")."""
    T = float(sde.T)
    if skip_type == "time_uniform":
        ts = np.linspace(T, eps, steps + 1).tolist()
    else:
        lams = np.linspace(score_sde_schedule(sde, T)[2], score_sde_schedule(sde, eps)[2], steps + 1)
        ts = [score_sde_inverse_lambda(sde, float(v)) for v in lams]
    ts[0], ts[-1] = T, float(eps)
    return ts


def sde_dpmpp_coefs(alpha, sigma, lam, orders):
    """SDE-DPM-Solver++ coefficients (c_x, c_0, c_1, g) of every step (data-prediction SDE form, 2M as the midpoint variant):
    x' = c_x x + c_0 m_i + c_1 m_{i-1} + g z, with h = lambda' - lambda, c_x = sigma'/sigma e^-h, k = alpha' (1 - e^-2h),
    order 1: c_0 = k; order 2: c_0 = k (1 + 1 / (2 r0)), c_1 = -k / (2 r0); g = sigma' sqrt(1 - e^-2h)."""
    rows = []
    for i, order in enumerate(orders):
        h = lam[i + 1] - lam[i]
        e2 = -math.expm1(-2.0 * h)
        k = alpha[i + 1] * e2
        cx, c0, c1 = sigma[i + 1] / sigma[i] * math.exp(-h), k, 0.0
        if order == 2:
            r0 = (lam[i] - lam[i - 1]) / h
            c0 = k * (1.0 + 1.0 / (2.0 * r0))
            c1 = -k / (2.0 * r0)
        rows.append((cx, c0, c1, sigma[i + 1] * math.sqrt(e2)))
    return rows


class DPMSolverSampler(torch.nn.Module):
    """Few-step sampler of a VP or VE score-SDE model: DPM-Solver++ multistep ("dpmsolver++", deterministic, orders 1-3) or
    SDE-DPM-Solver++ ("sde-dpmsolver++", orders 1-2) on a grid of `steps` + 1 times from sde.T to eps, uniform in logSNR or in t.
    One model evaluation per step (nfe = steps) and one update kernel (dmn_dpmpp_step / dmn_dpmpp_sde_step) with the earlier data
    predictions in a device ring; with this package's Unet the loop is one replayed CUDA graph (DMN_LOOP_DPMPP), and
    `guidance_scale` runs classifier-free guidance on a class-conditional Unet.  The data prediction is not clamped, like the
    PC and ODE samplers; the sampler returns the state at t = eps with no denoising step.

    `noise`: noise[0] is x_T (times sigma_max for VE); for "sde-dpmsolver++" noise[1 + s] is the z of step s.  Without it every
    draw is in-kernel Philox keyed (`seed` or a draw from torch's CPU generator, data-parallel rank); x_T is the draw the PC
    sampler makes for the same seed."""

    def __init__(self, steps: int = 20, order: int = 2, skip_type: str = "logSNR", algorithm_type: str = "dpmsolver++",
                 eps: float = None):
        super().__init__()
        if isinstance(steps, bool) or not isinstance(steps, (int, np.integer)) or steps < 1:
            raise ValueError(f"`steps` must be an integer >= 1, got {steps!r}")
        if algorithm_type not in ("dpmsolver++", "sde-dpmsolver++"):
            raise ValueError(f"`algorithm_type` must be 'dpmsolver++' or 'sde-dpmsolver++', got {algorithm_type!r}")
        max_order = 3 if algorithm_type == "dpmsolver++" else 2
        if isinstance(order, bool) or order not in range(1, max_order + 1):
            raise ValueError(f"`order` must be in 1..{max_order} for {algorithm_type}, got {order!r}")
        if skip_type not in ("logSNR", "time_uniform"):
            raise ValueError(f"`skip_type` must be 'logSNR' or 'time_uniform', got {skip_type!r}")
        if eps is not None and (isinstance(eps, bool) or not isinstance(eps, (int, float, np.floating, np.integer))
                                or not 0 < eps < 1):
            raise ValueError(f"`eps` must be a number in (0, 1), got {eps!r}")
        self.steps, self.order, self.skip_type, self.algorithm_type = int(steps), int(order), skip_type, algorithm_type
        self.eps = None if eps is None else float(eps)
        self.sde: Optional[SDE] = None
        self.seed: Optional[int] = None
        self.guidance_scale: Optional[float] = None
        self.trajectory_every = 0
        self.use_cuda_graph = True
        self._cache = {}

    def update_sde(self, sde: SDE):
        self.sde = sde
        self._cache = {}

    def timesteps(self) -> List[float]:
        """The fp64 grid: steps + 1 times from sde.T to eps."""
        sde = _checked_sde(self.sde)
        return score_sde_grid(sde, self.steps, sde.sampling_epsilon if self.eps is None else self.eps, self.skip_type)

    def step_orders(self) -> List[int]:
        """min(order, i + 1) at step i (warm-up); with fewer than 15 steps also at most steps - i, so the last step is first order."""
        k = self.steps
        return [min(self.order, i + 1, k - i) if k < 15 else min(self.order, i + 1) for i in range(k)]

    def rows(self):
        """(coef [steps][8], coef2 [steps][8] or None, labels [steps]) as CPU fp32: the kernel rows of dmn_dpmpp_step (mode 2:
        unclamped data prediction) / dmn_dpmpp_sde_step expanded in fp64 and rounded once, and the U-Net labels
        ScoreFunction.labels of the fp32 grid."""
        sde = _checked_sde(self.sde)
        ts = self.timesteps()
        alpha, sigma, lam = zip(*(score_sde_schedule(sde, t) for t in ts))
        orders = self.step_orders()
        vp = isinstance(sde, VPSDE)
        coef2 = None
        if self.algorithm_type == "dpmsolver++":
            coefs = multistep_coefs(alpha, sigma, lam, orders)
        else:
            sde_coefs = sde_dpmpp_coefs(alpha, sigma, lam, orders)
            coefs = [(cx, c0, c1, 0.0) for cx, c0, c1, _ in sde_coefs]
            coef2 = torch.zeros(self.steps, L.COEF_STRIDE, dtype=torch.float64)
            coef2[:, 0] = torch.tensor([r[3] for r in sde_coefs], dtype=torch.float64)
            coef2 = coef2.to(torch.float32)
        rows = []
        for i, c in enumerate(coefs):
            # m = k_x x - k_m out: VP (eps-like output, score = -out / sigma): x / alpha - sigma / alpha out; VE (the output is the
            # score): x + sigma^2 out
            kx, km = (1.0 / alpha[i], sigma[i] / alpha[i]) if vp else (1.0, -sigma[i] * sigma[i])
            rows.append(list(c) + [kx, km, float(i % 3), 2.0])
        labels = ScoreFunction(None, sde).labels(torch.tensor(ts[:-1], dtype=torch.float64).to(torch.float32))
        return torch.tensor(rows, dtype=torch.float64).to(torch.float32), coef2, labels.to(torch.float32)

    def forward(self, model, shape: List[int], device, return_nfe: bool = True, use_tqdm: bool = True, noise=None):
        sde = _checked_sde(self.sde)
        R.require_cuda(device)
        device = torch.device(device)
        if len(shape) != 4:
            raise ValueError(f"shape must be [B, C, H, W], got {list(shape)}")
        b, c, h, w = (int(v) for v in shape)
        if noise is not None:
            need = 1 + (self.steps if self.algorithm_type == "sde-dpmsolver++" else 0)
            if noise.dim() != 5 or tuple(noise.shape[1:]) != (b, c, h, w) or noise.shape[0] < need:
                raise ValueError(f"noise has shape {tuple(noise.shape)}; expected [n >= {need}, {b}, {c}, {h}, {w}]")
        key = str(device)
        hit = self._cache.get(key)
        if hit is None:
            coef, coef2, labels = self.rows()
            hit = (coef.to(device), None if coef2 is None else coef2.to(device), labels.to(device))
            self._cache[key] = hit
        coef, coef2, labels = hit
        unet, _ = R.resolve_model(model)
        if unet is not None:
            if c != unet.channels or h != w:
                raise ValueError(f"shape {list(shape)} does not fit the U-Net ({unet.channels} channels, square images)")
            if unet.out_dim != unet.channels:
                raise ValueError("the score-SDE data prediction needs a U-Net whose output has as many channels as its input")
        imgs = R.run_loop(model, kind=L.LOOP_DPMPP, shape=shape, device=device, times=labels, coef=coef, coef2=coef2, noise=noise,
                          seed=self.seed, traj_every=self.trajectory_every, use_graph=self.use_cuda_graph, init_scale=init_scale(sde),
                          guidance_scale=self.guidance_scale, model_arg=lambda s: labels[s].repeat(b))
        return (imgs, self.steps) if return_nfe else imgs

    def sample(self, model, shape: List[int], device=None, return_nfe: bool = False, noise=None):
        device = R.default_device(model, device)
        return self.forward(model=model, shape=shape, device=device, return_nfe=return_nfe, noise=noise)

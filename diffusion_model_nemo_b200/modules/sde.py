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
"""
import abc
import ctypes as C
import warnings
from typing import List, Optional

import numpy as np
import torch

from .. import _lib as L
from . import _runtime as R

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
        lmc = -0.25 * t ** 2 * (self.beta_1 - self.beta_0) - 0.5 * t * self.beta_0
        return torch.exp(lmc[:, None, None, None]) * x, torch.sqrt(1.0 - torch.exp(2.0 * lmc))

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
            lmc = -0.25 * t ** 2 * (self.sde.beta_1 - self.sde.beta_0) - 0.5 * t * self.sde.beta_0
            return -1.0 / torch.sqrt(1.0 - torch.exp(2.0 * lmc))
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
        std = sde.marginal_prob(None, t)[1] if isinstance(sde, VESDE) else torch.sqrt(
            1.0 - torch.exp(2.0 * (-0.25 * t ** 2 * (sde.beta_1 - sde.beta_0) - 0.5 * t * sde.beta_0)))
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
        if self.sde is None:
            raise ValueError("Must explicitly set `update_sde(sde)` for this module prior to calling forward()")
        R.require_cuda(device)
        sde = self.sde
        ts = self.timesteps()
        sf = ScoreFunction(model, sde, self.continuous)
        unet, classes = R.resolve_model(model)
        n_corr = self.n_steps if _NATIVE_CORRECTORS.get(self.corrector) else 0
        init_scale = float(sde.sigma_max) if isinstance(sde, VESDE) else 1.0
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
                                    use_graph=self.use_cuda_graph, init_scale=init_scale)
            final = res.aux if self.denoise else res.final
            imgs = R.to_image_list(final, res.traj)
        else:
            # plugin path: user-registered predictor/corrector classes or a foreign model -> per-step update_fn calls
            pred = (get_predictor(self.predictor) if self.predictor else NonePredictor)(sde, sf, self.probability_flow)
            corr = (get_corrector(self.corrector) if self.corrector else NoneCorrector)(sde, sf, self.snr, self.n_steps)
            k = 0
            if noise is not None:
                x = noise[0].to(device, torch.float32) * init_scale
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
        if method != "RK45":
            raise NotImplementedError(f"method={method!r}: only the RK45 solver is built")
        for name, v in (("rtol", rtol), ("atol", atol)):
            if isinstance(v, bool) or not isinstance(v, (int, float, np.floating, np.integer)):
                raise ValueError(f"{name} must be a scalar number (per-component tolerances are not supported), got {type(v).__name__}")
            if not np.isfinite(v) or v < 0 or (name == "rtol" and v == 0):
                raise ValueError(f"{name} must be finite and {'> 0' if name == 'rtol' else '>= 0'}, got {v}")
        if isinstance(max_nfe, bool) or not isinstance(max_nfe, (int, np.integer)) or max_nfe < 2:
            raise ValueError(f"max_nfe must be an integer >= 2, got {max_nfe!r}")
        self.denoise, self.rtol, self.atol, self.method, self.eps = denoise, float(rtol), float(atol), method, eps
        self.max_nfe = int(max_nfe)
        self.sde: Optional[SDE] = None
        self.use_cuda_graph = True
        self.last_stats: Optional[dict] = None

    def update_sde(self, sde: SDE):
        self.sde = sde

    def forward(self, model, shape: List[int], device, return_nfe: bool = True, use_tqdm: bool = True, noise=None):
        if self.sde is None:
            raise ValueError("Must explicitly set `update_sde(sde)` for this module prior to calling forward()")
        sde = self.sde
        if not isinstance(sde, (VPSDE, VESDE)):
            raise NotImplementedError(f"SDE class {sde.__class__.__name__} not yet supported.")
        R.require_cuda(device)
        device = torch.device(device)
        unet, classes = R.resolve_model(model)
        if unet is None:
            raise NotImplementedError("ProbabilityFlowSampler runs this package's Unet natively; other model callables have no "
                                      "host solver path")
        b, c, h, w = (int(v) for v in shape)
        if c != unet.channels or h != w:
            raise ValueError(f"shape {list(shape)} does not fit the U-Net ({unet.channels} channels, square images)")
        if unet.out_dim != unet.channels:
            raise ValueError("the probability-flow drift needs a U-Net whose output has as many channels as its input")
        eps = sde.sampling_epsilon if self.eps is None else float(self.eps)
        init_scale = float(sde.sigma_max) if isinstance(sde, VESDE) else 1.0
        x = noise[0] * init_scale if noise is not None else sde.prior_sampling(shape)
        if tuple(x.shape) != (b, c, h, w):
            raise ValueError(f"x_T has shape {tuple(x.shape)}; expected {(b, c, h, w)}")
        lib = L.lib()
        plan = unet.plan(h, b, device, time_rows=6)
        with torch.cuda.device(device):
            st = L.stream_ptr(device)
            # buffers live with the plan so the addresses baked into the cached graph stay valid
            bufs = plan.__dict__.setdefault("_ode_bufs", {})
            if b not in bufs:
                nbytes = int(lib.dmn_ode_work_bytes(plan.h, b))
                bufs[b] = {"state": torch.empty((b, c, h, w), dtype=torch.float32, device=device),
                           "work": torch.empty(nbytes + 256, dtype=torch.uint8, device=device),
                           "result": torch.zeros(3, dtype=torch.float64, device=device)}
            buf = bufs[b]
            state, work, result = buf["state"], buf["work"], buf["result"]
            state.copy_(x.to(device, torch.float32))
            if classes is not None:
                classes = R.stable_copy(buf, "classes", classes.to(device, torch.int64).reshape(-1))
            wp = (work.data_ptr() + 255) // 256 * 256
            d = L.OdeDesc()
            if isinstance(sde, VPSDE):
                d.sde_kind, d.N, d.beta_0, d.beta_1 = L.SDE_VP, int(sde.N), float(sde.beta_0), float(sde.beta_1)
            else:
                d.sde_kind, d.N, d.sigma_min, d.sigma_max = L.SDE_VE, int(sde.N), float(sde.sigma_min), float(sde.sigma_max)
            d.t0, d.t1, d.rtol, d.atol = float(sde.T), eps, self.rtol, self.atol
            d.max_nfe, d.batch, d.use_graph = self.max_nfe, b, int(bool(self.use_cuda_graph))
            d.classes_dev = classes.data_ptr() if classes is not None else None
            d.state_dev, d.state_elems = state.data_ptr(), state.numel()
            d.work_dev, d.work_bytes = wp, work.numel() - (wp - work.data_ptr())
            d.result_dev = result.data_ptr()
            L.check(lib.dmn_ode_sample(plan.h, C.byref(d), st), "dmn_ode_sample")
            plan.time_rows_key = None            # the solve rewrote rows 0..5 of the time table
            raw = result.cpu().numpy().tobytes()
            x = state.clone()
        res = L.OdeResult.from_buffer_copy(raw)
        self.last_stats = {"status": int(res.status), "nfev": int(res.nfev), "n_accepted": int(res.n_accepted),
                           "n_rejected": int(res.n_rejected), "t_final": float(res.t_final)}
        if res.status == L.ODE_LIMIT:
            raise RuntimeError(f"probability-flow ODE: stopped at {res.nfev} model evaluations (max_nfe={self.max_nfe}) at "
                               f"t={res.t_final:.6g}, before reaching eps={eps:g}")
        if res.status == L.ODE_TOO_SMALL_STEP:
            warnings.warn(f"probability-flow ODE: required step size became too small at t={res.t_final:.6g} (scipy status -1); "
                          "returning the last accepted state, as solve_ivp does")
        if self.denoise:      # one reverse-diffusion predictor step at eps, probability_flow=False, keeping x_mean
            vec_eps = torch.ones(b, device=device) * eps
            pred = ReverseDiffusionPredictor(sde, ScoreFunction(model, sde), probability_flow=False)
            _, x = pred.update_fn(x, vec_eps)
        imgs = R.to_image_list(x.float().contiguous(), None)
        return (imgs, int(res.nfev)) if return_nfe else imgs

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
        if method != "RK45":
            raise NotImplementedError(f"method={method!r}: only the RK45 solver is built")
        for name, v in (("rtol", rtol), ("atol", atol), ("eps", eps)):
            if isinstance(v, bool) or not isinstance(v, (int, float, np.floating, np.integer)):
                raise ValueError(f"{name} must be a scalar number, got {type(v).__name__}")
            if not np.isfinite(v) or v < 0 or (name != "atol" and v == 0):
                raise ValueError(f"{name} must be finite and {'>= 0' if name == 'atol' else '> 0'}, got {v}")
        if isinstance(max_nfe, bool) or not isinstance(max_nfe, (int, np.integer)) or max_nfe < 2:
            raise ValueError(f"max_nfe must be an integer >= 2, got {max_nfe!r}")
        self.hutchinson_type, self.rtol, self.atol, self.method = hutchinson_type, float(rtol), float(atol), method
        self.eps, self.max_nfe = float(eps), int(max_nfe)
        self.sde: Optional[SDE] = None
        self.seed: Optional[int] = None
        self.use_cuda_graph = True
        self.last_stats: Optional[dict] = None

    def update_sde(self, sde: SDE):
        self.sde = sde

    def likelihood(self, model, data: torch.Tensor, noise: Optional[torch.Tensor] = None):
        if self.sde is None:
            raise ValueError("Must explicitly set `update_sde(sde)` for this module prior to calling likelihood()")
        sde = self.sde
        if not isinstance(sde, (VPSDE, VESDE)):
            raise NotImplementedError(f"SDE class {sde.__class__.__name__} not yet supported.")
        unet, classes = R.resolve_model(model)
        if unet is None or unet._film:
            raise NotImplementedError("LikelihoodEstimate runs this package's Unet natively (its forward-mode JVP); other model "
                                      "callables have no host path")
        if unet.compute_dtype not in ("fp32", "float32"):
            raise ValueError("LikelihoodEstimate needs the Unet in fp32 (compute_dtype='fp32'): likelihoods are an fp32 metric")
        if data.dim() != 4:
            raise ValueError(f"data must be [B, C, H, W], got shape {tuple(data.shape)}")
        b, c, h, w = (int(v) for v in data.shape)
        if c != unet.channels or h != w:
            raise ValueError(f"data shape {tuple(data.shape)} does not fit the U-Net ({unet.channels} channels, square images)")
        if unet.out_dim != unet.channels:
            raise ValueError("the probability-flow drift needs a U-Net whose output has as many channels as its input")
        if noise is not None and tuple(noise.shape) != tuple(data.shape):
            raise ValueError(f"noise has shape {tuple(noise.shape)}; expected {tuple(data.shape)}")
        device = data.device
        R.require_cuda(device)
        lib = L.lib()
        plan = unet.plan(h, b, device, time_rows=6)
        n = b * c * h * w
        with torch.cuda.device(device):
            st = L.stream_ptr(device)
            # buffers live with the plan so the addresses baked into the cached graph stay valid
            bufs = plan.__dict__.setdefault("_lik_bufs", {})
            if b not in bufs:
                nbytes = int(lib.dmn_ode_likelihood_work_bytes(plan.h, b))
                bufs[b] = {"state": torch.empty(n + b, dtype=torch.float32, device=device),
                           "work": torch.empty(nbytes + 256, dtype=torch.uint8, device=device),
                           "result": torch.zeros(3, dtype=torch.float64, device=device)}
            buf = bufs[b]
            state, work, result = buf["state"], buf["work"], buf["result"]
            state[:n].copy_(data.reshape(-1).to(torch.float32))
            state[n:].zero_()
            if classes is not None:
                classes = R.stable_copy(buf, "classes", classes.to(device, torch.int64).reshape(-1))
            if noise is not None:
                noise = R.stable_copy(buf, "noise", noise.to(device, torch.float32).reshape(-1))
            wp = (work.data_ptr() + 255) // 256 * 256
            d = L.OdeLikelihoodDesc()
            if isinstance(sde, VPSDE):
                d.sde_kind, d.N, d.beta_0, d.beta_1 = L.SDE_VP, int(sde.N), float(sde.beta_0), float(sde.beta_1)
            else:
                d.sde_kind, d.N, d.sigma_min, d.sigma_max = L.SDE_VE, int(sde.N), float(sde.sigma_min), float(sde.sigma_max)
            d.t0, d.t1, d.rtol, d.atol = self.eps, float(sde.T), self.rtol, self.atol
            d.max_nfe, d.batch, d.use_graph = self.max_nfe, b, int(bool(self.use_cuda_graph))
            d.hutchinson = L.HUTCH_RADEMACHER if self.hutchinson_type == "Rademacher" else L.HUTCH_GAUSSIAN
            d.rng = L.Rng(self.seed if self.seed is not None else R.draw_seed(), R.rank_stream_id())
            d.noise_dev = noise.data_ptr() if noise is not None else None
            d.classes_dev = classes.data_ptr() if classes is not None else None
            d.state_dev, d.state_elems = state.data_ptr(), state.numel()
            d.work_dev, d.work_bytes = wp, work.numel() - (wp - work.data_ptr())
            d.result_dev = result.data_ptr()
            L.check(lib.dmn_ode_likelihood(plan.h, C.byref(d), st), "dmn_ode_likelihood")
            plan.time_rows_key = None            # the solve rewrote rows 0..5 of the time table
            raw = result.cpu().numpy().tobytes()
            z = state[:n].reshape(b, c, h, w).clone()
            delta_logp = state[n:].clone()
        res = L.OdeResult.from_buffer_copy(raw)
        self.last_stats = {"status": int(res.status), "nfev": int(res.nfev), "n_accepted": int(res.n_accepted),
                           "n_rejected": int(res.n_rejected), "t_final": float(res.t_final)}
        if res.status == L.ODE_LIMIT:
            raise RuntimeError(f"likelihood ODE: stopped at {res.nfev} model evaluations (max_nfe={self.max_nfe}) at "
                               f"t={res.t_final:.6g}, before reaching T={float(sde.T):g}")
        if res.status == L.ODE_TOO_SMALL_STEP:
            warnings.warn(f"likelihood ODE: required step size became too small at t={res.t_final:.6g} (scipy status -1); "
                          "returning the last accepted state, as solve_ivp does")
        bpd = likelihood_bpd(sde, z, delta_logp)
        return bpd, z, int(res.nfev)


def likelihood_bpd(sde: SDE, z: torch.Tensor, delta_logp: torch.Tensor) -> torch.Tensor:
    """score_sde likelihood_fn's tail: bpd = -(prior_logp(z) + delta_logp) / ln 2 / D + (7 - inverse_scaler(-1)) for centred data."""
    bpd = -(sde.prior_logp(z) + delta_logp) / np.log(2)
    return bpd / np.prod(z.shape[1:]) + 7.0

"""CPU oracle of the probability-flow pieces of score-SDE sampling.  TEST INFRASTRUCTURE ONLY.

Restates, with the fp32 torch ops of oracle/ref_port.py (SDESpec, score_fn), what the reference runs when probability_flow=True:
  * sde_lib.py reverse() (score_sde): drift = f(x,t) - g(t)^2 * score(x,t) * 0.5, diffusion 0, and the matching
    discretize(): rev_f = f - G^2 * score * 0.5, rev_G = 0;
  * modules/sde_samplers/probability_flow_sampler.py:46-100 (score_sde get_ode_sampler): scipy.integrate.solve_ivp over
    that drift from sde.T to eps with method='RK45', then the optional reverse-diffusion denoise step.
These are pinned to scipy's RK45 (scipy/integrate/_ivp/rk.py, common.py) and to the reverse-SDE algebra above, not to an
executed run of the reference, which is not available where the golden fixtures are regenerated.  The pinned oracle module
(oracle/ref_port.py) is left as it is; this file only composes its functions.
"""
import numpy as np
import torch
from scipy import integrate

from oracle import ref_port as O


def ode_drift(model, sde: O.SDESpec, x, t):
    """Probability-flow drift f(x,t) - 0.5 g(t)^2 score(x,t) in the reference's op order (RSDE.sde with probability_flow=True)."""
    drift, diffusion = sde.sde(x, t)
    return drift - diffusion[:, None, None, None] ** 2 * O.score_fn(model, sde, x, t) * 0.5


def rd_predictor_step(model, sde, x, t, z, probability_flow=False):
    """ReverseDiffusionPredictor.update_fn + RSDE.discretize (sde_lib.py:100-105) with the probability_flow switch."""
    f, G = sde.discretize(x, t)
    rev_f = f - G[:, None, None, None] ** 2 * O.score_fn(model, sde, x, t) * (0.5 if probability_flow else 1.0)
    rev_G = torch.zeros_like(G) if probability_flow else G
    x_mean = x - rev_f
    return x_mean + rev_G[:, None, None, None] * z, x_mean


def em_predictor_step(model, sde, x, t, z, probability_flow=False):
    """EulerMaruyamaPredictor.update_fn + RSDE.sde (sde_lib.py:91-98) with the probability_flow switch."""
    dt = -1.0 / sde.N
    drift, diffusion = sde.sde(x, t)
    drift = drift - diffusion[:, None, None, None] ** 2 * O.score_fn(model, sde, x, t) * (0.5 if probability_flow else 1.0)
    diffusion = torch.zeros_like(diffusion) if probability_flow else diffusion
    x_mean = x + drift * dt
    return x_mean + diffusion[:, None, None, None] * np.sqrt(-dt) * z, x_mean


def sample_pc(model, shape, sde: O.SDESpec, draw, predictor="reverse_diffusion", corrector="langevin", snr=0.16, n_steps=1,
              denoise=True, eps=None, probability_flow=False):
    """oracle.ref_port.sample_pc with the predictor's probability_flow switch (the predictor still draws its z)."""
    eps = sde.sampling_epsilon if eps is None else eps
    x = sde.prior(shape, draw)
    timesteps = torch.linspace(1, eps, sde.N)
    last = None
    for i in range(sde.N):
        vec_t = torch.ones(shape[0]) * timesteps[i]
        x_mean = x
        if corrector in ("langevin", "ald"):
            for _ in range(n_steps):
                z = draw(shape)
                x, x_mean = (O.langevin_step if corrector == "langevin" else O.ald_step)(model, sde, x, vec_t, z, snr)
        if predictor in ("reverse_diffusion", "euler_maruyama"):
            z = draw(shape)
            step = rd_predictor_step if predictor == "reverse_diffusion" else em_predictor_step
            x, x_mean = step(model, sde, x, vec_t, z, probability_flow)
        last = x_mean if denoise else x
    return last, x


def sample_probability_flow(model, shape, sde: O.SDESpec, draw, rtol=1e-5, atol=1e-5, eps=None, denoise=False):
    """ProbabilityFlowSampler.forward: x_T = prior, solve_ivp(ode_func, (T, eps), x_T (float64), rtol, atol, 'RK45') where
    ode_func casts y to fp32, uses vec_t = ones(B) * t (fp32) and returns the fp32 drift; then the optional denoise step
    (reverse diffusion at eps, probability_flow=False, keeping x_mean).  Returns (state in [-1,1] space, nfev, solution)."""
    eps = sde.sampling_epsilon if eps is None else eps
    x = sde.prior(shape, draw)

    def ode_func(t, y):
        xt = torch.from_numpy(y.reshape(shape)).type(torch.float32)
        vec_t = torch.ones(shape[0]) * t
        return ode_drift(model, sde, xt, vec_t).numpy().reshape((-1,))

    sol = integrate.solve_ivp(ode_func, (1, eps), x.numpy().reshape((-1,)), rtol=rtol, atol=atol, method="RK45")
    x = torch.tensor(sol.y[:, -1]).reshape(shape).type(torch.float32)
    if denoise:
        vec_eps = torch.ones(shape[0]) * eps
        _, x = rd_predictor_step(model, sde, x, vec_eps, torch.zeros_like(x), probability_flow=False)
    return x, sol.nfev, sol


def zero_model(x, labels):
    """The score model of the exact controller check: a U-Net whose final 1x1 convolution is zero returns exactly 0."""
    return torch.zeros_like(x)

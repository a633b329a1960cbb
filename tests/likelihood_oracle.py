"""CPU oracle of the U-Net JVP and of the probability-flow ODE likelihood.  TEST INFRASTRUCTURE ONLY.

  * unet_jvp: torch.func.jvp of oracle/ref_port.py's unet_forward in float64.
  * likelihood: score_sde's likelihood_fn (get_likelihood_fn): the augmented state [x ; delta_logp] integrated with
    scipy.integrate.solve_ivp from eps to sde.T, the divergence by the Hutchinson estimator of score_sde's div_fn (autograd of
    sum(drift * eps), fp32 as the reference runs it), then bpd = -(prior_logp(z) + delta_logp) / ln 2 / D + 7.
The pinned oracle module (oracle/ref_port.py) and tests/ode_oracle.py are used as they are; this file only composes them.
"""
import numpy as np
import torch
from scipy import integrate

from oracle import ref_port as O
from ode_oracle import ode_drift


def unet_jvp(sd, cfg, x, t, v, classes=None):
    """(u(x, t), du/dx . v) of ref_port.unet_forward in float64."""
    sd64 = {k: (w.double() if w.is_floating_point() else w) for k, w in sd.items()}
    return torch.func.jvp(lambda xx: O.unet_forward(sd64, cfg, xx, t.double(), classes), (x.double(),), (v.double(),))


def prior_logp(sde: O.SDESpec, z):
    """VPSDE.prior_logp / VESDE.prior_logp (modules/sde.py)."""
    n = np.prod(z.shape[1:])
    if sde.kind == "vp":
        return -n / 2.0 * np.log(2 * np.pi) - torch.sum(z ** 2, dim=(1, 2, 3)) / 2.0
    return -n / 2.0 * np.log(2 * np.pi * sde.sigma_max ** 2) - torch.sum(z ** 2, dim=(1, 2, 3)) / (2 * sde.sigma_max ** 2)


def likelihood(model, sde: O.SDESpec, data, epsilon, rtol=1e-5, atol=1e-5, eps=1e-5, div_fn=None):
    """score_sde likelihood_fn with the Hutchinson noise `epsilon` given.  Returns (bpd, z, delta_logp, solution).
    div_fn(x, t) replaces the autograd divergence when given (see linear_div)."""
    shape = data.shape
    b = shape[0]

    def autograd_div(x, t):
        with torch.enable_grad():
            x = x.detach().requires_grad_(True)
            fn_eps = torch.sum(ode_drift(model, sde, x, t) * epsilon)
            grad = torch.autograd.grad(fn_eps, x)[0]
        return torch.sum(grad * epsilon, dim=(1, 2, 3))

    def ode_func(t, y):
        x = torch.from_numpy(y[:-b].reshape(shape)).type(torch.float32)
        vec_t = torch.ones(b) * t
        with torch.no_grad():
            drift = ode_drift(model, sde, x, vec_t).numpy().reshape((-1,))
        logp_grad = (div_fn or autograd_div)(x, vec_t).detach().numpy().reshape((-1,))
        return np.concatenate([drift, logp_grad], axis=0)

    init = np.concatenate([data.numpy().reshape((-1,)), np.zeros((b,))], axis=0)
    sol = integrate.solve_ivp(ode_func, (eps, 1.0), init, rtol=rtol, atol=atol, method="RK45")
    zp = sol.y[:, -1]
    z = torch.from_numpy(zp[:-b].reshape(shape)).type(torch.float32)
    delta_logp = torch.from_numpy(zp[-b:]).type(torch.float32)
    bpd = -(prior_logp(sde, z) + delta_logp) / np.log(2)
    bpd = bpd / np.prod(shape[1:]) + 7.0
    return bpd, z, delta_logp, sol


def linear_div(model, sde: O.SDESpec, epsilon):
    """Divergence of a drift that is linear in x (the model output does not depend on x): eps . drift(eps), with the fp32 drift
    summed in float64 and rounded once -- the sum the device computes.  The exact controller check uses it so that both solvers
    integrate the same fp32 function: at the first step the log-density rows dominate select_initial_step, whose d2 is then the
    difference of two nearly equal fp32 divergences, so the rounding of a float32 sum would change the step sizes."""
    def div(x, t):
        return (ode_drift(model, sde, epsilon, t).double() * epsilon.double()).sum(dim=(1, 2, 3)).float()
    return div


def rademacher(shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 2, shape, generator=g).float() * 2 - 1.0


def gaussian(shape, seed):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed))

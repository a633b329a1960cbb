"""float64 DPM-Solver++ multistep oracle (Lu et al. 2022, Algorithm 2 and its third-order extension), written in the D1 / D2
difference form -- independent of the coefficient rows DPMSolverDiffusion builds.

Time grid: the DDIM grid (oracle.ref_port.ddim_pairs), last target -1 with alpha_bar = 1.  Per time: alpha = sqrt(abar),
sigma = sqrt(1 - abar), lambda = (log abar - log1p(-abar)) / 2, from the package's fp32 alphas_cumprod.  m_i is the clamped data
prediction (pred_noise: fp32 tables sqrt_recip_ac / sqrt_recipm1_ac as the kernels use them; the first C channels of a 2C output).

Also the Gaussian-data model with an exact answer: for data ~ N(0, s^2 I) the optimal eps is sigma / (alpha^2 s^2 + sigma^2) x, the
probability-flow solution from the first grid time t0 is x(t) = x_T sqrt(alpha_t^2 s^2 + sigma_t^2) / sqrt(alpha_t0^2 s^2 + sigma_t0^2)
and the exact sample is the data prediction at x(0).
"""
import math

import torch

from oracle import ref_port as O


def step_orders(k, order):
    return [1 if i == k - 1 else (min(order, 2, i + 1) if (k < 15 and i == k - 2) else min(order, i + 1)) for i in range(k)]


class Schedule:
    def __init__(self, timesteps, schedule="linear"):
        tb = O.ddpm_tables(timesteps, schedule)
        self.T = timesteps
        self.ac = tb["alphas_cumprod"].double()
        self.k_x = tb["sqrt_recip_alphas_cumprod"].double()
        self.k_m = tb["sqrt_recipm1_alphas_cumprod"].double()

    def abar(self, t):
        return 1.0 if t < 0 else float(self.ac[t])

    def alpha(self, t):
        return math.sqrt(self.abar(t))

    def sigma(self, t):
        return math.sqrt(1.0 - self.abar(t))

    def lam(self, t):
        a = self.abar(t)
        return 0.5 * (math.log(a) - math.log1p(-a))


def data_pred(sch, x, model_out, t, objective="pred_noise"):
    c = x.shape[1]
    mo = model_out[:, :c].double()
    m = mo if objective == "pred_x0" else sch.k_x[t] * x - sch.k_m[t] * mo
    return m.clamp(-1.0, 1.0)


def update(sch, x, ms, ts, t_next, order):
    """One DPM-Solver++ step from ts[0] to t_next with ms = [m_i, m_{i-1}, m_{i-2}] at ts = [t_i, t_{i-1}, t_{i-2}]."""
    t = ts[0]
    if t_next < 0:
        return ms[0]
    lt, ln = sch.lam(t), sch.lam(t_next)
    h = ln - lt
    a_n = sch.alpha(t_next)
    em = math.expm1(-h)
    base = (sch.sigma(t_next) / sch.sigma(t)) * x - a_n * em * ms[0]
    if order == 1:
        return base
    r0 = (lt - sch.lam(ts[1])) / h
    d10 = (ms[0] - ms[1]) / r0
    if order == 2:
        return base - 0.5 * a_n * em * d10
    r1 = (sch.lam(ts[1]) - sch.lam(ts[2])) / h
    d11 = (ms[1] - ms[2]) / r1
    d1 = d10 + r0 / (r0 + r1) * (d10 - d11)
    d2 = (d10 - d11) / (r0 + r1)
    return base + a_n * (em / h + 1.0) * d1 - a_n * ((em + h) / h ** 2 - 0.5) * d2


def solve(model, x_T, sch, steps, order, objective="pred_noise"):
    """model(x, t_long[B]) -> model output (any float dtype; evaluated on x cast to the model's dtype by the caller's callable).
    Returns (final state, [state before each step], [m_i per step])."""
    pairs = O.ddim_pairs(sch.T, steps)
    orders = step_orders(len(pairs), order)
    x = x_T.double()
    states, ms_all, ms, ts = [], [], [], []
    for i, (t, tn) in enumerate(pairs):
        states.append(x)
        out = model(x, torch.full((x.shape[0],), t, dtype=torch.long))
        m = data_pred(sch, x, out, t, objective)
        ms_all.append(m)
        ms.insert(0, m)
        ts.insert(0, t)
        del ms[3:], ts[3:]
        x = update(sch, x, ms, ts, tn, orders[i])
    return x, states, ms_all


def ref_unet_model(sd, cfg, classes=None):
    """The oracle.ref_port U-Net (fp32 weights) as a model callable of the fp64 solver."""
    return lambda x, t: O.unet_forward(sd, cfg, x.float(), t.float(), classes).double()


# ---- Gaussian data ~ N(0, s2 I) ---------------------------------------------------------------------------------------------------
def gaussian_eps_coef(sch, s2, t):
    a2 = sch.abar(t)
    return math.sqrt(1.0 - a2) / (a2 * s2 + 1.0 - a2)


def gaussian_model(sch, s2):
    def model(x, t):
        return gaussian_eps_coef(sch, s2, int(t[0])) * x
    return model


def gaussian_exact(sch, s2, x_T, t0):
    """The data prediction at the exact probability-flow state x(0), starting from x_T at grid time t0."""
    def norm(t):
        return math.sqrt(sch.abar(t) * s2 + 1.0 - sch.abar(t))
    x0 = x_T.double() * norm(0) / norm(t0)
    return sch.alpha(0) * s2 / (sch.abar(0) * s2 + 1.0 - sch.abar(0)) * x0

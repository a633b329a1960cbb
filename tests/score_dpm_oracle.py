"""float64 references for DPMSolverSampler (DPM-Solver++ and SDE-DPM-Solver++ on VP / VE score models), written in the D1 / D2
difference form as tests/dpm_oracle.py is -- independent of the coefficient rows the package builds.

Schedule of oracle.ref_port.SDESpec: VP alpha_t = exp(-t^2 (b1 - b0) / 4 - t b0 / 2), sigma_t = sqrt(1 - alpha_t^2); VE alpha_t = 1,
sigma_t = sigma_min (sigma_max / sigma_min)^t; lambda_t = log(alpha_t / sigma_t).  The data prediction is not clamped:
VP (eps-like output) m = (x - sigma out) / alpha; VE (the output is the score) m = x + sigma^2 out.

The analytic Gaussian problem, data ~ N(mu, s^2 I): the optimal model outputs, the exact probability-flow map from x_T and the law
of the SDE sampler's output, which is Gaussian because every step is affine in (x, m_prev, z).
"""
import math

import numpy as np
import torch


def schedule(spec, t):
    """(alpha, sigma, lambda) at time t, fp64."""
    t = float(t)
    if spec.kind == "vp":
        a = math.exp(-0.25 * t * t * (spec.beta_1 - spec.beta_0) - 0.5 * t * spec.beta_0)
        s = math.sqrt(1.0 - a * a)
    else:
        a, s = 1.0, spec.sigma_min * (spec.sigma_max / spec.sigma_min) ** t
    return a, s, math.log(a / s)


def labels(spec, t):
    """The U-Net label of time t (score_function_loss.py: VP t (N - 1), VE sigma_t) on an fp32 time tensor."""
    return t * (spec.N - 1) if spec.kind == "vp" else spec.marginal_std(t)


def data_pred(spec, x, out, t):
    a, s, _ = schedule(spec, t)
    return (x - s * out) / a if spec.kind == "vp" else x + s * s * out


def step_orders(steps, order):
    return [min(order, i + 1, steps - i) if steps < 15 else min(order, i + 1) for i in range(steps)]


def update(spec, x, ms, ts, t_next, order):
    """One DPM-Solver++ step from ts[0] to t_next with ms = [m_i, m_{i-1}, m_{i-2}] at ts = [t_i, t_{i-1}, t_{i-2}]."""
    _, s_t, lt = schedule(spec, ts[0])
    a_n, s_n, ln = schedule(spec, t_next)
    h = ln - lt
    em = math.expm1(-h)
    base = (s_n / s_t) * x - a_n * em * ms[0]
    if order == 1:
        return base
    r0 = (lt - schedule(spec, ts[1])[2]) / h
    d10 = (ms[0] - ms[1]) / r0
    if order == 2:
        return base - 0.5 * a_n * em * d10
    r1 = (schedule(spec, ts[1])[2] - schedule(spec, ts[2])[2]) / h
    d11 = (ms[1] - ms[2]) / r1
    d1 = d10 + r0 / (r0 + r1) * (d10 - d11)
    d2 = (d10 - d11) / (r0 + r1)
    return base + a_n * (em / h + 1.0) * d1 - a_n * ((em + h) / h ** 2 - 0.5) * d2


def sde_update(spec, x, ms, ts, t_next, order, z):
    """One SDE-DPM-Solver++ step (data-prediction SDE form; order 2 is the midpoint 2M variant)."""
    _, s_t, lt = schedule(spec, ts[0])
    a_n, s_n, ln = schedule(spec, t_next)
    h = ln - lt
    k = a_n * -math.expm1(-2.0 * h)
    out = (s_n / s_t) * math.exp(-h) * x + k * ms[0]
    if order == 2:
        r0 = (lt - schedule(spec, ts[1])[2]) / h
        out = out + 0.5 * k * (ms[0] - ms[1]) / r0
    return out + s_n * math.sqrt(-math.expm1(-2.0 * h)) * z


def solve(model, x_T, spec, grid, order, zs=None):
    """model(x, labels_fp32[B]) -> output.  grid: steps + 1 fp64 times; the labels are those of the fp32-rounded grid, as the
    sampler feeds them.  zs: the per-step N(0,1) draws of the SDE form (None = deterministic DPM-Solver++).
    Returns (final state, [state before each step], [m_i per step])."""
    steps = len(grid) - 1
    orders = step_orders(steps, order)
    lab = labels(spec, torch.tensor(grid[:-1], dtype=torch.float64).to(torch.float32))
    x = x_T.double()
    states, ms_all, ms, ts = [], [], [], []
    for i in range(steps):
        states.append(x)
        out = model(x, lab[i].repeat(x.shape[0]))
        m = data_pred(spec, x, out.double(), grid[i])
        ms_all.append(m)
        ms.insert(0, m)
        ts.insert(0, grid[i])
        del ms[3:], ts[3:]
        if zs is None:
            x = update(spec, x, ms, ts, grid[i + 1], orders[i])
        else:
            x = sde_update(spec, x, ms, ts, grid[i + 1], orders[i], zs[i].double())
    return x, states, ms_all


# ---- Gaussian data ~ N(mu, s^2 I) -------------------------------------------------------------------------------------------------
def gaussian_out(spec, mu, s, x, t):
    """The optimal model output at time t: VP sigma (x - alpha mu) / (alpha^2 s^2 + sigma^2); VE -(x - mu) / (s^2 + sigma^2)."""
    a, sg, _ = schedule(spec, t)
    if spec.kind == "vp":
        return sg * (x - a * mu) / (a * a * s * s + sg * sg)
    return -(x - mu) / (s * s + sg * sg)


def gaussian_model(spec, mu, s, grid):
    """The optimal model as a callable of the solvers: the label of grid step i selects time grid[i] exactly."""
    lab = labels(spec, torch.tensor(grid[:-1], dtype=torch.float64).to(torch.float32)).tolist()

    def model(x, lab_b):
        return gaussian_out(spec, mu, s, x, grid[lab.index(float(lab_b[0]))])
    return model


def _r(spec, s, t):
    a, sg, _ = schedule(spec, t)
    return math.sqrt(a * a * s * s + sg * sg)


def gaussian_exact(spec, mu, s, x_T, t_T, t):
    """The exact probability-flow map from x_T at t_T to time t: alpha_t mu + r_t / r_T (x_T - alpha_T mu)."""
    return schedule(spec, t)[0] * mu + _r(spec, s, t) / _r(spec, s, t_T) * (x_T - schedule(spec, t_T)[0] * mu)


def gaussian_conditional(spec, mu, s, x_T, t_T, t):
    """Mean and std of x_t given x_T under the forward process, the law the reverse SDE from x_T reaches at t."""
    a_t, a_T = schedule(spec, t)[0], schedule(spec, t_T)[0]
    r_t, r_T = _r(spec, s, t), _r(spec, s, t_T)
    cov = a_T / a_t * r_t * r_t          # Cov(x_t, x_T): x_T = (a_T / a_t) x_t + independent noise
    return a_t * mu + cov / (r_T * r_T) * (x_T - a_T * mu), math.sqrt(r_t * r_t - cov * cov / (r_T * r_T))


def sde_output_moments(spec, mu, s, x_T, grid, order):
    """Exact mean and std of SDE-DPM-Solver++'s final state on the Gaussian problem from a fixed x_T: every step is affine in
    (x, m_prev) plus g z, so the mean vector and the 2 x 2 covariance of (x, m_prev) propagate exactly."""
    orders = step_orders(len(grid) - 1, order)
    mean, cov = np.array([x_T, 0.0]), np.zeros((2, 2))
    for i in range(len(grid) - 1):
        a, sg, lt = schedule(spec, grid[i])
        a_n, s_n, ln = schedule(spec, grid[i + 1])
        # m_i = p x + q: the data prediction of the optimal output
        if spec.kind == "vp":
            d = a * a * s * s + sg * sg
            p, q = (1.0 - sg * sg / d) / a, sg * sg * a * mu / d / a
        else:
            d = s * s + sg * sg
            p, q = 1.0 - sg * sg / d, sg * sg * mu / d
        h = ln - lt
        k = a_n * -math.expm1(-2.0 * h)
        cx, c0, c1 = s_n / sg * math.exp(-h), k, 0.0
        if orders[i] == 2:
            r0 = (lt - schedule(spec, grid[i - 1])[2]) / h
            c0, c1 = k * (1.0 + 0.5 / r0), -0.5 * k / r0
        g = s_n * math.sqrt(-math.expm1(-2.0 * h))
        A = np.array([[cx + c0 * p, c1], [p, 0.0]])
        mean = A @ mean + np.array([c0 * q, q])
        cov = A @ cov @ A.T + np.diag([g * g, 0.0])
    return float(mean[0]), math.sqrt(cov[0, 0])

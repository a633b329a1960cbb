"""DPMSolverSampler on the host: the time grids, the order rule, the package's fp32 rows against the fp64 oracle update, the
unchanged DPMSolverDiffusion rows, argument validation and the convergence rates of the fp64 oracle on Gaussian data.  Needs no
GPU."""
import functools
import math

import numpy as np
import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from diffusion_model_nemo_b200.modules import sde as S
from oracle import ref_port as O
import dpm_oracle as D
import score_dpm_oracle as SO

MU, SD, XT = 0.3, 0.5, 1.7


def _sde(kind):
    return M.VPSDE() if kind == "vp" else M.VESDE()


def _sampler(kind, **kw):
    s = M.DPMSolverSampler(**kw)
    s.update_sde(_sde(kind))
    return s


@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("skip_type", ["logSNR", "time_uniform"])
@pytest.mark.parametrize("steps", [1, 2, 10, 20, 1000])
def test_grid_endpoints_and_monotonicity(kind, skip_type, steps):
    s = _sampler(kind, steps=steps, skip_type=skip_type)
    ts = s.timesteps()
    eps = _sde(kind).sampling_epsilon
    assert len(ts) == steps + 1 and ts[0] == 1.0 and ts[-1] == eps
    assert all(a > b for a, b in zip(ts, ts[1:]))
    assert _sampler(kind, steps=steps, skip_type=skip_type, eps=0.02).timesteps()[-1] == 0.02


@pytest.mark.parametrize("kind", ["vp", "ve"])
def test_logsnr_grid_is_uniform_in_lambda_and_the_inverse_round_trips(kind):
    sde = _sde(kind)
    ts = _sampler(kind, steps=25).timesteps()
    lam = np.array([S.score_sde_schedule(sde, t)[2] for t in ts])
    d = np.diff(lam)
    assert float(np.abs(d - d.mean()).max()) <= 1e-12 * float(np.abs(lam).max())
    for t in np.linspace(1e-5, 1.0, 97):
        back = S.score_sde_inverse_lambda(sde, S.score_sde_schedule(sde, float(t))[2])
        assert abs(back - t) <= 1e-12, (t, back)
    # the schedule is score_sde's marginal_prob and ScoreFunction.scale's std
    t = torch.tensor([0.001, 0.3, 1.0], dtype=torch.float64)
    a, sg, _ = zip(*(S.score_sde_schedule(sde, float(v)) for v in t))
    mean, std = sde.marginal_prob(torch.ones(3, 1, 1, 1, dtype=torch.float64), t)
    assert np.allclose(a, mean.flatten().numpy(), rtol=1e-14) and np.allclose(sg, std.numpy(), rtol=1e-13)


def test_ve_grids_coincide():
    for steps in (1, 7, 20, 100):
        a = _sampler("ve", steps=steps).timesteps()
        b = _sampler("ve", steps=steps, skip_type="time_uniform").timesteps()
        assert np.allclose(a, b, rtol=0, atol=1e-14)


@pytest.mark.parametrize("steps", [1, 2, 3, 5, 14, 15, 20])
@pytest.mark.parametrize("order", [1, 2, 3])
def test_order_rule(steps, order):
    got = _sampler("vp", steps=steps, order=order).step_orders()
    assert got == SO.step_orders(steps, order)
    assert got[0] == 1 and len(got) == steps
    assert got[:3] == [min(order, i + 1, steps - i) if steps < 15 else min(order, i + 1) for i in range(min(3, steps))]
    if steps < 15:
        assert got[-1] == 1 and all(o <= steps - i for i, o in enumerate(got))
    else:
        assert got[-1] == order


def _kernel_update(row, g_row, x, mo, ring, z):
    """dmn_dpmpp_step / dmn_dpmpp_sde_step's formula (include/dmn_b200.h) in fp64 from one fp32 row, mode 2 (no clamp)."""
    cx, c0, c1, c2, kx, km, slot, mode = (float(v) for v in row.double())
    assert mode == 2.0
    slot = int(slot)
    m = kx * x - km * mo
    out = cx * x + c0 * m
    if c1 != 0:
        out = out + c1 * ring[(slot + 2) % 3]
    if c2 != 0:
        out = out + c2 * ring[(slot + 1) % 3]
    if g_row is not None:
        out = out + float(g_row[0]) * z
    return out, m


# fp32 rounding of the rows only: measured max |dx| / max(1, |x'|) <= 6.7e-8 over the cases below (VE's k_m = -sigma^2 reaches -2500)
ROW_TOL = 3e-7


@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("algorithm", ["dpmsolver++", "sde-dpmsolver++"])
@pytest.mark.parametrize("skip_type,steps", [("logSNR", 20), ("logSNR", 10), ("time_uniform", 50)])
def test_package_rows_reproduce_oracle_update(kind, algorithm, skip_type, steps):
    g = torch.Generator().manual_seed(7)
    spec = O.SDESpec(kind)
    for order in ((1, 2, 3) if algorithm == "dpmsolver++" else (1, 2)):
        s = _sampler(kind, steps=steps, order=order, skip_type=skip_type, algorithm_type=algorithm)
        coef, coef2, labels = s.rows()
        ts, orders = s.timesteps(), s.step_orders()
        assert coef.shape == (steps, L.COEF_STRIDE) and coef.dtype == torch.float32
        assert (coef2 is None) == (algorithm == "dpmsolver++")
        assert torch.equal(labels, SO.labels(spec, torch.tensor(ts[:-1], dtype=torch.float64).to(torch.float32)))
        worst = 0.0
        for i in range(steps):
            row = coef[i]
            assert int(row[6]) == i % 3 and float(row[7]) == 2.0
            assert (float(row[2]) != 0) == (orders[i] >= 2) and (float(row[3]) != 0) == (orders[i] >= 3)
            sc = 1.0 if kind == "vp" else SO.schedule(spec, ts[i])[1]
            x = torch.randn(2, 3, 4, 4, generator=g, dtype=torch.float64) * sc
            mo = torch.randn(2, 3, 4, 4, generator=g, dtype=torch.float64) / (1.0 if kind == "vp" else sc)
            z = torch.randn(2, 3, 4, 4, generator=g, dtype=torch.float64)
            hist = [torch.rand(2, 3, 4, 4, generator=g, dtype=torch.float64) * 2 - 1 for _ in range(2)]
            ring = torch.full((3, 2, 3, 4, 4), float("nan"), dtype=torch.float64)
            for k in range(1, orders[i]):
                ring[(i - k) % 3] = hist[k - 1]
            got, m = _kernel_update(row, None if coef2 is None else coef2[i], x, mo, ring, z)
            m_ref = SO.data_pred(spec, x, mo, ts[i])
            tss = [ts[i - k] for k in range(orders[i])]
            if coef2 is None:
                ref = SO.update(spec, x, [m_ref] + hist[:orders[i] - 1], tss, ts[i + 1], orders[i])
            else:
                ref = SO.sde_update(spec, x, [m_ref] + hist[:orders[i] - 1], tss, ts[i + 1], orders[i], z)
            assert torch.isfinite(got).all()
            assert float((m - m_ref).abs().max()) <= 2e-7 * max(1.0, float(m_ref.abs().max()) + float(x.abs().max()))
            err = float((got - ref).abs().max()) / max(1.0, float(ref.abs().max()))
            worst = max(worst, err)
            assert err <= ROW_TOL, (order, i, err)
        print(f"{kind} {algorithm} {skip_type} steps={steps} order={order}: worst row error {worst:.2e}")


def test_dpm_solver_diffusion_rows_are_the_shared_algebra():
    """DPMSolverDiffusion builds its rows with multistep_coefs; they reproduce the oracle update of tests/dpm_oracle.py and end with
    the row into alpha_bar = 1 (test_dpm_host.py pins both; this checks the shared function on its own)."""
    from diffusion_model_nemo_b200.modules.dpm_solver_diffusion import multistep_coefs

    s = M.DPMSolverDiffusion(1000, "linear", steps=20, order=3)
    sch = D.Schedule(1000, "linear")
    pts = [t for t, _ in s.timestep_pairs()] + [-1]
    rows = multistep_coefs([sch.alpha(t) for t in pts], [sch.sigma(t) for t in pts],
                           [math.inf if t < 0 else sch.lam(t) for t in pts], s.step_orders())
    assert rows[-1] == (0.0, 1.0, 0.0, 0.0)
    assert torch.equal(torch.tensor(rows, dtype=torch.float64).to(torch.float32), s._dpm_rows()[:, :4])


def _gauss_final_err(kind, order, steps):
    spec = O.SDESpec(kind)
    s = _sampler(kind, steps=steps, order=order)
    grid = s.timesteps()
    x_T = XT * (spec.sigma_max if kind == "ve" else 1.0)
    x, _, _ = SO.solve(SO.gaussian_model(spec, MU, SD, grid), torch.full((1, 1, 1, 1), x_T, dtype=torch.float64), spec, grid, order)
    return abs(float(x) - SO.gaussian_exact(spec, MU, SD, x_T, grid[0], grid[-1]))


# measured (fp64): VP 80 -> 160 steps rates 0.99 / 1.99 / 2.05, errors at 160 steps 1.26e-2 / 1.90e-4 / 6.48e-5; VE 0.99 / 2.00 / 2.04.
# Order 3 converges at about 2: the published third-order weight of D2 integrates a quadratic data prediction wrongly.
@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("order,lo,hi", [(1, 0.9, 1.1), (2, 1.85, 2.15), (3, 1.85, 2.3)])
def test_oracle_rates_on_gaussian_data(kind, order, lo, hi):
    e80, e160 = _gauss_final_err(kind, order, 80), _gauss_final_err(kind, order, 160)
    rate = math.log2(e80 / e160)
    print(f"{kind} order {order}: err 80 {e80:.3e} 160 {e160:.3e} rate {rate:.3f}")
    assert lo <= rate <= hi
    if kind == "vp":
        assert e160 == pytest.approx({1: 1.26e-2, 2: 1.90e-4, 3: 6.48e-5}[order], rel=0.01)


# measured (fp64, VP): std error 80 -> 160 steps, order 1 2.8e-2 -> 1.5e-2, 2M 1.2e-3 -> 3.0e-4; the mean is exact to rounding
@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("order,lo,hi", [(1, 0.8, 1.1), (2, 1.8, 2.2)])
def test_sde_output_law_converges_on_gaussian_data(kind, order, lo, hi):
    spec = O.SDESpec(kind)
    x_T = XT * (spec.sigma_max if kind == "ve" else 1.0)
    errs = []
    for steps in (80, 160):
        grid = _sampler(kind, steps=steps, order=order, algorithm_type="sde-dpmsolver++").timesteps()
        m, sd = SO.sde_output_moments(spec, MU, SD, x_T, grid, order)
        em, esd = SO.gaussian_conditional(spec, MU, SD, x_T, grid[0], grid[-1])
        assert abs(m - em) <= 1e-12
        errs.append(abs(sd - esd))
    rate = math.log2(errs[0] / errs[1])
    print(f"{kind} sde order {order}: std err {errs[0]:.2e} -> {errs[1]:.2e}, rate {rate:.2f}")
    assert lo <= rate <= hi


def test_sde_moments_match_a_monte_carlo_run_of_the_oracle():
    """The closed-form law of the SDE sampler's output agrees with the fp64 oracle solver run on many independent draws."""
    spec = O.SDESpec("vp")
    grid = _sampler("vp", steps=10, order=2, algorithm_type="sde-dpmsolver++").timesteps()
    n = 200_000
    g = torch.Generator().manual_seed(3)
    zs = [torch.randn(n, 1, 1, 1, generator=g, dtype=torch.float64) for _ in range(10)]
    x, _, _ = SO.solve(SO.gaussian_model(spec, MU, SD, grid), torch.full((n, 1, 1, 1), XT, dtype=torch.float64), spec, grid, 2, zs)
    m, sd = SO.sde_output_moments(spec, MU, SD, XT, grid, 2)
    assert abs(float(x.mean()) - m) <= 5 * sd / math.sqrt(n)
    assert abs(float(x.std()) - sd) <= 5 * sd / math.sqrt(2 * n)


def test_argument_validation():
    for kw in (dict(steps=0), dict(steps=2.5), dict(steps=True), dict(order=0), dict(order=4),
               dict(order=3, algorithm_type="sde-dpmsolver++"), dict(skip_type="logSNR2"), dict(skip_type="time_quadratic"),
               dict(algorithm_type="dpmsolver"), dict(eps=0.0), dict(eps=1.5), dict(eps="1e-3")):
        with pytest.raises(ValueError):
            M.DPMSolverSampler(**kw)
    s = M.DPMSolverSampler()
    assert (s.steps, s.order, s.skip_type, s.algorithm_type, s.eps) == (20, 2, "logSNR", "dpmsolver++", None)
    assert s.seed is None and s.guidance_scale is None and s.trajectory_every == 0 and s.use_cuda_graph
    assert "DPMSolverSampler" in M.__all__
    with pytest.raises(ValueError, match="update_sde"):
        s.forward(lambda x, t: x, [1, 3, 8, 8], "cuda:0")
    with pytest.raises(ValueError, match="update_sde"):
        s.rows()

    class SubVPSDE(M.SDE):
        sampling_epsilon = 1e-3
        T = 1
        sde = marginal_prob = prior_sampling = None

    s.update_sde(SubVPSDE(1000))
    with pytest.raises(NotImplementedError, match="SDE class SubVPSDE not yet supported."):
        s.forward(lambda x, t: x, [1, 3, 8, 8], "cuda:0")
    s.update_sde(M.VPSDE())
    assert s.rows()[0].shape == (20, L.COEF_STRIDE)
    with pytest.raises(L.DmnError):          # no CPU fallback
        s.forward(lambda x, t: x, [1, 3, 8, 8], "cpu")


def test_cached_rows_follow_update_sde():
    s = _sampler("vp", steps=5)
    a = s.rows()[0]
    s.update_sde(M.VESDE())
    b = s.rows()[0]
    assert not torch.equal(a, b) and s._cache == {}


def test_config_swap_from_the_pc_sampler():
    """A config swaps `_target_` from PredictorCorrectorSampler to DPMSolverSampler; the resolved class takes its arguments."""
    cls = functools.reduce(getattr, "modules.DPMSolverSampler".split("."), __import__("diffusion_model_nemo_b200"))
    s = cls(steps=10, order=3, skip_type="time_uniform", eps=1e-3)
    s.update_sde(M.VESDE(N=2000))
    assert len(s.timesteps()) == 11 and s.timesteps()[-1] == 1e-3

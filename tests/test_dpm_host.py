"""DPM-Solver++ on the host: the fp64 oracle against the exact Gaussian-data answer, the package's fp32 coefficient rows against the
oracle's update, the order policy, the time grid and argument validation.  Needs no GPU."""
import ctypes as C
import math

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from oracle import ref_port as O
import dpm_oracle as D

S2 = 0.25


def _gauss_err(sch, order, steps, x_T):
    final, _, ms = D.solve(D.gaussian_model(sch, S2), x_T, sch, steps, order)
    exact = D.gaussian_exact(sch, S2, x_T, O.ddim_pairs(sch.T, steps)[0][0])
    # the clamp never binds, so the solver is linear and the exact answer applies
    m_max = max(float(m.abs().max()) for m in ms)
    assert m_max < 0.99, m_max
    return float((final - exact).abs().max() / exact.abs().max())


# measured slopes (linear beta, T = 1000, s^2 = 0.25): 0.99 / 2.04 / 2.89
@pytest.mark.parametrize("order,lo,hi", [(1, 0.9, 1.1), (2, 1.8, 2.3), (3, 2.6, 3.3)])
def test_oracle_converges_at_its_order_on_gaussian_data(order, lo, hi):
    sch = D.Schedule(1000, "linear")
    x_T = torch.linspace(-1.5, 1.5, 16, dtype=torch.float64).view(1, 1, 4, 4)
    e100, e200 = _gauss_err(sch, order, 100, x_T), _gauss_err(sch, order, 200, x_T)
    slope = math.log(e100 / e200) / math.log(2.0)
    print(f"order {order}: rel err K=100 {e100:.3e}, K=200 {e200:.3e}, slope {slope:.3f}")
    assert lo <= slope <= hi


def _kernel_update(row, x, mo, ring):
    """dmn_dpmpp_step's formula (include/dmn_b200.h) in fp64 from one fp32 row."""
    r = row.double()
    cx, c0, c1, c2, kx, km, slot, flag = (float(v) for v in r)
    slot = int(slot)
    e = mo[:, :x.shape[1]]
    m = (e if flag else kx * x - km * e).clamp(-1, 1)
    out = cx * x + c0 * m
    if c1 != 0:
        out = out + c1 * ring[(slot + 2) % 3]
    if c2 != 0:
        out = out + c2 * ring[(slot + 1) % 3]
    return out, m


# fp32 rounding of the rows only: measured max |dx| / max(1, |x'|) <= 4.1e-8 over the cases below
ROW_TOL = 2e-7


@pytest.mark.parametrize("objective", ["pred_noise", "pred_x0"])
@pytest.mark.parametrize("sched,T,steps", [("linear", 1000, 20), ("cosine", 1000, 50), ("linear", 1000, 10), ("cosine", 200, 200)])
def test_package_rows_reproduce_oracle_update(objective, sched, T, steps):
    g = torch.Generator().manual_seed(7)
    sch = D.Schedule(T, sched)
    for order in (1, 2, 3):
        s = M.DPMSolverDiffusion(T, sched, objective=objective, steps=steps, order=order)
        pairs = s.timestep_pairs()
        coef, _ = s._loop_tables(None, "cpu")
        orders = s.step_orders()
        assert coef.shape == (len(pairs), L.COEF_STRIDE)
        worst, bound = 0.0, False
        for i, (t, tn) in enumerate(pairs):
            row = coef[i]
            assert int(row[6]) == i % 3 and float(row[7]) == (1.0 if objective == "pred_x0" else 0.0)
            # the ring is uninitialised scratch: a slot the step's order does not use must have a zero coefficient
            assert (float(row[2]) != 0) == (orders[i] >= 2) and (float(row[3]) != 0) == (orders[i] >= 3)
            x = torch.randn(2, 3, 4, 4, generator=g, dtype=torch.float64) * 1.2
            mo = torch.randn(2, 6, 4, 4, generator=g, dtype=torch.float64) * (3.0 if i % 2 else 0.5)   # odd steps: clamp binds
            hist = [torch.rand(2, 3, 4, 4, generator=g, dtype=torch.float64) * 2 - 1 for _ in range(2)]
            ring = torch.full((3, 2, 3, 4, 4), float("nan"), dtype=torch.float64)
            if i >= 1:
                ring[(i - 1) % 3] = hist[0]
            if i >= 2:
                ring[(i - 2) % 3] = hist[1]
            got, m = _kernel_update(row, x, mo, ring)
            m_ref = D.data_pred(sch, x, mo, t, objective)
            raw = mo[:, :3] if objective == "pred_x0" else sch.k_x[t] * x - sch.k_m[t] * mo[:, :3]
            bound |= bool((raw.abs() > 1).any())
            ts = [t] + [pairs[i - k][0] for k in (1, 2) if i - k >= 0]
            ref = D.update(sch, x, [m_ref] + hist[:len(ts) - 1], ts, tn, orders[i])
            assert torch.equal(m, m_ref)
            assert torch.isfinite(got).all()
            err = float((got - ref).abs().max()) / max(1.0, float(ref.abs().max()))
            worst = max(worst, err)
            assert err <= ROW_TOL, (order, i, err)
        assert bound
        print(f"{sched} T={T} steps={steps} order={order} {objective}: worst row error {worst:.2e}")


def test_last_row_returns_the_data_prediction():
    s = M.DPMSolverDiffusion(1000, "linear", steps=20, order=3)
    coef, _ = s._loop_tables(None, "cpu")
    assert coef[-1, :4].tolist() == [0.0, 1.0, 0.0, 0.0]
    assert s.timestep_pairs()[-1] == (0, -1)


@pytest.mark.parametrize("k", [5, 10, 14, 15, 20])
@pytest.mark.parametrize("order", [1, 2, 3])
def test_step_orders(k, order):
    s = M.DPMSolverDiffusion(10 * k, "linear", steps=k, order=order)
    assert len(s.timestep_pairs()) == k
    got = s.step_orders()
    assert got == D.step_orders(k, order)
    assert got[-1] == 1 and got[0] == 1
    assert max(got) == min(order, k - 1)
    if k < 15 and k >= 3:
        assert got[-2] == min(order, 2)
    elif k >= 15:
        assert got[-2] == order
    assert got[:3] == [min(order, 1), min(order, 2), min(order, 3)][:3]


def test_grid_is_the_ddim_grid():
    for T, steps in ((1000, 20), (1000, 14), (1000, 1000), (1000, 1), (50, 7)):
        s = M.DPMSolverDiffusion(T, "cosine", steps=steps)
        assert s.timestep_pairs() == O.ddim_pairs(T, steps)
        assert s.timestep_pairs() == M.GeneralizedGaussianDiffusion(T, "cosine", ddim_timesteps=steps).timestep_pairs()
    assert len(M.DPMSolverDiffusion(1000, "linear", steps=14).timestep_pairs()) == 15     # stride 71 leaves 15 grid points
    assert M.DPMSolverDiffusion(1000, "linear", steps=1, order=3).step_orders() == [1]


def test_constructor_validation():
    for kw in (dict(steps=0), dict(steps=101), dict(steps=2.5), dict(order=0), dict(order=4)):
        with pytest.raises(ValueError):
            M.DPMSolverDiffusion(100, "linear", **kw)
    s = M.DPMSolverDiffusion(100, "linear", schedule_cfg=None, objective="pred_x0", class_conditional=True, steps=100, order=3)
    assert (s.steps, s.order, s.objective, s.use_class_conditioning) == (100, 3, "pred_x0", True)
    assert s.seed is None and s.trajectory_every == 0 and s.use_cuda_graph and s.guidance_scale is None
    with pytest.raises(NotImplementedError):
        s.p_sample(None, torch.zeros(1, 1, 4, 4), torch.zeros(1, dtype=torch.long))
    assert "DPMSolverDiffusion" in M.__all__


def test_step_entry_point_rejects_bad_arguments_before_any_launch():
    lib = L.lib()
    p = C.c_void_p(1 << 20)        # never dereferenced: the checks run first
    for batch, chw, mo_chw, hist in ((1, 6, 6, p), (1, 8, 4, p), (0, 8, 8, p), (1, 8, 10, p), (1, 8, 8, None)):
        assert lib.dmn_dpmpp_step(p, p, hist, p, batch, chw, mo_chw, p, None, 0, None) == -1
        assert lib.dmn_last_error()

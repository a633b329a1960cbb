"""Probability-flow sampling, host side (no GPU): the drift algebra of the oracle, the probability-flow predictor rows of the PC
sampler against the oracle's predictor steps, argument validation of ProbabilityFlowSampler, and of dmn_ode_sample."""
import ctypes as C
import math

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from diffusion_model_nemo_b200.modules import sde as S
from conftest import CFGS
from oracle import ref_port as O
import ode_oracle as OO


def _model(x, labels):
    """A smooth stand-in score model: depends on x and on the time label."""
    return torch.tanh(x * 0.7) * (1.0 + 0.1 * labels.float()[:, None, None, None].clamp(max=50.0)) - 0.2 * x


@pytest.mark.parametrize("kind", ["vp", "ve"])
def test_ode_drift_is_f_minus_half_g2_score(kind):
    sde = O.SDESpec(kind)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(3, 2, 4, 4, generator=g) * (1.0 if kind == "vp" else 20.0)
    t = torch.tensor([0.9, 0.5, 0.01])
    f, gg = sde.sde(x, t)
    want = f - 0.5 * gg[:, None, None, None] ** 2 * O.score_fn(_model, sde, x, t)
    got = OO.ode_drift(_model, sde, x, t)
    assert torch.allclose(got, want, rtol=1e-6, atol=1e-6 * float(want.abs().max()))
    # the probability-flow drift halves the score term of the reverse SDE and keeps f
    full = f - gg[:, None, None, None] ** 2 * O.score_fn(_model, sde, x, t)
    assert torch.allclose(2 * got - f, full, rtol=1e-5, atol=1e-5 * float(full.abs().max()))


@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("name", ["reverse_diffusion", "euler_maruyama"])
def test_probability_flow_predictor_rows_match_oracle(kind, name):
    sde = M.VPSDE(0.1, 20.0, 40) if kind == "vp" else M.VESDE(0.01, 50.0, 40)
    spec = O.SDESpec(kind, N=40)
    sf = S.ScoreFunction(_model, sde)
    g = torch.Generator().manual_seed(2)
    shape = (2, 3, 8, 8)
    for tv in (1.0, 0.6, 0.123, 1e-3):
        t = torch.ones(shape[0]) * tv
        x = torch.randn(shape, generator=g) * (1.0 if kind == "vp" else 10.0)
        z = torch.randn(shape, generator=g)
        a, b, gcol = S.predictor_rows(name, sde, sf, t[:1], probability_flow=True)
        assert float(gcol.abs().max()) == 0.0                  # no diffusion term: z is drawn but multiplied by 0
        m = _model(x, sf.labels(t))
        mean = a[0] * x + b[0] * m
        step = OO.rd_predictor_step if name == "reverse_diffusion" else OO.em_predictor_step
        ref_x, ref_mean = step(_model, spec, x, t, z, probability_flow=True)
        scale = max(1.0, float(ref_mean.abs().max()))
        assert float((mean - ref_mean).abs().max()) <= 1e-6 * scale, (kind, name, tv)
        assert torch.equal(ref_x, ref_mean)
        # probability_flow=False keeps the existing rows
        a0, b0, g0 = S.predictor_rows(name, sde, sf, t[:1])
        ref_x0, ref_mean0 = step(_model, spec, x, t, z)
        assert float((a0[0] * x + b0[0] * m - ref_mean0).abs().max()) <= 1e-6 * max(1.0, float(ref_mean0.abs().max()))


def test_probability_flow_sampler_validation():
    with pytest.raises(NotImplementedError):
        M.ProbabilityFlowSampler(method="RK23")
    for bad in (dict(rtol=[1e-5, 1e-4]), dict(atol=torch.ones(3)), dict(rtol=0.0), dict(atol=-1.0), dict(rtol=float("nan")),
                dict(max_nfe=1), dict(max_nfe=2.5)):
        with pytest.raises(ValueError):
            M.ProbabilityFlowSampler(**bad)
    s = M.ProbabilityFlowSampler()
    assert (s.denoise, s.rtol, s.atol, s.method, s.eps, s.max_nfe) == (False, 1e-5, 1e-5, "RK45", None, 100_000)
    with pytest.raises(ValueError):        # update_sde first, as the reference asks
        s.forward(lambda x, t: x, [1, 3, 8, 8], "cuda:0")
    s.update_sde(M.VPSDE())
    with pytest.raises(Exception):         # CUDA devices only; no CPU path
        s.forward(lambda x, t: x, [1, 3, 8, 8], "cpu")
    # the PC predictors accept the flag now
    sde = M.VPSDE()
    p = M.ReverseDiffusionPredictor(sde, S.ScoreFunction(_model, sde), probability_flow=True)
    assert p.probability_flow


def _desc(**kw):
    d = L.OdeDesc()
    d.sde_kind, d.N, d.beta_0, d.beta_1 = L.SDE_VP, 1000, 0.1, 20.0
    d.t0, d.t1, d.rtol, d.atol, d.max_nfe, d.batch, d.use_graph = 1.0, 1e-3, 1e-5, 1e-5, 1000, 2, 0
    d.state_dev, d.work_dev, d.result_dev = 256, 4096, 512
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def test_ode_sample_argument_validation():
    lib = L.lib()
    cfg, size, b = CFGS["tiny"]
    c = L.UnetCfg()
    c.dim, c.n_mults = cfg["dim"], len(cfg["dim_mults"])
    for i, m in enumerate(cfg["dim_mults"]):
        c.dim_mults[i] = m
    c.channels, c.out_dim, c.groups, c.with_time_emb, c.num_classes = 1, 1, cfg["groups"], 1, -1
    c.image_size, c.max_batch, c.act_dtype, c.conv_engine, c.max_time_rows = size, b, L.ACT_F32, L.CONV_SIMT, 8
    h = C.c_void_p()
    L.check(lib.dmn_plan_create(C.byref(c), C.byref(h)))
    try:
        n = b * size * size
        need = lib.dmn_ode_work_bytes(h, b)
        assert need >= n * (2 * 8 + 9 * 4)                  # y / y_new fp64, K[7] + U-Net input + output fp32
        assert lib.dmn_ode_work_bytes(h, 0) == 0
        good = dict(state_elems=n, work_bytes=need)
        assert lib.dmn_ode_sample(None, C.byref(_desc(**good)), None) == -1
        assert lib.dmn_ode_sample(h, None, None) == -1
        bad = [dict(rtol=0.0), dict(rtol=-1e-3), dict(atol=-1.0), dict(rtol=math.nan), dict(atol=math.inf), dict(t1=1.0),
               dict(max_nfe=1), dict(sde_kind=7), dict(batch=b + 1), dict(batch=0), dict(state_dev=None), dict(work_dev=None),
               dict(result_dev=None), dict(work_bytes=need - 1), dict(state_elems=n + 4), dict(work_dev=4096 + 8),
               dict(sde_kind=L.SDE_VE, sigma_min=0.0, sigma_max=50.0)]
        for kw in bad:
            d = _desc(**{**good, **kw})
            assert lib.dmn_ode_sample(h, C.byref(d), None) == -1, kw
            assert lib.dmn_last_error()
        # a valid descriptor reaches the plan-state check (nothing bound or loaded): call-order error, not a launch
        assert lib.dmn_ode_sample(h, C.byref(_desc(**good)), None) == -4
    finally:
        lib.dmn_plan_destroy(h)


def test_ode_oracle_reproduces_scipy_counts_for_the_zero_model():
    """The counts the exact controller check on the GPU compares against (B=2, 3x16x16, randn seed 0)."""
    shape = [2, 3, 16, 16]
    for kind, tol, eps, nfev, n_acc in (("vp", 1e-5, 1e-3, 92, 14), ("vp", 1e-3, 1e-3, 38, 6), ("ve", 1e-5, 1e-5, 44, 7)):
        g = torch.Generator().manual_seed(0)
        x, got, sol = OO.sample_probability_flow(OO.zero_model, shape, O.SDESpec(kind), lambda s: torch.randn(tuple(s), generator=g),
                                                 rtol=tol, atol=tol, eps=eps)
        assert (got, len(sol.t) - 1) == (nfev, n_acc), (kind, tol)

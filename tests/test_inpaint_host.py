"""RePaint inpainting on the host: the jump schedule and its events, the package's per-event rows against the sampler's own rows and
the fp64 formulas of tests/inpaint_oracle.py, argument validation, the C entry points' argument checks, and what the event recursion
computes on a two-pixel Gaussian prior with a closed-form eps-model.  Needs no GPU."""
import ctypes as C

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from diffusion_model_nemo_b200.modules.gaussian_diffusion import inpaint_events, repaint_schedule
import inpaint_oracle as IO


@pytest.mark.parametrize("k,j,r", [(1, 1, 1), (10, 1, 1), (10, 3, 1), (10, 3, 2), (10, 1, 4), (20, 5, 3), (50, 3, 3), (250, 10, 10),
                                   (7, 6, 2)])
def test_schedule_and_event_count(k, j, r):
    ts = repaint_schedule(k, j, r)
    assert ts == IO.schedule(k, j, r)
    assert ts[0] == k - 1 and ts[-1] == -1 and min(ts) == -1 and max(ts) == k - 1
    assert all(abs(b - a) == 1 for a, b in zip(ts[:-1], ts[1:]))
    ev = inpaint_events(ts)
    assert ev == IO.events(ts)
    assert len(ev) == IO.n_events(k, j, r) == sum(b < a for a, b in zip(ts[:-1], ts[1:]))
    assert ev[0] == (k - 1, None) and ev[-1][0] == 0
    for i, a in ev:
        assert a is None or (0 <= a < i and i - a == j)
    if r == 1:
        assert ts == list(range(k - 1, -2, -1)) and all(a is None for _, a in ev)
    assert IO.n_events(250, 10, 10) == 2410


def _samplers():
    return [M.GaussianDiffusion(40, "linear"), M.GaussianDiffusion(30, "cosine", objective="pred_x0"),
            M.LearnedGaussianDiffusion(40, "cosine"), M.GeneralizedGaussianDiffusion(200, "linear", eta=0.5, ddim_timesteps=20),
            M.GeneralizedGaussianDiffusion(100, "cosine", eta=0.0, ddim_timesteps=30)]


def _grid(s):
    if isinstance(s, M.GeneralizedGaussianDiffusion):
        return IO.Grid("ddim", s.timesteps, s.schedule_name, s.ddim_timesteps, s.eta, s.objective)
    return IO.Grid("learned" if isinstance(s, M.LearnedGaussianDiffusion) else "ddpm", s.timesteps, s.schedule_name,
                   objective=s.objective)


# fp32 rounding of the prepare rows: measured max |row - fp64| <= 3.0e-8
PREP_TOL = 1.2e-7


@pytest.mark.parametrize("jr", [(1, 1), (3, 3), (5, 2)])
def test_event_rows(jr):
    j, r = jr
    for s in _samplers():
        grid = _grid(s)
        k = len(grid.g)
        coef, times, prep, labels = s._inpaint_tables(j, r, "cpu")
        base, base_t = s._loop_tables(s._visit_order(), "cpu")
        ev = IO.events(IO.schedule(k, j, r))
        assert coef.shape == (len(ev), L.COEF_STRIDE) and prep.shape == (len(ev) + 1, L.COEF_STRIDE)
        assert labels == [grid.g[i] for i, _ in ev] and times.tolist() == [float(t) for t in labels]
        worst = 0.0
        for e, (i, a) in enumerate(ev):
            # the update row of an event is the sampler's own visit-order row for its grid index
            assert torch.equal(coef[e], base[k - 1 - i]) and float(base_t[k - 1 - i]) == grid.g[i]
            ref = torch.tensor(grid.prep_row(i, a), dtype=torch.float64)
            worst = max(worst, float((prep[e, :4].double() - ref).abs().max()))
            assert (float(prep[e, 1]) != 0) == (a is not None) and float(prep[e, 3]) > 0
            assert not prep[e, 4:].any()
            if a is None:
                assert prep[e, 0] == 1.0 and prep[e, 1] == 0.0
        assert worst <= PREP_TOL, worst
        assert prep[-1].tolist() == [1.0, 0.0, 1.0, 0.0, 0.0, 0.0, 0.0, 0.0]
        assert ev[0] == (k - 1, None) and labels[0] == grid.g[-1] and labels[-1] == grid.g[0]
        # j = r = 1: the update rows are the sampler's table in visit order
        if (j, r) == (1, 1):
            assert torch.equal(coef, base) and torch.equal(times, base_t)


def test_tables_are_cached():
    s = M.GaussianDiffusion(20, "linear")
    a = s._inpaint_tables(2, 2, "cpu")
    b = s._inpaint_tables(2, 2, "cpu")
    assert all(x is y for x, y in zip(a[:3], b[:3]))
    assert s._inpaint_tables(2, 3, "cpu")[0] is not a[0]


def test_argument_validation():
    s = M.GaussianDiffusion(20, "linear")
    x = torch.zeros(2, 3, 8, 8)
    m = torch.ones(1, 1, 8, 8)
    bad = [
        dict(x_known=torch.zeros(3, 8, 8), mask=m),
        dict(x_known=x, mask=torch.ones(2, 2, 8, 8)),
        dict(x_known=x, mask=torch.ones(4, 3, 8, 8)),
        dict(x_known=x, mask=m * 1.5),
        dict(x_known=x, mask=m - 1.01),
        dict(x_known=x, mask=m * float("nan")),
        dict(x_known=x, mask=[1.0]),
        dict(x_known=x, mask=m, jump_length=0),
        dict(x_known=x, mask=m, jump_n_sample=0),
        dict(x_known=x, mask=m, jump_length=1.5),
        dict(x_known=x, mask=m, jump_length=20, jump_n_sample=2),
    ]
    for kw in bad:
        kw = dict(kw)
        with pytest.raises(ValueError):
            s._check_inpaint_args(kw.pop("x_known"), kw.pop("mask"), kw.get("jump_length", 1), kw.get("jump_n_sample", 1))
    s._check_inpaint_args(x, m, 19, 2)           # j < K is fine
    s._check_inpaint_args(x, m, 20, 1)           # j is unused without resampling
    s._check_inpaint_args(x, torch.tensor(0.5), 1, 1)
    d = M.GeneralizedGaussianDiffusion(100, "linear", ddim_timesteps=10)
    with pytest.raises(ValueError):
        d._check_inpaint_args(x, m, 10, 2)       # K is the DDIM grid's length
    d._check_inpaint_args(x, m, 9, 2)
    for other in (M.DPMSolverDiffusion(100, "linear", steps=10), M.WaveGradDiffusion(50, "linear")):
        with pytest.raises(NotImplementedError):
            other.inpaint(None, x, m)


def test_entry_points_reject_bad_arguments_before_any_launch():
    lib = L.lib()
    p = C.c_void_p(1 << 20)        # never dereferenced: the checks run first
    for n, args in ((6, (p, p, p, p)), (0, (p, p, p, p)), (8, (None, p, p, p)), (8, (p, None, p, p)), (8, (p, p, None, p)),
                    (8, (p, p, p, None))):
        assert lib.dmn_inpaint_prepare(*args, n, p, None, 0, L.Rng(1, 0), None) == -1
        assert lib.dmn_last_error()
    d = L.LoopDesc()
    ip = L.InpaintDesc()
    ip.known_dev = ip.mask_dev = ip.prep_coef_dev = 1 << 20
    for kind in (L.LOOP_PC, L.LOOP_BPD, L.LOOP_DPMPP, 17):
        d.kind = kind
        assert lib.dmn_sample_loop_inpaint(p, C.byref(d), C.byref(ip), None) == -1
        assert b"inpaint" in lib.dmn_last_error()
    d.kind, d.noise_dev = L.LOOP_DDPM, 1 << 20
    assert lib.dmn_sample_loop_inpaint(p, C.byref(d), C.byref(ip), None) == -1
    d.noise_dev = None
    ip.mask_dev = None
    assert lib.dmn_sample_loop_inpaint(p, C.byref(d), C.byref(ip), None) == -1
    assert lib.dmn_sample_loop_inpaint(p, C.byref(d), None, None) == -1


# ---- semantics: two correlated pixels, the first known ----------------------------------------------------------------------------
# x0 ~ N(0, s^2 [[1, rho], [rho, 1]]) with the exact eps-model; x_known = (XK, *), so E[x_u | x_k] = rho XK.  DDPM, cosine T = 250,
# B = 4096, Philox seed 1234.  Measured error of the mean of x_u: -0.0847 (r = 1, plain replacement) and -0.0260 (j = r = 10); the
# Monte-Carlo standard error of the mean is 0.0011.
S, RHO, XK = 0.15, 0.9, 0.3


def _pair_error(j, r):
    grid = IO.Grid("ddpm", 250, "cosine")
    model, seen = IO.pair_model(grid, S * S, RHO)
    shape = (4096, 1, 1, 2)
    known = torch.zeros(shape, dtype=torch.float64)
    known[..., 0] = XK
    mask = torch.tensor([1.0, 0.0], dtype=torch.float64).view(1, 1, 1, 2)
    draw = IO.philox_draws(1234, 0, shape)
    out, _ = IO.run(grid, model, draw(-1, 0), known, mask, IO.schedule(250, j, r), draw)
    assert seen[0] < 0.9, seen[0]                 # the x0 clamp never binds: the model is the exact posterior mean
    assert torch.equal(out[..., 0], known[..., 0])
    return float(out[..., 1].mean()) - RHO * XK


def test_resampling_reduces_the_conditional_mean_error():
    e1, e10 = _pair_error(10, 1), _pair_error(10, 10)
    print(f"E[x_u | x_k] error: r=1 {e1:+.4f}, j=r=10 {e10:+.4f} (target {RHO * XK:.3f})")
    assert 0.07 <= abs(e1) <= 0.10
    assert abs(e10) <= 0.035
    assert abs(e10) < 0.5 * abs(e1)

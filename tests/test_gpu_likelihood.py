"""Probability-flow ODE likelihood on the GPU (LikelihoodEstimate / dmn_ode_likelihood) against score_sde's likelihood_fn run on
the CPU oracle (tests/likelihood_oracle.py: scipy solve_ivp over the augmented state, autograd Hutchinson divergence).

  exact controller check (zero final 1x1, model == 0): VP z = x exp(-1/2 int beta) within the solver's absolute tolerance
    (z ~ 7e-3 x, so atol dominates) and equal to scipy's z, delta_logp = -1/2 D int_eps^1 beta for Rademacher noise; VE z = x and delta_logp = 0 exactly; evaluation / accepted counts equal scipy's on the same system;
  parity (random-init tiny U-Nets, injected noise; GATES below): VE at rtol = atol = 1e-3 takes scipy's evaluation count,
    |bpd - bpd_ref| <= 1e-3 and z rel-L2 <= 1e-4; VP at 1e-5 within 2 % of scipy's count, |bpd - bpd_ref| <= 5e-3 and
    z rel-L2 <= 1e-2;
  graph == plain launches == a second graph solve, bit for bit.
"""
import functools

import numpy as np
import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from conftest import CFGS, make_unet, rel_l2
from oracle import ref_port as O
from ode_oracle import zero_model
import likelihood_oracle as LO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _data(shape, seed=0):
    return torch.rand(tuple(shape), generator=torch.Generator().manual_seed(seed)) * 2 - 1


def _estimate(kind, tol, hutch="Rademacher", graph=True):
    le = M.LikelihoodEstimate(hutchinson_type=hutch, rtol=tol, atol=tol)
    le.update_sde(M.VPSDE() if kind == "vp" else M.VESDE())
    le.use_cuda_graph = graph
    return le


def _zero_tail(cfg):
    sd = O.random_state_dict(cfg, seed=0)
    for k in ("final_conv.3.weight", "final_conv.3.bias"):
        sd[k] = torch.zeros_like(sd[k])
    return sd


@pytest.mark.parametrize("kind", ["vp", "ve"])
def test_exact_controller_zero_model(kind):
    cfg = dict(dim=32, dim_mults=[1, 2], channels=3, groups=8)
    u = make_unet(cfg, _zero_tail(cfg), dtype="fp32", engine="simt", device=DEV)
    shape = (2, 3, 16, 16)
    x = _data(shape)
    e = LO.rademacher(shape, 1)
    spec = O.SDESpec(kind)
    _, zref, dref, sol = LO.likelihood(zero_model, spec, x, e, rtol=1e-5, atol=1e-5, eps=1e-5, div_fn=LO.linear_div(zero_model, spec, e))
    for graph in (False, True):
        le = _estimate(kind, 1e-5, graph=graph)
        bpd, z, nfe = le.likelihood(u, x.to(DEV), noise=e.to(DEV))
        st = le.last_stats
        assert st["status"] == L.ODE_DONE
        assert (nfe, st["n_accepted"]) == (sol.nfev, len(sol.t) - 1), (kind, graph, st, sol.nfev, len(sol.t) - 1)
        assert st["n_rejected"] == (nfe - 2) // 6 - st["n_accepted"]
        if kind == "ve":
            assert torch.equal(z.cpu(), x) and torch.equal(le_dlp(u, x), torch.zeros(2))
        else:
            ib = spec.beta_0 * (1 - 1e-5) + 0.5 * (spec.beta_1 - spec.beta_0) * (1 - 1e-10)
            D = np.prod(shape[1:])
            assert rel_l2(z.cpu(), zref) <= 1e-6
            assert float((z.cpu() - x * np.exp(-0.5 * ib)).abs().max()) <= 1e-4          # within the solver's atol-bound error
            exact = torch.full((2,), -0.5 * D * ib, dtype=torch.float64)
            got = le_dlp(u, x).double()
            assert float((got - exact).abs().max()) <= 1e-4 * abs(float(exact[0])), (got, exact)
            assert float((got - dref.double()).abs().max()) <= 1e-5 * abs(float(exact[0]))


def le_dlp(u, x):
    """delta_logp of the last solve (the log-density rows of the plan's likelihood state)."""
    plan = u.plan(x.shape[-1], x.shape[0], DEV, time_rows=6)
    n = x.numel()
    return plan._lik_bufs[x.shape[0]]["state"][n:].cpu()


# VE at rtol = atol = 1e-3 takes scipy's evaluation count.  VP runs at the default 1e-5 (at 1e-3 the absolute tolerance dominates
# z ~ 7e-3 x and both solvers are only tolerance-accurate): the flow from eps towards T expands perturbations of the stiff start,
# where the score is divided by std(eps) ~ 3e-3, so the fp32 rounding differences of a forward-mode and a reverse-mode divergence grow
# along the solve.  Measured on a B200: VE max |dbpd| 3.1e-4, z rel-L2 2.9e-5, equal counts; VP max |dbpd| 1.9e-3, z rel-L2 2.1e-3,
# counts within 0.7 %.
GATES = {"ve": dict(tol=1e-3, bpd=1e-3, z_rel=1e-4, nfe=0.0), "vp": dict(tol=1e-5, bpd=5e-3, z_rel=1e-2, nfe=0.02)}


@pytest.mark.parametrize("name", ["tiny", "tiny_cls"])
@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("hutch", ["Rademacher", "Gaussian"])
def test_parity_with_oracle(name, kind, hutch):
    cfg, size, b = CFGS[name]
    gate = GATES[kind]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = (b, cfg["channels"], size, size)
    x = _data(shape, 2)
    e = (LO.rademacher if hutch == "Rademacher" else LO.gaussian)(shape, 4)
    spec = O.SDESpec(kind)
    omodel, model = O.make_model(sd, cfg), u
    if cfg.get("num_classes") is not None:
        classes = torch.tensor([1, 7][:b])
        model = functools.partial(u.forward, classes=classes.to(DEV))
        omodel = functools.partial(O.make_model(sd, cfg), classes=classes)
    bref, zref, _, sol = LO.likelihood(omodel, spec, x, e, rtol=gate["tol"], atol=gate["tol"], eps=1e-5)
    le = _estimate(kind, gate["tol"], hutch)
    bpd, z, nfe = le.likelihood(model, x.to(DEV), noise=e.to(DEV))
    dbpd = float((bpd.cpu().double() - bref.double()).abs().max())
    zerr = rel_l2(z.cpu(), zref)
    print(f"likelihood parity {name}/{kind}/{hutch}: nfe {nfe} (scipy {sol.nfev}), |dbpd| {dbpd:.3e}, z rel-L2 {zerr:.3e}")
    assert abs(nfe - sol.nfev) <= gate["nfe"] * sol.nfev, (nfe, sol.nfev)
    assert dbpd <= gate["bpd"], dbpd
    assert zerr <= gate["z_rel"], zerr


def test_graph_equals_plain_and_is_reproducible():
    cfg, size, b = CFGS["tiny_cls"]
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="fp32", engine="simt", device=DEV)
    x = _data((4, 3, size, size), 5).to(DEV)
    runs = []
    for graph in (True, True, False):
        le = _estimate("vp", 1e-3, graph=graph)
        le.seed = 1234
        bpd, z, nfe = le.likelihood(functools.partial(u, classes=torch.tensor([0, 1, 2, 10], device=DEV)), x)
        runs.append((bpd, z, nfe, le.last_stats))
    for r in runs[1:]:
        assert torch.equal(r[0], runs[0][0]) and torch.equal(r[1], runs[0][1]) and r[2:] == runs[0][2:]
    assert runs[0][3]["status"] == L.ODE_DONE and torch.isfinite(runs[0][0]).all()
    # a different seed draws different Hutchinson noise
    le = _estimate("vp", 1e-3)
    le.seed = 99
    other, _, _ = le.likelihood(functools.partial(u, classes=torch.tensor([0, 1, 2, 10], device=DEV)), x)
    assert not torch.equal(other, runs[0][0])

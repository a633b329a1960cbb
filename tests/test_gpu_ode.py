"""Probability-flow sampling on the GPU: the device-side RK45 controller against scipy, ProbabilityFlowSampler against the CPU
oracle (tests/ode_oracle.py: scipy solve_ivp over the oracle U-Net), graph == plain launches, the max_nfe stop, and the PC
sampler with probability_flow=True.

Tolerances:
  exact controller check (zero model, drift -0.5 beta(t) x computed bit-identically): equal nfev / accepted / rejected counts and
    final max-abs <= 1e-6 * max|y| against scipy;
  parity with the oracle (random-init tiny U-Nets, fp32 mode, tolerances 1e-3): equal nfev and final rel-L2 <= 1e-5 (measured on a
    B200: at most 2.1e-6, VE; 5e-7 VP; the proposed 1e-3 was far looser than needed);
  PC with probability_flow=True: the existing PC gate, fp32 rel-L2 <= 1e-4.
"""
import functools

import numpy as np
import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from conftest import CFGS, make_unet, rel_l2
from oracle import ref_port as O
import ode_oracle as OO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _xT(shape, seed=0):
    return torch.randn(tuple(shape), generator=torch.Generator().manual_seed(seed))


def _pkg_sde(kind):
    return M.VPSDE() if kind == "vp" else M.VESDE()


def _solve(u, shape, kind, tol, z, denoise=False, graph=True, model=None, **kw):
    """z: the N(0,1) draw of x_T (the sampler scales it by sigma_max for VE, as the prior does)."""
    s = M.ProbabilityFlowSampler(denoise=denoise, rtol=tol, atol=tol, **kw)
    s.update_sde(_pkg_sde(kind))
    s.use_cuda_graph = graph
    imgs, nfe = s.sample(model if model is not None else u, shape, device=DEV, return_nfe=True, noise=z[None])
    return imgs[-1] * 2 - 1, nfe, s.last_stats


def _zero_tail(cfg, seed=0):
    sd = O.random_state_dict(cfg, seed=seed)
    for k in ("final_conv.3.weight", "final_conv.3.bias"):
        sd[k] = torch.zeros_like(sd[k])
    return sd


@pytest.mark.parametrize("mode", [("fp32", "simt", "tiny3"), ("bf16", "tcgen05", "cfg2")])
def test_exact_controller_against_scipy(mode):
    """Model output exactly 0: the drift is -0.5 beta(t) x (VP) or 0 (VE), which the device computes bit-identically to torch, so
    the device controller must take the same decisions as scipy.integrate.RK45."""
    dtype, engine, which = mode
    cfg, size = (dict(dim=32, dim_mults=[1, 2], channels=3, groups=8), 16) if which == "tiny3" else CFGS["cfg2"][:2]
    u = make_unet(cfg, _zero_tail(cfg), dtype=dtype, engine=engine, device=DEV)
    shape = [2, 3, size, size]
    cases = [("vp", 1e-5), ("vp", 1e-3), ("ve", 1e-5)]
    for kind, tol in cases:
        spec = O.SDESpec(kind)
        ref, nfev, sol = OO.sample_probability_flow(OO.zero_model, shape, spec, lambda s: _xT(s), rtol=tol, atol=tol)
        n_acc = len(sol.t) - 1
        for graph in (False, True):
            got, nfe, st = _solve(u, shape, kind, tol, _xT(shape), graph=graph)
            assert (nfe, st["n_accepted"]) == (nfev, n_acc), (mode, kind, tol, graph, st, nfev, n_acc)
            assert st["n_rejected"] == nfev // 6 - n_acc, st       # every attempt costs 6 evaluations after the 2 of the init
            assert st["status"] == L.ODE_DONE
            # the [0,1] image round trip costs one fp32 rounding of |x| <= max|y|
            scale = float(ref.abs().max())
            assert float((got - ref).abs().max()) <= 1e-6 * scale + 2 * np.finfo(np.float32).eps * scale, (mode, kind, tol, graph)


@pytest.mark.parametrize("name", ["tiny", "tiny_cls"])
@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("denoise", [False, True])
def test_parity_with_oracle(name, kind, denoise):
    cfg, size, b = CFGS[name]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = [b, cfg["channels"], size, size]
    spec = O.SDESpec(kind)
    omodel = O.make_model(sd, cfg)
    model = u
    if cfg.get("num_classes") is not None:
        classes = torch.tensor([1, 7][:b])
        model = functools.partial(u.forward, classes=classes.to(DEV))
        omodel = functools.partial(O.make_model(sd, cfg), classes=classes)
    ref, nfev, _ = OO.sample_probability_flow(omodel, shape, spec, lambda s: _xT(s, 3), rtol=1e-3, atol=1e-3, denoise=denoise)
    got, nfe, st = _solve(u, shape, kind, 1e-3, _xT(shape, 3), denoise=denoise, model=model)
    assert nfe == nfev, (name, kind, denoise, st, nfev)
    err = rel_l2(got, ref)
    assert err <= 1e-5, (name, kind, denoise, err)
    print(f"parity {name}/{kind}/denoise={denoise}: nfev {nfe}, rel-L2 {err:.3e}")


def test_graph_equals_plain_and_is_reproducible():
    """Benchmark shape at B=8 in bf16: graph and plain launches, and two graph runs, give the same bits and the same counts."""
    cfg, size, _ = CFGS["cfg2"]
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
    shape = [8, 3, size, size]
    xT = _xT(shape, 5)
    a, na, sa = _solve(u, shape, "vp", 1e-3, xT, graph=True)
    b, nb, sb = _solve(u, shape, "vp", 1e-3, xT, graph=True)
    c, nc, sc = _solve(u, shape, "vp", 1e-3, xT, graph=False)
    assert torch.equal(a, b) and torch.equal(a, c)
    assert sa == sb == sc and na == nb == nc
    assert sa["status"] == L.ODE_DONE and torch.isfinite(a).all()


def test_max_nfe_stops_the_solve():
    cfg, size, b = CFGS["tiny"]
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="fp32", engine="simt", device=DEV)
    shape = [b, 1, size, size]
    for graph in (True, False):
        s = M.ProbabilityFlowSampler(max_nfe=20)
        s.update_sde(M.VPSDE())
        s.use_cuda_graph = graph
        with pytest.raises(RuntimeError, match="20 model evaluations"):
            s.sample(u, shape, device=DEV, noise=_xT(shape)[None])
        assert s.last_stats["status"] == L.ODE_LIMIT and s.last_stats["nfev"] == 20
        assert s.last_stats["t_final"] > 1e-3
    # the sampler is usable again afterwards
    s.max_nfe = 100_000
    s.sample(u, shape, device=DEV, noise=_xT(shape)[None])
    assert s.last_stats["status"] == L.ODE_DONE


def test_foreign_model_is_rejected():
    s = M.ProbabilityFlowSampler()
    s.update_sde(M.VPSDE())
    with pytest.raises(NotImplementedError):
        s.sample(lambda x, t: torch.zeros_like(x), [1, 1, 16, 16], device=DEV)


@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("pc", [("reverse_diffusion", "langevin"), ("euler_maruyama", "none")])
def test_pc_probability_flow(kind, pc):
    cfg, size, b = CFGS["tiny_g4"]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = [b, 3, size, size]
    N = 40
    draws = 1 + N * (2 if pc[1] != "none" else 1)
    q = O.NoiseQueue(5)
    noise = torch.stack([q(shape) for _ in range(draws)])
    spec = O.SDESpec(kind, N=N)
    ref, _ = OO.sample_pc(O.make_model(sd, cfg), shape, spec, O.NoiseQueue(5), predictor=pc[0], corrector=pc[1], snr=0.16,
                          denoise=True, probability_flow=True)
    sde = M.VPSDE(0.1, 20.0, N) if kind == "vp" else M.VESDE(0.01, 50.0, N)
    outs = []
    for model in (u, lambda x, t: u(x, t)):           # native loop, then the plugin path (per-step update_fn calls)
        s = M.PredictorCorrectorSampler(pc[0], pc[1], snr=0.16, n_steps=1, probability_flow=True, denoise=True)
        s.update_sde(sde)
        imgs = s.sample(model, shape, device=DEV, noise=noise)
        outs.append(imgs[-1] * 2 - 1)
    for got in outs:
        assert rel_l2(got, ref) <= 1e-4, (kind, pc, rel_l2(got, ref))
    assert rel_l2(outs[0], outs[1]) <= 1e-5

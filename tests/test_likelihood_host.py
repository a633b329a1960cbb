"""LikelihoodEstimate and Unet.jvp without a GPU: argument validation and error types, the bits/dim tail against the oracle,
and the C-ABI checks of dmn_unet_jvp / dmn_ode_likelihood that need no device."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from diffusion_model_nemo_b200.modules.sde import likelihood_bpd
from conftest import CFGS, make_unet, make_wavegrad_unet, WG_CFGS
from oracle import ref_port as O
import likelihood_oracle as LO


def test_constructor_validation():
    with pytest.raises(NotImplementedError):
        M.LikelihoodEstimate(hutchinson_type="Bernoulli")
    with pytest.raises(NotImplementedError):
        M.LikelihoodEstimate(method="RK23")
    for kw in (dict(rtol=0), dict(atol=-1.0), dict(eps=float("nan")), dict(rtol=[1e-5]), dict(max_nfe=1), dict(max_nfe=True)):
        with pytest.raises(ValueError):
            M.LikelihoodEstimate(**kw)
    le = M.LikelihoodEstimate()
    assert (le.hutchinson_type, le.rtol, le.atol, le.eps, le.max_nfe) == ("Rademacher", 1e-5, 1e-5, 1e-5, 100_000)
    assert le.use_cuda_graph and le.seed is None and le.last_stats is None


def test_likelihood_argument_errors():
    cfg = CFGS["tiny"][0]
    data = torch.zeros(2, 1, 16, 16)
    le = M.LikelihoodEstimate()
    with pytest.raises(ValueError):                         # no SDE yet
        le.likelihood(make_unet(cfg), data)
    le.update_sde(M.VPSDE())
    with pytest.raises(NotImplementedError):                # not this package's Unet
        le.likelihood(lambda x, t: x, data)
    with pytest.raises(ValueError):                         # bf16 U-Net
        le.likelihood(make_unet(cfg, dtype="bf16", engine="tcgen05"), data)
    wg = make_wavegrad_unet(WG_CFGS["wg_tiny"][0])
    with pytest.raises(NotImplementedError):
        le.likelihood(wg, torch.zeros(2, 3, 16, 16))
    u = make_unet(cfg)
    with pytest.raises(ValueError):                         # wrong channel count
        le.likelihood(u, torch.zeros(2, 3, 16, 16))
    with pytest.raises(ValueError):                         # noise of another shape
        le.likelihood(u, data, noise=torch.zeros(2, 1, 8, 8))
    with pytest.raises(L.DmnError):                         # CPU tensors: no CPU fallback
        le.likelihood(functools.partial(u, classes=None), data)


def test_jvp_errors():
    cfg = CFGS["tiny"][0]
    x = torch.zeros(2, 1, 16, 16)
    with pytest.raises(ValueError):
        make_unet(cfg, dtype="bf16", engine="tcgen05").jvp(x, torch.zeros(2), x)
    with pytest.raises(NotImplementedError):
        make_wavegrad_unet(WG_CFGS["wg_tiny"][0]).jvp(torch.zeros(2, 3, 16, 16), torch.zeros(2), torch.zeros(2, 3, 16, 16))


@pytest.mark.parametrize("kind", ["vp", "ve"])
def test_bpd_formula_matches_oracle(kind):
    sde = M.VPSDE() if kind == "vp" else M.VESDE()
    spec = O.SDESpec(kind)
    g = torch.Generator().manual_seed(3)
    z = torch.randn(3, 3, 8, 8, generator=g) * (1.0 if kind == "vp" else 50.0)
    dlp = torch.randn(3, generator=g) * 100
    ref = -(LO.prior_logp(spec, z) + dlp) / np.log(2) / (3 * 8 * 8) + 7.0
    assert torch.allclose(likelihood_bpd(sde, z, dlp), ref, rtol=0, atol=1e-6)


def _plan(act, eng):
    cfg, size, b = CFGS["tiny"]
    c = L.UnetCfg()
    c.dim, c.n_mults = cfg["dim"], len(cfg["dim_mults"])
    for i, m in enumerate(cfg["dim_mults"]):
        c.dim_mults[i] = m
    c.channels, c.out_dim, c.groups, c.with_time_emb, c.num_classes = cfg["channels"], cfg["channels"], cfg["groups"], 1, -1
    c.image_size, c.max_batch, c.act_dtype, c.conv_engine, c.max_time_rows = size, b, act, eng, 8
    h = C.c_void_p()
    L.check(L.lib().dmn_plan_create(C.byref(c), C.byref(h)))
    return h


def test_cabi_checks_without_device():
    lib = L.lib()
    h = _plan(L.ACT_BF16, L.CONV_TCGEN05)
    try:
        assert lib.dmn_unet_jvp(h, None, None, None, None, None, None, None, 0, 1, None) == -2
        assert b"fp32" in lib.dmn_last_error()
        d = L.OdeLikelihoodDesc()
        assert lib.dmn_ode_likelihood(h, C.byref(d), None) == -2
    finally:
        lib.dmn_plan_destroy(h)
    h = _plan(L.ACT_F32, L.CONV_SIMT)
    try:
        assert lib.dmn_unet_jvp(h, None, None, None, None, None, None, None, 0, 1, None) == -1      # null tensors
        assert lib.dmn_ode_likelihood(h, None, None) == -1
        assert lib.dmn_unet_jvp_work_bytes(h, 2) > lib.dmn_plan_workspace_bytes(h)
        assert lib.dmn_unet_jvp_work_bytes(h, 0) == 0
        assert lib.dmn_ode_likelihood_work_bytes(h, 2) > lib.dmn_ode_work_bytes(h, 2) + lib.dmn_unet_jvp_work_bytes(h, 2)
        d = L.OdeLikelihoodDesc()
        d.sde_kind, d.N, d.beta_0, d.beta_1, d.t0, d.t1, d.rtol, d.atol, d.max_nfe, d.batch = L.SDE_VP, 1000, 0.1, 20, 1e-5, 1, 1e-5, 1e-5, 100, 2
        d.hutchinson = 5
        d.state_dev = d.work_dev = d.result_dev = 256
        assert lib.dmn_ode_likelihood(h, C.byref(d), None) == -1
        assert b"Hutchinson" in lib.dmn_last_error()
        d.hutchinson = L.HUTCH_RADEMACHER
        d.state_elems = 2 * 16 * 16                          # missing the log-density rows
        assert lib.dmn_ode_likelihood(h, C.byref(d), None) == -1
        assert b"state_dev" in lib.dmn_last_error()
    finally:
        lib.dmn_plan_destroy(h)

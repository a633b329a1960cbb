"""DPMSolverSampler (DPM-Solver++ and SDE-DPM-Solver++ for VP / VE score models) on the GPU.

1. dmn_dpmpp_step (mode 2, no clamp) and dmn_dpmpp_sde_step against the fp64 row formula for every order and ring slot, with
   injected noise; the in-kernel draw of step s is dmn_randn's draw for step s.
2. The Gaussian-data problem (exact answer known) through the foreign-callable path: the device's error against the exact
   probability-flow map equals the fp64 oracle's to fp32 rounding.
3. SDE-DPM-Solver++ with Philox noise on the Gaussian problem at 786k elements: sample moments against the closed-form law,
   reproducibility per seed.
4. Native loops on tiny / tiny_cls fp32 U-Nets against the fp64 oracle solver over oracle.ref_port's U-Net, graph == plain
   launches, native == foreign path, classifier-free guidance against two oracle calls.
5. Convergence towards ProbabilityFlowSampler's tight RK45 solve from the same x_T.

Gates: measured maxima on an NVIDIA B200 (1000 W power limit) beside each constant.  Moments of test 3 measured within 1.6
standard errors; distances to RK45 (rtol = atol = 1e-6) at 10 / 20 / 50 / 100 steps: VP 5.6e-2 / 2.1e-2 / 6.9e-3 / 2.1e-3,
VE 0.97 / 0.60 / 0.31 / 0.17 (random-init weights).
"""
import functools
import math

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from conftest import CFGS, make_unet, rel_l2
from oracle import ref_port as O
import score_dpm_oracle as SO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 0x5EED0FD9A11CE
MU, SD = 0.3, 0.5


def _sampler(kind, **kw):
    s = M.DPMSolverSampler(**kw)
    s.update_sde(M.VPSDE() if kind == "vp" else M.VESDE())
    return s


def _state(img):
    return img.double() * 2.0 - 1.0


def _randn_dev(shape, seed, step=-1):
    out = torch.empty(shape, device=DEV)
    L.check(L.lib().dmn_randn(L.ptr(out), out.numel(), L.Rng(seed, 0), step, L.stream_ptr(DEV)), "dmn_randn")
    return out


# ---- 1. the update kernel ----------------------------------------------------------------------------------------------------
# Gate in units of fp32 rounding: |x' - ref| <= KTOL * 2^-24 * (|c_x x| + |c_0| (|m| + |k_x x| + |k_m e|) + |c_1 m1| + |c_2 m2| + |g z|)
# and |m - ref| <= KTOL * 2^-24 * (|k_x x| + |k_m e|).  KTOL as test_gpu_dpm.py's kernel test; measured on a B200: ratios <= 2.43
# (update) and <= 1.96 (ring).
KTOL = 8.0
EPS32 = 2.0 ** -24


@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("algorithm", ["dpmsolver++", "sde-dpmsolver++"])
def test_step_kernel_matches_fp64_update(kind, algorithm):
    lib = L.lib()
    st = L.stream_ptr(DEV)
    b, shape = 512, (512, 3, 32, 32)         # 196608 float4 > the 1184 x 256 grid: the grid-stride loop runs
    chw = 3 * 32 * 32
    g = torch.Generator().manual_seed(1)
    worst = [0.0, 0.0]
    for order in ((1, 2, 3) if algorithm == "dpmsolver++" else (1, 2)):
        s = _sampler(kind, steps=20, order=order, algorithm_type=algorithm)
        coef, coef2, _ = s.rows()
        coef_d = coef.to(DEV)
        coef2_d = None if coef2 is None else coef2.to(DEV)
        orders, ts = s.step_orders(), s.timesteps()
        for i in [order - 1, order, order + 1, 19]:
            o = orders[i]
            sc = 1.0 if kind == "vp" else SO.schedule(O.SDESpec(kind), ts[i])[1]
            x = torch.randn(shape, generator=g) * sc
            mo = torch.randn(shape, generator=g) / (1.0 if kind == "vp" else sc)
            z = torch.randn(shape, generator=g)
            hist = [torch.rand(shape, generator=g) * 2 - 1 for _ in range(2)]
            ring = torch.full((3,) + shape, float("nan"), device=DEV)
            for k in range(1, o):
                ring[(i - k) % 3] = hist[k - 1].to(DEV)
            xd, mod, zd = x.to(DEV), mo.to(DEV), z.to(DEV)
            if coef2 is None:
                rc = lib.dmn_dpmpp_step(L.ptr(xd), L.ptr(mod), L.ptr(ring), L.ptr(xd), b, chw, chw, L.ptr(coef_d), None, i, st)
            else:
                rc = lib.dmn_dpmpp_sde_step(L.ptr(xd), L.ptr(mod), L.ptr(zd), L.ptr(ring), L.ptr(xd), b, chw, chw, L.ptr(coef_d),
                                            L.ptr(coef2_d), None, i, L.Rng(1, 0), st)
            L.check(rc, "dpmpp step")
            torch.cuda.synchronize()
            r = [float(v) for v in coef[i].double()]
            gz = 0.0 if coef2 is None else float(coef2[i, 0])
            xx, e = x.double(), mo.double()
            m_ref = r[4] * xx - r[5] * e
            ref = r[0] * xx + r[1] * m_ref + gz * z.double()
            if o >= 2:
                ref = ref + r[2] * hist[0].double()
            if o >= 3:
                ref = ref + r[3] * hist[1].double()
            got = xd.double().cpu()
            assert torch.isfinite(got).all(), (order, i)
            sm = abs(r[4]) * xx.abs() + abs(r[5]) * e.abs()
            bound = (abs(r[0]) * xx.abs() + abs(r[1]) * (m_ref.abs() + sm) + abs(r[2]) * hist[0].double().abs()
                     + abs(r[3]) * hist[1].double().abs() + abs(gz) * z.double().abs())
            err = float(((got - ref).abs() / (EPS32 * bound + 1e-30)).max())
            merr = float(((ring[i % 3].double().cpu() - m_ref).abs() / (EPS32 * sm + 1e-30)).max())
            worst = [max(worst[0], err), max(worst[1], merr)]
            assert err <= KTOL, (order, i, err)
            assert merr <= KTOL, (order, i, merr)
            if coef2 is not None:
                # in-kernel noise: step i draws dmn_randn's quads for step i (counter word (i + 1) * 8, never x_T's word 0)
                xa, xb = x.to(DEV), x.to(DEV)
                for zz, out in ((None, xa), (_randn_dev(shape, SEED, step=i), xb)):
                    L.check(lib.dmn_dpmpp_sde_step(L.ptr(out), L.ptr(mod), L.ptr(zz), L.ptr(ring), L.ptr(out), b, chw, chw,
                                                   L.ptr(coef_d), L.ptr(coef2_d), None, i, L.Rng(SEED, 0), st), "dmn_dpmpp_sde_step")
                assert torch.equal(xa, xb)
    print(f"{kind} {algorithm}: worst update error {worst[0]:.2f}, ring {worst[1]:.2f} (units of fp32 rounding)")


def test_sde_step_entry_point_rejects_bad_arguments():
    lib = L.lib()
    p = L.ptr(torch.zeros(64, device=DEV))
    assert lib.dmn_dpmpp_sde_step(p, p, None, p, p, 1, 8, 8, p, None, None, 0, L.Rng(1, 0), None) == -1      # no noise table
    assert lib.dmn_dpmpp_sde_step(p, p, None, p, p, 1, 6, 6, p, p, None, 0, L.Rng(1, 0), None) == -1         # chw % 4
    assert lib.dmn_last_error()


# ---- 2. Gaussian data through the foreign-callable path ------------------------------------------------------------------------
def _gauss_device_model(kind, grid):
    """The optimal output on the device (fp32 affine map per grid time), looked up by the label the sampler passes."""
    spec = O.SDESpec(kind)
    lab = SO.labels(spec, torch.tensor(grid[:-1], dtype=torch.float64).to(torch.float32)).tolist()
    ab = []
    for t in grid[:-1]:
        a, sg, _ = SO.schedule(spec, t)
        d = a * a * SD * SD + sg * sg if kind == "vp" else SD * SD + sg * sg
        ab.append((sg / d, -sg * a * MU / d) if kind == "vp" else (-1.0 / d, MU / d))

    def model(x, lab_b):
        assert lab_b.shape == (x.shape[0],) and lab_b.dtype == torch.float32
        p, q = ab[lab.index(float(lab_b[0]))]
        return p * x + q
    return model


# measured on a B200: device vs fp64 oracle max |dx| <= 1.9e-6 (VE order 3, 40 steps; VP <= 1.4e-6)
GAUSS_TOL = 1e-5


@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("order", [1, 2, 3])
def test_gaussian_data_foreign_path_matches_oracle(kind, order):
    spec = O.SDESpec(kind)
    shape = [4, 3, 16, 16]
    x_T = torch.linspace(-1.7, 1.7, 4 * 3 * 16 * 16).view(shape)
    scale = spec.sigma_max if kind == "ve" else 1.0
    for steps in (10, 20, 40):
        s = _sampler(kind, steps=steps, order=order)
        grid = s.timesteps()
        got = _state(s.sample(_gauss_device_model(kind, grid), shape, device=DEV, noise=x_T[None])[-1])
        ref, _, _ = SO.solve(SO.gaussian_model(spec, MU, SD, grid), x_T.double() * scale, spec, grid, order)
        exact = SO.gaussian_exact(spec, MU, SD, x_T.double() * scale, grid[0], grid[-1])
        d_dev, d_orc = float((got - exact).abs().max()), float((ref - exact).abs().max())
        print(f"gaussian {kind} order {order} steps {steps}: device err {d_dev:.3e}, oracle err {d_orc:.3e}, "
              f"device vs oracle {float((got - ref).abs().max()):.2e}")
        assert float((got - ref).abs().max()) <= GAUSS_TOL
        assert abs(d_dev - d_orc) <= GAUSS_TOL


# ---- 3. SDE-DPM-Solver++ with Philox noise ---------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("order", [1, 2])
def test_sde_philox_moments_and_reproducibility(kind, order):
    spec = O.SDESpec(kind)
    shape = [256, 3, 32, 32]                  # 786432 independent elements
    s = _sampler(kind, steps=10, order=order, algorithm_type="sde-dpmsolver++")
    grid = s.timesteps()
    model = _gauss_device_model(kind, grid)
    s.seed = SEED
    a = _state(s.sample(model, shape, device=DEV)[-1])
    b = _state(s.sample(model, shape, device=DEV)[-1])
    assert torch.equal(a, b)
    s.seed = SEED + 1
    c = _state(s.sample(model, shape, device=DEV)[-1])
    assert not torch.equal(a, c)
    # x_T ~ N(0, scale^2) from Philox; the output is affine in x_T plus independent Gaussian noise
    scale = spec.sigma_max if kind == "ve" else 1.0
    m0, sd = SO.sde_output_moments(spec, MU, SD, 0.0, grid, order)
    m1, _ = SO.sde_output_moments(spec, MU, SD, 1.0, grid, order)
    mean, std = m0, math.sqrt(((m1 - m0) * scale) ** 2 + sd ** 2)
    n = a.numel()
    for x in (a, c):
        zm = (float(x.mean()) - mean) / (std / math.sqrt(n))
        zs = (float(x.std()) - std) / (std / math.sqrt(2 * n))
        print(f"{kind} sde order {order}: mean {float(x.mean()):.5f} (exact {mean:.5f}, {zm:+.2f} SE), std {float(x.std()):.5f} "
              f"(exact {std:.5f}, {zs:+.2f} SE)")
        assert abs(zm) <= 5 and abs(zs) <= 5


# ---- 4. native loops against the oracle over ref_port's U-Net ----------------------------------------------------------------
# measured on a B200: tiny / tiny_cls fp32 U-Net vs the oracle over ref_port's U-Net, rel-L2 <= 1.2e-6 (VE sde-dpmsolver++ 2M;
# deterministic <= 7.9e-7); guidance <= 1.5e-6
REAL_TOL = 1e-5


def _injected(shape, steps, seed):
    return torch.randn([1 + steps] + list(shape), generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("name", ["tiny", "tiny_cls"])
@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("algorithm,order", [("dpmsolver++", 1), ("dpmsolver++", 2), ("dpmsolver++", 3), ("sde-dpmsolver++", 1),
                                             ("sde-dpmsolver++", 2)])
def test_native_loop_matches_oracle(name, kind, algorithm, order):
    cfg, size, b = CFGS[name]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = [b, cfg["channels"], size, size]
    spec = O.SDESpec(kind)
    steps = 12
    noise = _injected(shape, steps, 9)
    model, omodel = u, O.make_model(sd, cfg)
    if cfg.get("num_classes") is not None:
        classes = torch.tensor([1, 7][:b])
        model = functools.partial(u.forward, classes=classes.to(DEV))
        omodel = functools.partial(omodel, classes=classes)
    s = _sampler(kind, steps=steps, order=order, algorithm_type=algorithm)
    imgs, nfe = s.sample(model, shape, device=DEV, noise=noise, return_nfe=True)
    assert nfe == steps
    scale = spec.sigma_max if kind == "ve" else 1.0
    zs = None if algorithm == "dpmsolver++" else list(noise[1:])
    ref, _, _ = SO.solve(lambda x, t: omodel(x.float(), t).double(), noise[0].double() * scale, spec, s.timesteps(), order, zs)
    err = rel_l2(_state(imgs[-1]), ref)
    print(f"{name} {kind} {algorithm} order {order}: rel-L2 vs oracle {err:.2e}")
    assert err <= REAL_TOL


@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("algorithm", ["dpmsolver++", "sde-dpmsolver++"])
def test_graph_plain_and_foreign_paths_are_bit_identical(kind, algorithm):
    cfg, size, b = CFGS["tiny"]
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="fp32", engine="simt", device=DEV)
    shape = [b, 1, size, size]
    s = _sampler(kind, steps=10, order=2, algorithm_type=algorithm)
    s.seed = SEED
    graph = s.sample(u, shape, device=DEV)[-1]
    again = s.sample(u, shape, device=DEV)[-1]
    s.use_cuda_graph = False
    plain = s.sample(u, shape, device=DEV)[-1]
    foreign = s.sample(lambda x, t: u(x, t), shape, device=DEV)[-1]
    assert torch.isfinite(graph).all()
    assert torch.equal(graph, again) and torch.equal(graph, plain) and torch.equal(graph, foreign)
    # injected noise: native (plain launches with the host step) == foreign
    noise = _injected(shape, 10, 4)
    assert torch.equal(s.sample(u, shape, device=DEV, noise=noise)[-1], s.sample(lambda x, t: u(x, t), shape, device=DEV, noise=noise)[-1])
    # x_T is the draw the PC sampler makes for the same seed: one step with a zero model maps it by (c_x + c_0 k_x)
    s1 = _sampler(kind, steps=1, order=1, algorithm_type=algorithm)
    s1.seed = SEED
    one = _state(s1.sample(lambda x, t: torch.zeros_like(x), shape, device=DEV)[-1])
    assert one.shape == tuple(shape) and torch.isfinite(one).all()
    if algorithm == "dpmsolver++":
        coef = s1.rows()[0][0].double()
        x_T = _randn_dev(shape, SEED).double().cpu() * (50.0 if kind == "ve" else 1.0)
        want = (coef[0] + coef[1] * coef[4]) * x_T           # m = k_x x_T, x' = c_x x_T + c_0 m
        assert float((one - want).abs().max()) <= 1e-6 * max(1.0, float(want.abs().max()))


@pytest.mark.parametrize("algorithm", ["dpmsolver++", "sde-dpmsolver++"])
def test_guidance_matches_two_oracle_calls(algorithm):
    cfg, size, b = CFGS["tiny_cls"]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = [b, 3, size, size]
    labels = torch.tensor([3, 7])
    w = 3.0

    def guided(x, t):
        ec = O.unet_forward(sd, cfg, x.float(), t.float(), labels)
        eu = O.unet_forward(sd, cfg, x.float(), t.float(), torch.full_like(labels, cfg["num_classes"]))
        return (eu + w * (ec - eu)).double()

    spec = O.SDESpec("vp")
    noise = _injected(shape, 12, 2)
    s = _sampler("vp", steps=12, order=2, algorithm_type=algorithm)
    s.guidance_scale = w
    img = s.sample(functools.partial(u.forward, classes=labels.to(DEV)), shape, device=DEV, noise=noise)[-1]
    ref, _, _ = SO.solve(guided, noise[0].double(), spec, s.timesteps(), 2, None if algorithm == "dpmsolver++" else list(noise[1:]))
    err = rel_l2(_state(img), ref)
    print(f"guidance w=3 {algorithm}: rel-L2 vs two oracle calls {err:.2e}")
    assert err <= REAL_TOL
    with pytest.raises(NotImplementedError):
        s.sample(lambda x, t: u(x, t, labels.to(DEV)), shape, device=DEV, noise=noise)


def test_argument_checks_on_the_device():
    cfg, size, b = CFGS["tiny"]
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="fp32", engine="simt", device=DEV)
    s = _sampler("vp", steps=4, algorithm_type="sde-dpmsolver++")
    with pytest.raises(ValueError):
        s.sample(u, [b, 3, size, size], device=DEV)                     # channels
    with pytest.raises(ValueError):
        s.sample(u, [b, 1, size, size // 2], device=DEV)                # not square
    with pytest.raises(ValueError):
        s.sample(u, [b, 1, size, size], device=DEV, noise=_injected([b, 1, size, size], 2, 0))     # needs 1 + steps tensors
    with pytest.raises(ValueError):
        s.sample(lambda x, t: torch.zeros(x.shape[0], 2, *x.shape[2:], device=x.device), [b, 1, size, size], device=DEV)
    lv, lsize, lb = CFGS["tiny_lv"]
    ul = make_unet(lv, O.random_state_dict(lv, seed=0), dtype="fp32", engine="simt", device=DEV)
    with pytest.raises(ValueError, match="output"):
        s.sample(ul, [lb, 3, lsize, lsize], device=DEV)


# ---- 5. against the probability-flow ODE solve ---------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["vp", "ve"])
def test_converges_to_the_probability_flow_solve(kind):
    cfg, size, b = CFGS["tiny"]
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="fp32", engine="simt", device=DEV)
    shape = [b, 1, size, size]
    x_T = _injected(shape, 0, 5)
    ode = M.ProbabilityFlowSampler(rtol=1e-6, atol=1e-6)
    ode.update_sde(M.VPSDE() if kind == "vp" else M.VESDE())
    ref = _state(ode.sample(u, shape, device=DEV, noise=x_T)[-1])
    dist = []
    for steps in (10, 20, 50, 100):
        s = _sampler(kind, steps=steps, order=3)
        dist.append(rel_l2(_state(s.sample(u, shape, device=DEV, noise=x_T)[-1]), ref))
    print(f"{kind}: rel-L2 to RK45 (rtol 1e-6, {ode.last_stats['nfev']} evaluations) at 10/20/50/100 steps: "
          + " ".join(f"{d:.2e}" for d in dist))
    assert all(a > b for a, b in zip(dist, dist[1:]))

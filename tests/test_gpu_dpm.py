"""DPMSolverDiffusion (DPM-Solver++ multistep, DMN_LOOP_DPMPP) on the GPU.

1. dmn_dpmpp_step against the fp64 update of tests/dpm_oracle.py for every order, ring slot and objective, with C- and 2C-channel
   model outputs; ring slots a step must not read hold NaN.
2. The Gaussian-data model (exact answer known) through the foreign-callable path: matches the fp64 oracle to fp32 rounding and
   converges at the solver's order.
3. Whole native loops with the U-Net's last 1x1 conv zeroed and a per-channel bias: the model output is that bias exactly, so each
   loop must match the fp64 oracle recursion to rounding (fp32 / simt and the production bf16 / tcgen05 graph at B = 256; graph,
   plain and injected-x_T modes; trajectory capture; a 2C-output learned-variance U-Net).
4. Real random weights against the oracle over oracle.ref_port's U-Net, classifier-free guidance, determinism, descriptor checks.

Gates: measured maxima on an NVIDIA B200 (1000 W power limit) beside each constant.
"""
import ctypes as C
import functools
import math

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from conftest import CFGS, make_unet, rel_l2
from oracle import ref_port as O
import dpm_oracle as D

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 0xDEADBEEF12345678
CFG2 = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
BIAS = torch.tensor([0.31, -0.17, 0.08, 0.6, -0.4, 0.2])


def _randn_dev(shape, seed, step=-1):
    out = torch.empty(shape, device=DEV)
    L.check(L.lib().dmn_randn(L.ptr(out), out.numel(), L.Rng(seed, 0), step, L.stream_ptr(DEV)), "dmn_randn")
    return out


def _state(img):
    """[-1, 1] state from the [0, 1] image the sampler returns."""
    return img.double() * 2.0 - 1.0


# ---- 1. the update kernel ----------------------------------------------------------------------------------------------------
# Gate in units of fp32 rounding: |x' - ref| <= KTOL * 2^-24 * (|c_x x| + |c_0| (|m| + |k_x x| + |k_m e|) + |c_1 m1| + |c_2 m2|)
# (the data prediction at high t cancels two terms of order 1e3) and |m - ref| <= KTOL * 2^-24 * (1 + |k_x x| + |k_m e|).
# measured on a B200: ratios <= 3.3 (update) and <= 0.63 (ring)
KTOL = 8.0
EPS32 = 2.0 ** -24


@pytest.mark.parametrize("objective", ["pred_noise", "pred_x0"])
@pytest.mark.parametrize("mo_ch", [3, 6])
def test_step_kernel_matches_fp64_update(objective, mo_ch):
    lib = L.lib()
    st = L.stream_ptr(DEV)
    sch = D.Schedule(1000, "linear")
    b, shape = 512, (512, 3, 32, 32)         # 196608 float4 > the 1184 x 256 grid: the grid-stride loop runs
    g = torch.Generator().manual_seed(1)
    worst = [0.0, 0.0]
    for order in (1, 2, 3):
        s = M.DPMSolverDiffusion(1000, "linear", objective=objective, steps=20, order=order)
        coef, _ = s._loop_tables(None, DEV)
        pairs, orders = s.timestep_pairs(), s.step_orders()
        steps = [order - 1, order, order + 1] + ([len(pairs) - 1] if order == 3 else [])   # every slot, and the last step
        for i in steps:
            o = orders[i]
            assert o == (order if i < len(pairs) - 1 else 1)
            t, tn = pairs[i]
            x = torch.randn(shape, generator=g) * 1.3
            mo = torch.randn(b, mo_ch, 32, 32, generator=g) * (2.5 if i % 2 else 0.6)     # odd steps: the clamp binds
            hist = [torch.rand(shape, generator=g) * 2 - 1 for _ in range(2)]               # m_{i-1}, m_{i-2}
            ring = torch.full((3,) + shape, float("nan"), device=DEV)                      # slots the step must not read stay NaN
            for k in range(1, o):
                ring[(i - k) % 3] = hist[k - 1].to(DEV)
            xd, mod = x.to(DEV), mo.to(DEV)
            L.check(lib.dmn_dpmpp_step(L.ptr(xd), L.ptr(mod), L.ptr(ring), L.ptr(xd), b, 3 * 1024, mo_ch * 1024, L.ptr(coef), None, i,
                                       st), "dmn_dpmpp_step")          # x_out aliases x
            torch.cuda.synchronize()
            m_ref = D.data_pred(sch, x.double(), mo.double(), t, objective)
            ts = [pairs[i - k][0] for k in range(o)]
            ref = D.update(sch, x.double(), [m_ref] + [h.double() for h in hist][:o - 1], ts, tn, o)
            got = xd.double().cpu()
            assert torch.isfinite(got).all(), (order, i)
            cx, c0, c1, c2 = (abs(float(v)) for v in coef[i, :4].cpu())
            xx, e = x.double(), mo[:, :3].double()
            sm = 0.0 if objective == "pred_x0" else sch.k_x[t] * xx.abs() + sch.k_m[t] * e.abs()
            bound = cx * xx.abs() + c0 * (m_ref.abs() + sm) + c1 * hist[0].double().abs() + c2 * hist[1].double().abs()
            err = float(((got - ref).abs() / (EPS32 * bound + 1e-30)).max())
            merr = float(((ring[i % 3].double().cpu() - m_ref).abs() / (EPS32 * (1.0 + sm))).max())
            worst = [max(worst[0], err), max(worst[1], merr)]
            assert err <= KTOL, (order, i, err)
            assert merr <= KTOL, (order, i, merr)
    print(f"dpmpp_step {objective} out_ch={mo_ch}: worst update error {worst[0]:.2f}, ring {worst[1]:.2f} (units of fp32 rounding)")


# ---- 2. Gaussian data through the foreign-callable path ------------------------------------------------------------------------
S2 = 0.25
# measured on a B200: device vs fp64 oracle max |dx| <= 1.5e-6
GAUSS_TOL = 1e-5


def _gauss_device_model(sch):
    tab = torch.tensor([D.gaussian_eps_coef(sch, S2, t) for t in range(sch.T)], dtype=torch.float32, device=DEV)
    return lambda x, t: tab[t].view(-1, 1, 1, 1) * x


@pytest.mark.parametrize("order", [1, 2, 3])
def test_gaussian_data_foreign_path_matches_oracle_and_converges(order):
    sch = D.Schedule(1000, "linear")
    shape = [4, 3, 16, 16]
    x_T = torch.linspace(-1.5, 1.5, 4 * 3 * 16 * 16).view(shape)
    model = _gauss_device_model(sch)
    errs = {}
    for k in (100, 200):
        s = M.DPMSolverDiffusion(1000, "linear", steps=k, order=order)
        got = _state(s.sample(model, shape, device=DEV, noise=x_T[None])[-1])
        ref, _, ms = D.solve(D.gaussian_model(sch, S2), x_T, sch, k, order)
        assert max(float(m.abs().max()) for m in ms) < 0.99      # the clamp never binds
        d = float((got - ref).abs().max())
        print(f"gaussian order {order} K={k}: device vs oracle max|dx| {d:.2e}")
        assert d <= GAUSS_TOL
        exact = D.gaussian_exact(sch, S2, x_T, O.ddim_pairs(1000, k)[0][0])
        errs[k] = float((got - exact).abs().max() / exact.abs().max())
    slope = math.log(errs[100] / errs[200]) / math.log(2.0)
    print(f"gaussian order {order}: device slope K=100->200 {slope:.3f}")
    lo, hi = {1: (0.9, 1.1), 2: (1.8, 2.3), 3: (2.6, 3.3)}[order]
    assert lo <= slope <= hi


# ---- 3. native loops with a constant model output ---------------------------------------------------------------------------------
def _const_unet(cfg, dtype, engine, out_ch=3):
    sd = O.random_state_dict(cfg, seed=0)
    sd["final_conv.3.weight"].zero_()
    sd["final_conv.3.bias"].copy_(BIAS[:out_ch])
    return make_unet(cfg, sd, dtype=dtype, engine=engine, device=DEV)


def _const_model(out_ch):
    return lambda x, t: BIAS[:out_ch].double().view(1, -1, 1, 1).expand(x.shape[0], -1, *x.shape[2:]).to(x.device)


# measured on a B200: every constant-output loop max|err| <= 4.8e-6 (bf16 B=256; fp32 / simt <= 4.1e-6)
LOOP_TOL = 2e-5


def _check_const_loop(s, u, shape, out_ch, mode, label):
    sch = D.Schedule(s.timesteps, s.schedule_name)
    if mode == "noise":
        x_T = torch.randn([3] + shape, generator=torch.Generator().manual_seed(4))     # extra elements are ignored
        imgs = s.sample(u, shape, device=DEV, noise=x_T)
        x_T = x_T[0].double()
    else:
        s.use_cuda_graph = mode == "graph"
        s.seed = SEED
        imgs = s.sample(u, shape, device=DEV)
        s.use_cuda_graph = True
        x_T = _randn_dev(shape, SEED).double().cpu()
    ref, states, _ = D.solve(_const_model(out_ch), x_T, sch, s.steps, s.order, s.objective)
    err = float((_state(imgs[-1]) - ref).abs().max())
    print(f"{label} {mode} order {s.order}: max|err| {err:.2e}")
    assert err <= LOOP_TOL * max(1.0, float(ref.abs().max()))
    return imgs, states + [ref]


@pytest.mark.parametrize("order", [1, 2, 3])
def test_const_output_loops_fp32(order):
    u = _const_unet(CFG2, "fp32", "simt")
    shape = [16, 3, 32, 32]
    for steps in (20, 10):
        s = M.DPMSolverDiffusion(1000, "linear", steps=steps, order=order)
        for mode in ("graph", "plain", "noise"):
            _check_const_loop(s, u, shape, 3, mode, f"fp32 K={steps}")
    # trajectory capture: states after steps 5, 10, 15 and the final one
    s = M.DPMSolverDiffusion(1000, "cosine", objective="pred_x0", steps=20, order=order)
    s.trajectory_every = 5
    imgs, states = _check_const_loop(s, u, shape, 3, "graph", "fp32 traj pred_x0")
    assert len(imgs) == 4
    for k, img in enumerate(imgs[:-1]):
        ref = states[5 * (k + 1)]
        assert float((_state(img) - ref).abs().max()) <= LOOP_TOL * max(1.0, float(ref.abs().max())), k
    # learned-variance U-Net: 2C outputs, the variance channels are ignored
    ul = _const_unet(dict(CFG2, learned_variance=True), "fp32", "simt", out_ch=6)
    s = M.DPMSolverDiffusion(1000, "cosine", steps=20, order=order)
    for mode in ("graph", "noise"):
        _check_const_loop(s, ul, shape, 6, mode, "learned-variance")


@pytest.mark.parametrize("order", [1, 2, 3])
def test_const_output_production_loop_bf16(order):
    u = _const_unet(CFG2, "bf16", "tcgen05")
    shape = [256, 3, 32, 32]
    s = M.DPMSolverDiffusion(1000, "linear", steps=20, order=order)
    for mode in ("graph", "plain", "noise"):
        _check_const_loop(s, u, shape, 3, mode, "bf16 B=256")
    s.trajectory_every = 10
    imgs, states = _check_const_loop(s, u, shape, 3, "graph", "bf16 B=256 traj")
    assert len(imgs) == 2 and float((_state(imgs[0]) - states[10]).abs().max()) <= LOOP_TOL * max(1.0, float(states[10].abs().max()))


# ---- 4. real weights -------------------------------------------------------------------------------------------------------
# measured on a B200: tiny fp32 U-Net vs the oracle over ref_port's U-Net, rel-L2 <= 1.6e-5 (pred_x0 order 3; pred_noise <= 2.3e-6)
REAL_TOL = 1e-4


@pytest.mark.parametrize("objective", ["pred_noise", "pred_x0"])
@pytest.mark.parametrize("order", [1, 2, 3])
def test_tiny_unet_matches_oracle(objective, order):
    cfg, size, b = CFGS["tiny"]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = [b, cfg["channels"], size, size]
    x_T = torch.randn([1] + shape, generator=torch.Generator().manual_seed(9))
    s = M.DPMSolverDiffusion(1000, "linear", objective=objective, steps=20, order=order)
    native = s.sample(u, shape, device=DEV, noise=x_T)[-1]
    ref, _, _ = D.solve(D.ref_unet_model(sd, cfg), x_T[0], D.Schedule(1000, "linear"), 20, order, objective)
    err = rel_l2(_state(native), ref)
    plugin = s.sample(lambda x, t: u(x, t), shape, device=DEV, noise=x_T)[-1]
    d = float((plugin - native).abs().max())
    print(f"tiny {objective} order {order}: rel-L2 vs oracle {err:.2e}; native vs plugin max|d| {d:.2e} (identical: {d == 0})")
    assert err <= REAL_TOL
    assert torch.equal(plugin, native)           # same kernels, same rows: bit-identical on a B200


def test_guidance_matches_two_reference_calls():
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

    x_T = torch.randn([1] + shape, generator=torch.Generator().manual_seed(2))
    s = M.DPMSolverDiffusion(1000, "linear", class_conditional=True, steps=20, order=2)
    s.guidance_scale = w
    img = s.sample(functools.partial(u.forward, classes=labels.to(DEV)), shape, device=DEV, noise=x_T)[-1]
    ref, _, _ = D.solve(guided, x_T[0], D.Schedule(1000, "linear"), 20, 2)
    err = float((img - (ref.float() + 1) * 0.5).abs().max())
    print(f"guidance w=3: max|err| on the [0,1] image {err:.2e}")
    assert err <= 2e-4                           # the gate of test_classifier_free_guidance_doubled_batch; measured on a B200 1.8e-5
    with pytest.raises(NotImplementedError):
        s.sample(lambda x, t: u(x, t), shape, device=DEV, noise=x_T)


def test_seeded_production_runs_are_bit_identical():
    u = make_unet(CFG2, O.random_state_dict(CFG2, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
    shape = [256, 3, 32, 32]
    s = M.DPMSolverDiffusion(1000, "linear", steps=20, order=3)
    s.seed = SEED
    a = s.sample(u, shape, device=DEV)[-1]
    b = s.sample(u, shape, device=DEV)[-1]
    s.use_cuda_graph = False
    c = s.sample(u, shape, device=DEV)[-1]
    assert torch.isfinite(a).all()
    assert torch.equal(a, b) and torch.equal(a, c)


def test_foreign_path_seeded_x_T():
    """Without noise the foreign-callable path draws x_T with dmn_randn(seed, step -1), the draw DDIM makes for that seed.  One step
    (t = 0 into alpha_bar = 1) with eps = 0 returns clamp(sqrt_recip_ac[0] * x_T)."""
    shape = [2, 3, 8, 8]
    s = M.DPMSolverDiffusion(1000, "linear", steps=1, order=3)
    s.seed = SEED
    one = _state(s.sample(lambda x, t: torch.zeros_like(x), shape, device=DEV)[-1])
    x_T = _randn_dev(shape, SEED).double().cpu()
    assert float((one - (x_T * float(s.sqrt_recip_alphas_cumprod[0])).clamp(-1, 1)).abs().max()) <= 1e-6


def test_foreign_model_output_shape_is_checked():
    s = M.DPMSolverDiffusion(100, "linear", steps=5)
    with pytest.raises(ValueError):
        s.sample(lambda x, t: torch.zeros(x.shape[0], 5, *x.shape[2:], device=x.device), [2, 3, 8, 8], device=DEV)


def _desc(kind, scratch, state, coef, batch):
    d = L.LoopDesc()
    d.kind, d.n_steps, d.batch, d.use_graph = kind, 4, batch, 1
    d.coef_dev, d.state_dev, d.scratch_dev, d.scratch_bytes = coef.data_ptr(), state.data_ptr(), scratch.data_ptr(), scratch.numel() * 4
    d.rng = L.Rng(1, 0)
    d.state_elems = state.numel()
    return d


def test_loop_descriptor_checks_with_a_bound_plan():
    lib = L.lib()
    b, c, hw = 2, 3, 16
    n = b * c * hw * hw
    coef = torch.zeros(4, L.COEF_STRIDE, device=DEV)
    state = torch.full((b, c, hw, hw), 0.25, device=DEV)
    for out_dim, ok in ((3, True), (6, True), (5, False)):
        u = M.Unet(None, dim=32, dim_mults=[1, 2], channels=c, out_dim=out_dim, use_convnext=False, compute_dtype="fp32",
                   conv_engine="simt").to(DEV)
        plan = u.plan(hw, b, DEV, time_rows=4)
        one = torch.zeros(1, device=DEV)
        need = lib.dmn_loop_scratch_bytes(plan.h, C.byref(_desc(L.LOOP_DPMPP, one, state, coef, b))) // 4
        no_ring = lib.dmn_loop_scratch_bytes(plan.h, C.byref(_desc(L.LOOP_DDIM, one, state, coef, b))) // 4
        assert no_ring + 3 * n <= need
        st = L.stream_ptr(DEV)
        for floats, fits in ((need, True), (need - 4, False), (no_ring, False)):
            scratch = torch.zeros(floats, device=DEV)
            d = _desc(L.LOOP_DPMPP, scratch, state, coef, b)
            if ok and fits:
                continue                 # accepted: the loop tests above run this layout
            rc = lib.dmn_sample_loop(plan.h, C.byref(d), st)
            torch.cuda.synchronize()
            assert rc == -1, (out_dim, floats)
            assert torch.equal(state, torch.full_like(state, 0.25)) and not scratch.any()     # nothing was launched
        # the new kind is counted like the other single-update loops
        d = _desc(L.LOOP_DPMPP, torch.zeros(1, device=DEV), state, coef, b)
        d2 = _desc(L.LOOP_DDIM, torch.zeros(1, device=DEV), state, coef, b)
        assert lib.dmn_loop_launches_per_step(plan.h, C.byref(d)) == lib.dmn_loop_launches_per_step(plan.h, C.byref(d2))

"""RePaint inpainting (GaussianDiffusion.inpaint and its DDPM / learned-variance / DDIM subclasses) on the GPU.

1. dmn_inpaint_prepare against the fp64 formula with the host reference noise (tests/philox_ref.py) for mask 0, 1 and fractional, with
   and without a jump; the exact cases are checked bit for bit.
2. Whole native loops with the U-Net's last 1x1 conv zeroed and a per-channel bias (the model output is that bias exactly) against
   the fp64 event recursion of tests/inpaint_oracle.py: DDPM (production bf16 graph at B = 256 with the fused tail, fp32), learned
   variance, DDIM eta = 0 and 0.5, each without and with resampling jumps.  The recursion is fed the device's own draws (pinned to the
   host reference by 1. and tests/test_gpu_philox.py): DDIM with eta = 0 is a deterministic map whose slope is up to
   sqrt(abar_0 / abar_T) ~ 150 where the x0 clamp does not bind, so the fast-math departure of a draw (about 1e-4 at most) would dominate.
3. The tiny fp32 U-Net with random weights against the recursion over oracle.ref_port's U-Net, the plain-callable path, guidance.
4. Output properties (exact known pixels, all-zero mask == sample(), all-one mask == x_known) and run modes (graph == plain launches
   == second graph run, batch-64 slice of a batch-256 run).

Gates: measured maxima on an NVIDIA B200 (1000 W power limit) beside each constant.
"""
import functools

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from conftest import CFGS, make_unet
from oracle import ref_port as O
import inpaint_oracle as IO
import philox_ref as P

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED = 0xDEADBEEF12345678
CFG2 = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
BIAS = torch.tensor([0.31, -0.17, 0.08, 0.6, -0.4, 0.2])


def _state(img):
    """[-1, 1] state from the [0, 1] image the sampler returns."""
    return img.double() * 2.0 - 1.0


def _known_and_mask(b, c, hw, seed=5):
    """A random known image and a mask with a kept left half, a generated right half and a fractional column between them."""
    known = torch.rand(b, c, hw, hw, generator=torch.Generator().manual_seed(seed)) * 2 - 1
    mask = torch.zeros(1, 1, hw, hw)
    mask[..., : hw // 2] = 1.0
    mask[..., hw // 2] = 0.375
    return known, mask


# ---- 1. the prepare kernel -----------------------------------------------------------------------------------------------------
# the noise of the kernel departs from the host reference by its fast-math intrinsics (<= 3.5e-5 on a B200, tests/test_gpu_philox.py);
# measured on a B200: max |x' - ref| <= 8.4e-5
KTOL = 2e-3


def test_prepare_kernel_matches_fp64_formula():
    lib, st, sid = L.lib(), L.stream_ptr(DEV), 1
    b, c, hw = 512, 3, 32                       # 196608 float4 > the 1184 x 256 grid: the grid-stride loop runs
    n = b * c * hw * hw
    g = torch.Generator().manual_seed(3)
    x = torch.randn(b, c, hw, hw, generator=g) * 1.3
    known = torch.rand(b, c, hw, hw, generator=g) * 2 - 1
    mask = torch.rand(b, c, hw, hw, generator=g)
    mask[mask < 0.3] = 0.0
    mask[mask > 0.7] = 1.0                      # about 30 % each of 0 and 1, the rest fractional
    rows = torch.tensor([[1.0, 0.0, 0.8, 0.6], [0.9, 0.43589, 0.3, 0.9539392], [1.0, 0.0, 1.0, 0.0], [0.7, 0.7141428, 1.0, 0.0]])
    coef = torch.zeros(4, L.COEF_STRIDE)
    coef[:, :4] = rows
    xd, kd, md, cd = x.to(DEV), known.to(DEV), mask.to(DEV), coef.to(DEV)
    worst = 0.0
    for step in range(4):
        out = torch.empty_like(xd)
        L.check(lib.dmn_inpaint_prepare(L.ptr(xd), L.ptr(kd), L.ptr(md), L.ptr(out), n, L.ptr(cd), None, step, L.Rng(SEED, sid), st),
                "dmn_inpaint_prepare")
        aj, gj, a0, s0 = (float(v) for v in coef[step, :4])
        z1 = torch.from_numpy(P.randn(SEED, sid, step, n, draw=1)).view_as(x) if s0 else 0.0
        z2 = torch.from_numpy(P.randn(SEED, sid, step, n, draw=2)).view_as(x) if gj else 0.0
        y = aj * x.double() + gj * z2
        ref = mask.double() * (a0 * known.double() + s0 * z1) + (1.0 - mask.double()) * y
        got = out.double().cpu()
        err = float((got - ref).abs().max())
        worst = max(worst, err)
        assert err <= KTOL, (step, err)
        keep, free = mask == 1.0, mask == 0.0
        if a0 == 1.0 and s0 == 0.0:             # m = 1, s_0 = 0: x_known exactly
            assert torch.equal(out.cpu()[keep], known[keep])
        if gj == 0.0:                           # m = 0 without a jump: x exactly
            assert torch.equal(out.cpu()[free], x[free])
    # in place (x_out aliases x) gives the same result as out of place
    out = torch.empty_like(xd)
    for dst in (out, xd):
        L.check(lib.dmn_inpaint_prepare(L.ptr(xd), L.ptr(kd), L.ptr(md), L.ptr(dst), n, L.ptr(cd), None, 1, L.Rng(SEED, sid), st))
    assert torch.equal(out, xd)
    print(f"inpaint_prepare: max|err| vs fp64 with reference noise {worst:.2e}")


# ---- 2. native loops with a constant model output ---------------------------------------------------------------------------------
def _device_draws(seed, shape):
    """draw(step, slot) -> fp64 CPU copy of the in-kernel normals the loop uses at that step: slot 0 (x_T at step -1, the update's
    draw) from dmn_randn, slots 1 / 2 from dmn_inpaint_prepare with the rows {0, 0, 0, 1} (mask 1: returns z1 exactly) and
    {0, 1, 0, 0} (mask 0: returns z2 exactly)."""
    lib, st = L.lib(), L.stream_ptr(DEV)
    n = 1
    for v in shape:
        n *= v
    zeros = torch.zeros(shape, device=DEV)
    masks = {1: torch.ones(shape, device=DEV), 2: zeros}
    rows = {1: [0.0, 0.0, 0.0, 1.0], 2: [0.0, 1.0, 0.0, 0.0]}
    tabs = {}

    def draw(step, slot):
        out = torch.empty(shape, device=DEV)
        if slot == 0:
            L.check(lib.dmn_randn(L.ptr(out), n, L.Rng(seed, 0), step, st), "dmn_randn")
        else:
            if slot not in tabs or tabs[slot].shape[0] <= step:
                tabs[slot] = torch.zeros(step + 256, L.COEF_STRIDE, device=DEV)
                tabs[slot][:, :4] = torch.tensor(rows[slot], device=DEV)
            L.check(lib.dmn_inpaint_prepare(L.ptr(zeros), L.ptr(zeros), L.ptr(masks[slot]), L.ptr(out), n, L.ptr(tabs[slot]), None, step,
                                            L.Rng(seed, 0), st), "dmn_inpaint_prepare")
        return out.double().cpu()

    return draw


def _const_unet(cfg, dtype, engine, out_ch=3):
    sd = O.random_state_dict(cfg, seed=0)
    sd["final_conv.3.weight"].zero_()
    sd["final_conv.3.bias"].copy_(BIAS[:out_ch])
    return make_unet(cfg, sd, dtype=dtype, engine=engine, device=DEV)


def _const_model(out_ch):
    return lambda x, t: BIAS[:out_ch].double().view(1, -1, 1, 1).expand(x.shape[0], -1, *x.shape[2:])


def _grid(s):
    if isinstance(s, M.GeneralizedGaussianDiffusion):
        return IO.Grid("ddim", s.timesteps, s.schedule_name, s.ddim_timesteps, s.eta, s.objective)
    return IO.Grid("learned" if isinstance(s, M.LearnedGaussianDiffusion) else "ddpm", s.timesteps, s.schedule_name,
                   objective=s.objective)


# measured on a B200: every constant-output loop max|err| / max(1, |x|max) <= 3.6e-6 (DDIM eta = 0; bf16 B=256: 1.2e-6)
LOOP_TOL = 2e-5
NB = 8                   # samples compared with the recursion (the update is elementwise, so a batch prefix draws the same noise)


def _check_const_loop(s, u, shape, out_ch, jr, label, keep_every=0):
    b, c, hw = shape[0], shape[1], shape[2]
    known, mask = _known_and_mask(b, c, hw)
    s.seed = SEED
    s.trajectory_every = keep_every
    imgs = s.inpaint(u, known, mask, device=DEV, jump_length=jr[0], jump_n_sample=jr[1])
    s.trajectory_every = 0
    sub = (NB, c, hw, hw)
    draw = _device_draws(SEED, sub)
    grid = _grid(s)
    ts = IO.schedule(len(grid.g), *jr)
    ref, traj = IO.run(grid, _const_model(out_ch), draw(-1, 0), known[:NB], mask, ts, draw, keep_every)
    err = float((_state(imgs[-1][:NB]) - ref).abs().max()) / max(1.0, float(ref.abs().max()))
    print(f"{label} j,r={jr}: {len(IO.events(ts))} events, max|err| {err:.2e}")
    assert err <= LOOP_TOL
    kept = mask.expand_as(known) == 1.0
    assert torch.equal(imgs[-1][kept], ((known + 1) * 0.5)[kept])          # the known pixels exactly
    for k, xr in enumerate(traj):
        assert float((_state(imgs[k][:NB]) - xr).abs().max()) <= LOOP_TOL * max(1.0, float(xr.abs().max())), k
    return imgs


@pytest.mark.parametrize("jr", [(1, 1), (3, 3)])
def test_const_output_production_ddpm_loop_bf16(jr):
    u = _const_unet(CFG2, "bf16", "tcgen05")
    _check_const_loop(M.GaussianDiffusion(50, "linear"), u, [256, 3, 32, 32], 3, jr, "DDPM bf16 B=256")


@pytest.mark.parametrize("jr", [(1, 1), (3, 3)])
def test_const_output_loops_fp32(jr):
    u = _const_unet(CFG2, "fp32", "simt")
    shape = [16, 3, 32, 32]
    imgs = _check_const_loop(M.GaussianDiffusion(50, "linear"), u, shape, 3, jr, "DDPM fp32", keep_every=20)
    assert len(imgs) == 1 + len(IO.events(IO.schedule(50, *jr))) // 20
    _check_const_loop(M.GaussianDiffusion(50, "cosine", objective="pred_x0"), u, shape, 3, jr, "DDPM fp32 pred_x0")
    ul = _const_unet(dict(CFG2, learned_variance=True), "fp32", "simt", out_ch=6)
    _check_const_loop(M.LearnedGaussianDiffusion(50, "cosine"), ul, shape, 6, jr, "learned variance")
    for eta in (0.0, 0.5):
        _check_const_loop(M.GeneralizedGaussianDiffusion(1000, "linear", eta=eta, ddim_timesteps=50), u, shape, 3, jr, f"DDIM eta={eta}")


# ---- 3. real weights -------------------------------------------------------------------------------------------------------
# the gate of tests/test_gpu_philox.py::test_seeded_ddpm_loop_matches_oracle on the [0, 1] image; measured on a B200 <= 1.9e-6
REAL_TOL = 2e-4


@pytest.mark.parametrize("kind", ["ddpm", "ddim"])
@pytest.mark.parametrize("jr", [(1, 1), (2, 3)])
def test_tiny_unet_matches_oracle(kind, jr):
    cfg, size, b = CFGS["tiny"]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = (b, cfg["channels"], size, size)
    known, mask = _known_and_mask(*shape[:3], seed=8)
    s = M.GaussianDiffusion(20, "linear") if kind == "ddpm" else M.GeneralizedGaussianDiffusion(100, "linear", eta=0.5, ddim_timesteps=20)
    s.seed = SEED
    native = s.inpaint(u, known, mask, device=DEV, jump_length=jr[0], jump_n_sample=jr[1])[-1]
    draw = _device_draws(SEED, shape)
    grid = _grid(s)
    ref, _ = IO.run(grid, IO.ref_unet_model(sd, cfg), draw(-1, 0), known, mask, IO.schedule(len(grid.g), *jr), draw)
    err = float((native - (ref.float() + 1) * 0.5).abs().max())
    plugin = s.inpaint(lambda x, t: u(x, t), known, mask, device=DEV, jump_length=jr[0], jump_n_sample=jr[1])[-1]
    print(f"tiny {kind} j,r={jr}: max|err| on the [0,1] image {err:.2e}; plugin identical: {torch.equal(plugin, native)}")
    assert err <= REAL_TOL
    assert torch.equal(plugin, native)           # same kernels, rows and step words


def test_guidance_matches_two_reference_calls():
    cfg, size, b = CFGS["tiny_cls"]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = (b, 3, size, size)
    labels = torch.tensor([3, 7])
    w = 3.0

    def guided(x, t):
        ec = O.unet_forward(sd, cfg, x.float(), t.float(), labels)
        eu = O.unet_forward(sd, cfg, x.float(), t.float(), torch.full_like(labels, cfg["num_classes"]))
        return (eu + w * (ec - eu)).double()

    known, mask = _known_and_mask(*shape[:3], seed=9)
    s = M.GaussianDiffusion(20, "linear", class_conditional=True)
    s.seed, s.guidance_scale = SEED, w
    img = s.inpaint(functools.partial(u.forward, classes=labels.to(DEV)), known, mask, device=DEV, jump_length=2, jump_n_sample=2)[-1]
    draw = _device_draws(SEED, shape)
    ref, _ = IO.run(_grid(s), guided, draw(-1, 0), known, mask, IO.schedule(20, 2, 2), draw)
    err = float((img - (ref.float() + 1) * 0.5).abs().max())
    print(f"guidance w=3: max|err| on the [0,1] image {err:.2e}")
    assert err <= 2e-4                           # the gate of the other guidance tests; measured on a B200 1.3e-6
    with pytest.raises(NotImplementedError):
        s.inpaint(lambda x, t: u(x, t), known, mask, device=DEV)


# ---- 4. output properties and run modes ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def prod_unet():
    return make_unet(CFG2, O.random_state_dict(CFG2, seed=0), dtype="bf16", engine="tcgen05", device=DEV)


def test_mask_extremes(prod_unet):
    shape = [256, 3, 32, 32]
    known, _ = _known_and_mask(256, 3, 32)
    s = M.GaussianDiffusion(20, "linear")
    s.seed = SEED
    free = s.inpaint(prod_unet, known, torch.zeros(1), device=DEV)[-1]
    assert torch.equal(free, s.sample(prod_unet, shape, device=DEV)[-1])
    full = s.inpaint(prod_unet, known, torch.ones(1, 3, 1, 1), device=DEV, jump_length=2, jump_n_sample=2)[-1]
    assert torch.equal(full, (known + 1) * 0.5)
    # noise[0] is x_T and further elements are ignored
    x_T = torch.randn([3] + shape, generator=torch.Generator().manual_seed(4))
    a = s.inpaint(prod_unet, known, torch.zeros(1), device=DEV, noise=x_T)[-1]
    assert torch.equal(a, s.inpaint(prod_unet, known, torch.zeros(1), device=DEV, noise=x_T[:1])[-1])
    assert torch.isfinite(a).all() and not torch.equal(a, free)


def test_run_modes_are_bit_identical(prod_unet):
    known, mask = _known_and_mask(256, 3, 32)
    s = M.GaussianDiffusion(20, "linear")
    s.seed = SEED
    run = functools.partial(s.inpaint, prod_unet, known, mask, device=DEV, jump_length=2, jump_n_sample=2)
    a = run()[-1]
    b = run()[-1]
    plan = prod_unet.plan(32, 256, DEV)
    n_ev = len(IO.events(IO.schedule(20, 2, 2)))
    launches = plan.last_loop_launches
    s.use_cuda_graph = False
    c = run()[-1]
    s.use_cuda_graph = True
    assert torch.isfinite(a).all()
    assert torch.equal(a, b) and torch.equal(a, c)
    s.sample(prod_unet, [256, 3, 32, 32], device=DEV)
    assert launches == (plan.last_loop_launches // 20 + 1) * n_ev + 1      # one prepare per event + the final composite
    d = M.GaussianDiffusion(20, "linear")
    d.seed = SEED
    e = d.inpaint(prod_unet, known[:64], mask, device=DEV, jump_length=2, jump_n_sample=2)[-1]
    diff = float((a[:64] - e).abs().max())
    print(f"batch-64 slice of a batch-256 inpaint: max|d| {diff:.2e}")
    assert diff <= 1e-6

"""The seeded mode (noise=None: x_T and every step's z drawn in-kernel by Philox) against the host reference tests/philox_ref.py.

1. dmn_randn bit layout: every element of a >= 2^22-float buffer (the grid-stride loop runs) against the float64 reference, for
   keys with a nonzero high seed word, stream ids >= 2^32 and steps up to 2^20.
2. Box-Muller edge quads (u at 1, at 1 - 2^-24, the angle at 2 pi, the largest radius found) stay finite and accurate.
3. Every update kernel's in-kernel draw (z_dev = NULL) against its fp64 formula with the reference z.
4. Whole seeded loops against an exact fp64 recursion: with the U-Net's last 1x1 conv zeroed and a per-channel bias, the model output
   is that bias exactly, so each loop is an affine-plus-clamp recursion whose only randomness is the reference noise.  This pins the
   device step counter (coefficient row, step word), the fused DDPM tail's quad mapping and the rank stream.
5. Seeded loops on the tiny fp32 U-Nets against the CPU oracle fed the reference noise, which also pins the time-table row.

Gates: measured maxima on an NVIDIA B200 (1000 W power limit) beside each constant.  The edge-quad search meets u == 1, u == 1 - 2^-24
and the angle 2 pi; the B200 draws no NaN there (0 non-finite values in 2.7e8 draws), so Box-Muller needs no clamp.
"""
import os

import numpy as np
import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from diffusion_model_nemo_b200.modules import _runtime as R
from conftest import CFGS, make_unet
from oracle import ref_port as O
import philox_ref as P

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEED_HI = 0xDEADBEEF12345678            # a seed with a nonzero high word, like draw_seed() returns
LOG_ERR = 2.0 ** -21.41                 # documented absolute error of __logf on [0.5, 2] (CUDA C Programming Guide, intrinsics)


def _randn_dev(n, seed, sid, step):
    out = torch.empty(n, device=DEV)
    L.check(L.lib().dmn_randn(L.ptr(out), n, L.Rng(seed, sid), step, L.stream_ptr(DEV)), "dmn_randn")
    return out


def _check_normals(got, ref, u_even):
    """got float32 [n] (device), ref float64 [n] (host), u_even float32 [n/2] radius uniforms -> (max |dz|, max radius excess)."""
    g = got.double().cpu().numpy()
    assert np.isfinite(g).all()
    dz = float(np.abs(g - ref).max())
    pairs = g.reshape(-1, 2)
    r2_ref = -2.0 * np.log(u_even.astype(np.float64))
    excess = np.abs((pairs ** 2).sum(1) - r2_ref) - 1e-6 * r2_ref
    return dz, float(excess.max())


# ---- 1. dmn_randn against the reference, whole buffer ---------------------------------------------------------------------
# measured on a B200: max |dz| <= 2.2e-4 (gate 1e-3), max radius excess over 1e-6 r^2 <= 1.35e-7 (gate 2 * 2^-21.41 = 7.2e-7)
@pytest.mark.parametrize("seed", [1234, SEED_HI, 2 ** 62 - 1])
@pytest.mark.parametrize("sid", [0, 3, 2 ** 32 + 5])
def test_randn_matches_host_reference(seed, sid):
    n = 1 << 22                         # n / 4 quads > the 1184 x 256 grid cap
    worst = [0.0, -1.0]
    for step in (-1, 0, 999, 1 << 20):
        got = _randn_dev(n, seed, sid, step)
        r = P.raw_quads(seed, sid, P.step_word(step), np.arange(n // 4))
        ref = P.box_muller(P.uniforms(r)).reshape(-1)
        dz, ex = _check_normals(got, ref, P.uniforms(r)[:, 0::2].reshape(-1))
        worst = [max(worst[0], dz), max(worst[1], ex)]
        assert dz <= 1e-3, (seed, sid, step, dz)
        assert ex <= 2 * LOG_ERR, (seed, sid, step, ex)
    print(f"randn seed={seed:#x} sid={sid:#x}: max|dz|={worst[0]:.3e} radius excess={worst[1]:.3e}")


def test_randn_keys_and_streams_are_distinct():
    """Each half of the key, the folded stream id and the step word change the draw (guards against a dropped word)."""
    n = 1 << 12
    base = _randn_dev(n, SEED_HI, 2 ** 32 + 5, 3)
    for seed, sid, step in ((SEED_HI & 0xFFFFFFFF, 2 ** 32 + 5, 3), (SEED_HI, 5, 3), (SEED_HI, 2 ** 32 + 5, 2), (SEED_HI ^ (1 << 40), 2 ** 32 + 5, 3)):
        assert not torch.equal(base, _randn_dev(n, seed, sid, step)), (seed, sid, step)


# ---- 2. Box-Muller edge quads ------------------------------------------------------------------------------------------------
def _edge_quads(seed, sid, word, n_quads=1 << 26, chunk=1 << 22):
    """Quad indices below n_quads whose uniforms sit at the edges of Box-Muller: r.x / r.z giving u == 1, u == 1 - 2^-24 or u within
    2^-21 of 1; r.y / r.w giving the angle 2 pi; and the smallest r.x / r.z found (the largest radius)."""
    hits, best = {}, (1 << 33, -1)
    one, below = np.float32(1.0), np.float32(1.0 - 2.0 ** -24)
    for q0 in range(0, n_quads, chunk):
        r = P.raw_quads(seed, sid, word, np.arange(q0, q0 + chunk))
        u = P.uniforms(r)
        for j in (0, 2):
            for tag, m in (("u=1", u[:, j] == one), ("u=1-2^-24", u[:, j] == below),
                           ("u>1-2^-21", (u[:, j] < below) & (u[:, j] >= np.float32(1.0 - 2.0 ** -21)))):
                hits.setdefault(tag, []).extend((q0 + np.nonzero(m)[0]).tolist())
            i = int(np.argmin(r[:, j]))
            if int(r[i, j]) < best[0]:
                best = (int(r[i, j]), q0 + i)
        for j in (1, 3):
            hits.setdefault("angle=2pi", []).extend((q0 + np.nonzero(u[:, j] == one)[0]).tolist())
    hits["max radius"] = [best[1]]
    return hits


def test_box_muller_edge_quads():
    seed, sid, step = 1234, 0, -1
    hits = _edge_quads(seed, sid, P.step_word(step))
    for tag in ("u=1", "u=1-2^-24", "u>1-2^-21", "angle=2pi"):
        assert hits[tag], tag                      # the search is big enough to meet every edge at this key
    quads = np.array(sorted({q for v in hits.values() for q in v}))
    n = 4 * (int(quads.max()) + 1)                 # <= 2^28 floats = 1 GiB
    got = _randn_dev(n, seed, sid, step)
    n_bad = int((~torch.isfinite(got)).sum())
    sel = got.view(-1, 4)[torch.from_numpy(quads).to(DEV)].reshape(-1)
    del got
    r = P.raw_quads(seed, sid, P.step_word(step), quads)
    dz, ex = _check_normals(sel, P.box_muller(P.uniforms(r)).reshape(-1), P.uniforms(r)[:, 0::2].reshape(-1))
    print(f"edge quads: {dict((k, len(v)) for k, v in hits.items())}, non-finite in {n} draws: {n_bad}, "
          f"max|dz|={dz:.3e} radius excess={ex:.3e}")
    assert n_bad == 0
    assert dz <= 1e-3 and ex <= 2 * LOG_ERR


# ---- 3. update kernels, in-kernel draw against fp64 formulas -------------------------------------------------------------------
B, C, HW = 256, 3, 32
CHW = C * HW * HW
N_EL = B * CHW


def _z_ref(seed, sid, step, draw, n=N_EL):
    return torch.from_numpy(P.randn(seed, sid, step, n, draw)).reshape(-1, C, HW, HW)


def _coef_table(seed, rows=1000, lo=0.5, hi=1.5):
    g = torch.Generator().manual_seed(seed)
    return lo + (hi - lo) * torch.rand(rows, L.COEF_STRIDE, generator=g)


def _rnd(*shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def _close(got, ref, tol, what):
    err = float((got.double().cpu() - ref).abs().max())
    print(f"{what}: max|err|={err:.3e} (gate {tol:.1e})")
    assert err <= tol, (what, err)


STEPS = (0, 1, 999)
KTOL = 2e-3        # the 1e-3 noise gate times coefficients <= 1.5, plus fp32 rounding; measured on a B200 <= 3.5e-5


def test_ddpm_learned_ddim_kernels_draw_reference_noise():
    lib, st, sid = L.lib(), L.stream_ptr(DEV), 2
    x, e, v = _rnd(B, C, HW, HW, seed=1), _rnd(B, C, HW, HW, seed=2), _rnd(B, C, HW, HW, seed=3).clamp(-1, 1)
    xd, ed = x.to(DEV), e.to(DEV)
    mo = torch.cat([e, v], 1).contiguous()
    mod = mo.to(DEV)
    tab = _coef_table(0)
    tab[:, 0] = 1.0 + tab[:, 0]                    # x0 = c0 x - c1 eps reaches the clamp for part of the batch
    tab[:, 5] = 0.0
    tlearn = _coef_table(1)
    tlearn[:, 5], tlearn[:, 6] = -4.0 + tlearn[:, 5], -1.0 - tlearn[:, 6]
    tddim = _coef_table(2)
    tddim[:, 5] = 0.0
    out = torch.empty_like(xd)
    tabd, tlearnd = tab.to(DEV), tlearn.to(DEV)
    for step in STEPS:
        z = _z_ref(SEED_HI, sid, step, 0)
        c = tab[step].double()
        ref = c[2] * (c[0] * x.double() - c[1] * e.double()).clamp(-1, 1) + c[3] * x.double() + c[4] * z
        L.check(lib.dmn_ddpm_step(L.ptr(xd), L.ptr(ed), None, L.ptr(out), N_EL, L.ptr(tabd), None, step, L.Rng(SEED_HI, sid), st))
        _close(out, ref, KTOL, f"ddpm step {step}")
        c = tlearn[step].double()
        frac = (v.double() + 1) * 0.5
        lv = frac * c[6] + (1 - frac) * c[5]
        ref = c[2] * (c[0] * x.double() - c[1] * e.double()).clamp(-1, 1) + c[3] * x.double() + c[4] * torch.exp(0.5 * lv) * z
        L.check(lib.dmn_learned_step(L.ptr(xd), L.ptr(mod), None, L.ptr(out), B, CHW, L.ptr(tlearnd), None, step,
                                     L.Rng(SEED_HI, sid), st))
        _close(out, ref, KTOL, f"learned step {step}")
        for k1 in (0.0, None):                     # k1 == 0 is DDIM with eta = 0: deterministic, no draw
            t = tddim.clone()
            if k1 is not None:
                t[:, 3] = k1
            c, td = t[step].double(), t.to(DEV)
            x0 = ((x.double() - e.double() * c[0]) / c[1]).clamp(-1, 1)
            ref = c[2] * x0 + c[3] * (z if k1 is None else 0) + c[4] * e.double()
            L.check(lib.dmn_ddim_step(L.ptr(xd), L.ptr(ed), None, L.ptr(out), N_EL, L.ptr(td), None, step, L.Rng(SEED_HI, sid), st))
            _close(out, ref, KTOL if k1 is None else 1e-5, f"ddim k1={k1} step {step}")


def test_pc_and_bpd_kernels_draw_reference_noise():
    lib, st, sid = L.lib(), L.stream_ptr(DEV), 0
    x, mo, x0 = _rnd(B, C, HW, HW, seed=4), _rnd(B, C, HW, HW, seed=5), _rnd(B, C, HW, HW, seed=6).clamp(-1, 1)
    xd, mod, x0d = x.to(DEV), mo.to(DEV), x0.to(DEV)
    out, mean = torch.empty_like(xd), torch.empty_like(xd)
    taff, tlan, tbpd = _coef_table(3), _coef_table(4), _coef_table(5)
    scratch = torch.empty(2 * B + 2, device=DEV)   # include/dmn_b200.h: 2*batch + 2 floats
    snr = 0.16
    taffd, tland, tbpdd = taff.to(DEV), tlan.to(DEV), tbpd.to(DEV)
    for step in STEPS:
        c = taff[step].double()
        z7 = _z_ref(SEED_HI, sid, step, 7)
        m_ref = c[0] * x.double() + c[1] * mo.double()
        L.check(lib.dmn_affine_noise_step(L.ptr(xd), L.ptr(mod), None, L.ptr(out), L.ptr(mean), N_EL, L.ptr(taffd), None, step,
                                          L.Rng(SEED_HI, sid), st))
        _close(mean, m_ref, 1e-5, f"affine mean step {step}")
        _close(out, m_ref + c[2] * z7, KTOL, f"affine step {step} (draw 7)")
        # Langevin: the norms kernel and the update kernel must draw the same z (draw 0)
        z0 = _z_ref(SEED_HI, sid, step, 0)
        c = tlan[step].double()
        g = c[0] * mo.double()
        ratio = snr * z0.flatten(1).norm(dim=1).mean() / g.flatten(1).norm(dim=1).mean()
        ss = ratio ** 2 * 2 * c[1]
        m_ref = x.double() + ss * g
        runs = []
        for _ in range(3):
            L.check(lib.dmn_langevin_step(L.ptr(xd), L.ptr(mod), None, L.ptr(out), L.ptr(mean), B, CHW, snr, L.ptr(tland), None,
                                          step, L.ptr(scratch), L.Rng(SEED_HI, sid), st))
            runs.append(out.clone())
        assert all(torch.equal(runs[0], r) for r in runs[1:]), "Langevin step is not bit-reproducible"
        _close(mean, m_ref, 1e-5 * max(1.0, float(m_ref.abs().max())), f"langevin mean step {step}")
        _close(out, m_ref + torch.sqrt(2 * ss) * z0, KTOL, f"langevin step {step}")
        c = tbpd[step].double()
        L.check(lib.dmn_bpd_qsample(L.ptr(x0d), None, L.ptr(out), N_EL, L.ptr(tbpdd), None, step, L.Rng(SEED_HI, sid), st))
        _close(out, c[6] * x0.double() + c[7] * z0, KTOL, f"bpd q_sample step {step}")


# ---- 4. seeded loops against an exact recursion --------------------------------------------------------------------------------
CFG2 = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
BIAS = torch.tensor([0.31, -0.17, 0.08, 0.6, -0.4, 0.2])     # per output channel (learned variance uses all 6)


def _const_unet(cfg, dtype, engine, out_ch=3):
    """A U-Net whose output is exactly BIAS per channel: the last 1x1 conv's weight is zero."""
    sd = O.random_state_dict(cfg, seed=0)
    sd["final_conv.3.weight"].zero_()
    sd["final_conv.3.bias"].copy_(BIAS[:out_ch])
    return make_unet(cfg, sd, dtype=dtype, engine=engine, device=DEV)


@pytest.fixture
def loop_tables(monkeypatch):
    """Records the coefficient tables every native loop is run with (the fp32 rows the kernels index)."""
    seen = []
    real = R.run_native_loop

    def spy(unet, **kw):
        seen.append(kw)
        kw["result"] = real(unet, **kw)
        return kw["result"]

    monkeypatch.setattr(R, "run_native_loop", spy)
    return seen


def _eps(out_ch=3):
    return BIAS[:out_ch].double().to(DEV).view(1, -1, 1, 1)


def _ddpm_ref(coef, x, seed, sid, n_steps, kind="ddpm", keep=0, z_of=None):
    """fp64 replay of the DDPM / learned / DDIM update with the constant model output.  z_s = dmn_randn(step = s) (pinned to the
    host reference by test_randn_matches_host_reference).  Returns (final, [state after step k*keep - 1 ...])."""
    coef = coef.double()
    e = _eps(6 if kind == "learned" else 3)
    traj = []
    for s in range(n_steps):
        c = coef[s]
        z = (z_of(s) if z_of else _randn_dev(x.numel(), seed, sid, s).double().view_as(x))
        if kind == "ddim":
            x0 = ((x - e * c[0]) / c[1]).clamp(-1, 1)
            x = c[2] * x0 + c[3] * z + c[4] * e
        else:
            x0 = (c[0] * x - c[1] * e[:, :3]).clamp(-1, 1)
            mean = c[2] * x0 + c[3] * x
            if kind == "learned":
                frac = (e[:, 3:] + 1) * 0.5
                x = mean + c[4] * torch.exp(0.5 * (frac * c[6] + (1 - frac) * c[5])) * z
            else:
                x = mean + c[4] * z
        if keep and (s + 1) % keep == 0:
            traj.append(x)
    return x, traj


def _img_err(img, x):
    return float((img.double().to(DEV) - (x + 1) * 0.5).abs().max())


# measured on a B200: production DDPM loop max|err| <= 2.5e-6, fp32 / foreign / learned / DDIM loops <= 9.5e-7
LOOP_TOL = 2e-5
STEP_TOL = 4e-6    # one step from the device's own previous state; measured on a B200 <= 3.5e-7


@pytest.mark.parametrize("traj_every", [0, 100])
def test_seeded_ddpm_production_loop_matches_recursion(loop_tables, traj_every):
    """cfg2, bf16 / tcgen05, B = 256, CUDA graph, seed above 2^32: the fused final_conv + DDPM tail (counter advanced in the tail
    without a trajectory; tail, trajectory copy and a separate counter kernel with one)."""
    u = _const_unet(CFG2, "bf16", "tcgen05")
    s = M.GaussianDiffusion(1000, "linear")
    s.seed, s.trajectory_every = SEED_HI, traj_every
    shape = [B, C, HW, HW]
    for rank in (0, 3):
        os.environ["RANK"] = str(rank)
        try:
            imgs = s.sample(u, shape, device=DEV)
        finally:
            os.environ.pop("RANK")
        coef = loop_tables[-1]["coef"]
        x = _randn_dev(N_EL, SEED_HI, rank, -1).double().view(*shape)
        ref, traj = _ddpm_ref(coef, x, SEED_HI, rank, 1000, keep=traj_every)
        err = _img_err(imgs[-1], ref)
        print(f"production DDPM rank {rank} traj_every={traj_every}: final max|err|={err:.3e}")
        assert err <= LOOP_TOL * max(1.0, float(ref.abs().max()))
        if traj_every:
            assert len(imgs) == 10
            for k, (img, xr) in enumerate(zip(imgs[:-1], traj)):
                assert _img_err(img, xr) <= LOOP_TOL * max(1.0, float(xr.abs().max())), (rank, (k + 1) * traj_every)


def test_seeded_ddpm_step_by_step(loop_tables):
    """T = 50 with every state kept: each step is replayed from the device's previous state, so a wrong coefficient row, step word or
    quad shows up at the first step it happens."""
    u = _const_unet(CFG2, "bf16", "tcgen05")
    s = M.GaussianDiffusion(50, "linear")
    s.seed = SEED_HI
    shape = [64, C, HW, HW]
    n = 64 * CHW
    s.trajectory_every = 1
    s.sample(u, shape, device=DEV)
    kw = loop_tables[-1]
    traj = kw["result"].traj
    prev = _randn_dev(n, SEED_HI, 0, -1).double().view(*shape)
    coef = kw["coef"].double()
    worst = 0.0
    for st in range(50):
        ref, _ = _ddpm_ref(coef[st:st + 1], prev, SEED_HI, 0, 1, z_of=lambda _s: _randn_dev(n, SEED_HI, 0, st).double().view(*shape))
        err = float((traj[st].double() - ref).abs().max())
        worst = max(worst, err)
        assert err <= STEP_TOL * max(1.0, float(ref.abs().max())), f"first wrong step: {st} (max|err| {err:.3e})"
        prev = traj[st].double()
    print(f"step-by-step DDPM T=50: worst one-step max|err|={worst:.3e}")


def test_seeded_other_ddpm_paths_match_recursion(loop_tables):
    """fp32 / simt (unfused ddpm_step_kernel), the foreign-callable path (model called per step, same step words), learned variance
    and DDIM with eta = 0.5."""
    shape = [16, C, HW, HW]
    n = 16 * CHW
    u = _const_unet(CFG2, "fp32", "simt")
    s = M.GaussianDiffusion(100, "linear")
    s.seed = SEED_HI
    x = _randn_dev(n, SEED_HI, 0, -1).double().view(*shape)
    img = s.sample(u, shape, device=DEV)[-1]
    coef = loop_tables[-1]["coef"]
    ref, _ = _ddpm_ref(coef, x, SEED_HI, 0, 100)
    tol = LOOP_TOL * max(1.0, float(ref.abs().max()))
    err = _img_err(img, ref)
    print(f"fp32/simt DDPM: {err:.3e}")
    assert err <= tol
    img = s.sample(lambda xx, tt: u(xx, tt), shape, device=DEV)[-1]
    err = _img_err(img, ref)
    print(f"foreign-callable DDPM: {err:.3e}")
    assert err <= tol
    ul = _const_unet(dict(CFG2, learned_variance=True), "fp32", "simt", out_ch=6)
    sl = M.LearnedGaussianDiffusion(100, "cosine")
    sl.seed = SEED_HI
    img = sl.sample(ul, shape, device=DEV)[-1]
    ref, _ = _ddpm_ref(loop_tables[-1]["coef"], x, SEED_HI, 0, 100, kind="learned")
    err = _img_err(img, ref)
    print(f"learned-variance loop: {err:.3e}")
    assert err <= LOOP_TOL * max(1.0, float(ref.abs().max()))
    d = M.GeneralizedGaussianDiffusion(1000, "linear", eta=0.5, ddim_timesteps=50)
    d.seed = SEED_HI
    img = d.sample(u, shape, device=DEV)[-1]
    kw = loop_tables[-1]
    ref, _ = _ddpm_ref(kw["coef"], x, SEED_HI, 0, int(kw["times"].shape[0]), kind="ddim")
    err = _img_err(img, ref)
    print(f"DDIM eta=0.5 loop: {err:.3e}")
    assert err <= LOOP_TOL * max(1.0, float(ref.abs().max()))


def _pc_ref(kw, x, seed, sid):
    """fp64 replay of the PC loop with the constant model output and the host reference noise (draws k = 0..n_corr-1, then 7)."""
    coef, coef2 = kw["coef"].double(), None if kw.get("coef2") is None else kw["coef2"].double()
    mo = _eps(3)
    n_corr, snr = kw.get("n_corr", 0), kw.get("snr", 0.0)
    x_mean = x
    for i in range(int(kw["times"].shape[0])):
        for k in range(n_corr):
            z = torch.from_numpy(P.randn(seed, sid, i, x.numel(), draw=k)).to(DEV).view_as(x)
            c = coef2[i]
            g = (c[0] * mo).expand_as(x)
            ratio = snr * z.flatten(1).norm(dim=1).mean() / g.flatten(1).norm(dim=1).mean()
            ss = ratio ** 2 * 2 * c[1]
            x_mean = x + ss * g
            x = x_mean + torch.sqrt(2 * ss) * z
        c = coef[i]
        z = torch.from_numpy(P.randn(seed, sid, i, x.numel(), draw=7)).to(DEV).view_as(x)
        x_mean = c[0] * x + c[1] * mo
        x = x_mean + c[2] * z
    return x, x_mean


# measured on a B200: PC loops max|err| / max(1, |x|max) <= 5.3e-7 (the constant model output drives |x| to ~1e3)
PC_TOL = 5e-6


@pytest.mark.parametrize("kind", ["vp", "ve"])
@pytest.mark.parametrize("pc", [("reverse_diffusion", "langevin"), ("euler_maruyama", "none")])
def test_seeded_pc_loop_matches_recursion(loop_tables, kind, pc):
    cfg = dict(CFG2, groups=4)
    u = _const_unet(cfg, "bf16", "tcgen05")
    sde = M.VPSDE(0.1, 20.0, 40) if kind == "vp" else M.VESDE(0.01, 50.0, 40)
    shape = [8, C, HW, HW]
    s = M.PredictorCorrectorSampler(pc[0], pc[1], snr=0.16, n_steps=2, denoise=True)
    s.update_sde(sde)
    s.seed = SEED_HI
    img = s.sample(u, shape, device=DEV)[-1]
    kw = loop_tables[-1]
    x = torch.from_numpy(P.randn(SEED_HI, 0, -1, 8 * CHW)).to(DEV).view(*shape) * kw.get("init_scale", 1.0)
    _, ref = _pc_ref(kw, x, SEED_HI, 0)
    err = _img_err(img, ref)
    print(f"PC {kind} {pc}: max|err|={err:.3e}, |x|max={float(ref.abs().max()):.2f}")
    assert err <= PC_TOL * max(1.0, float(ref.abs().max()))


# ---- 5. seeded loops on the tiny fp32 U-Nets against the oracle fed the reference noise ---------------------------------------------
def _ref_draws(seed, sid, words):
    """draw(shape) for the oracle: the host reference noise of the given step words, in order."""
    it = iter(words)

    def draw(shape):
        n = int(np.prod(shape))
        step, dr = next(it)
        return torch.from_numpy(P.randn(seed, sid, step, n, draw=dr)).float().view(*shape)

    return draw


def test_seeded_ddpm_loop_matches_oracle():
    cfg, size, b = CFGS["tiny"]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = [b, cfg["channels"], size, size]
    s = M.GaussianDiffusion(20, "linear")
    s.seed = SEED_HI
    img = s.sample(u, shape, device=DEV)[-1]
    ref, _ = O.sample_ddpm(O.make_model(sd, cfg), shape, O.ddpm_tables(20, "linear"),
                           _ref_draws(SEED_HI, 0, [(-1, 0)] + [(i, 0) for i in range(20)]))
    err = float((img - (ref + 1) * 0.5).abs().max())
    print(f"seeded DDPM vs oracle: {err:.3e}")
    assert err <= 2e-4


@pytest.mark.parametrize("kind", ["vp", "ve"])
def test_seeded_pc_loop_matches_oracle(kind):
    cfg, size, b = CFGS["tiny_g4"]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    shape = [b, 3, size, size]
    N = 40
    s = M.PredictorCorrectorSampler("reverse_diffusion", "langevin", snr=0.16, n_steps=1, denoise=True)
    s.update_sde(M.VPSDE(0.1, 20.0, N) if kind == "vp" else M.VESDE(0.01, 50.0, N))
    s.seed = SEED_HI
    img = s.sample(u, shape, device=DEV)[-1]
    words = [(-1, 0)] + [w for i in range(N) for w in ((i, 0), (i, 7))]
    ref, _ = O.sample_pc(O.make_model(sd, cfg), shape, O.SDESpec(kind, N=N), _ref_draws(SEED_HI, 0, words),
                         "reverse_diffusion", "langevin", snr=0.16, n_steps=1, denoise=True)
    ref01 = (ref + 1) * 0.5
    err = float((img - ref01).abs().max())
    print(f"seeded PC {kind} vs oracle: {err:.3e}")
    assert err <= 5e-4 * max(1.0, float(ref01.abs().max()))

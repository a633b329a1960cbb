"""The GroupNorm finalize, the final projection and the fused final-conv + DDPM tail, element by element, at the shapes and grid
sizes the production plans launch them.

Every ResnetBlock ends in gn_finalize_kernel (SiLU(GroupNorm(h2)) + residual, plus the fixed-point statistics of its output for the
next PreNorm or the final GroupNorm), and every U-Net forward ends in final_proj*_kernel or, in the DDPM loop, final_proj_ddpm_kernel.
Each case runs the production dispatch through dmn_gn_finalize_forward / dmn_final_proj_forward with inputs that make a wrong row of
statistics visible: bf16 values with their own mean and scale per (sample, group), some groups at |mean| / std = 8 (where
E[x^2] - m^2 cancels), and input statistics handed in exactly in the engine's fixed-point format, so the mirror (tests/tail_ref.py)
reads what the kernel reads.  Per case:

  * gn_finalize: every stored element within the derived bound of the fp64 mirror; the kernel's integer output sums within their
    bound; two runs bit-identical;
  * projection: eps within the bound of the fp64 mirror (K = C fmaf chain + the propagated affine / SiLU error);
  * fused tail: x_{t-1} within the bound of the mirror (eps bound carried through c1 and c2, clamp-aware), with injected noise and with
    Philox noise from tests/philox_ref.py; and torch.equal to final_proj followed by dmn_ddpm_step on the same inputs;
  * the production handoff: gn_finalize with ogroups = G feeding the fused tail.

A coverage test walks the op tables of the production plans and requires a case for every finalize / projection key.
The references run on the GPU in float64.
"""

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200 import _lib as L
from conftest import make_unet
from gpu_helpers import final_proj_forward, gn_finalize_forward
from oracle import ref_port as O
import philox_ref as P
import tail_ref as T

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BF, F32 = L.ACT_BF16, L.ACT_F32


def _fin(tag, c, h, b, g, og, silu=1, res=True, act=BF):
    return (f"fin_{tag}_c{c}_{h}x{h}_g{g}_og{og}{'' if silu else '_nosilu'}{'' if res else '_nores'}{'_f32' if act == F32 else ''}"
            f"_b{b}", c, h, b, g, og, silu, res, act)


# (name, C, H, B, groups, ogroups, silu, residual, act): one case per finalize key of configs[1] / [2] / [3] (ResnetBlock ends:
# ogroups 0, 1 before a PreNorm, G before the final GroupNorm), at the plan's batch, plus the other instantiations and forms
_LEVELS = {"cfg1": (32, 256), "cfg2": (64, 128)}
FIN_CASES = []
for _tag, (_s, _b) in _LEVELS.items():
    for _c, _h in ((128, _s), (256, _s // 2), (256, _s // 4), (256, _s // 8), (128, _s // 2)):
        for _og in (0, 1):
            FIN_CASES.append(_fin(_tag, _c, _h, _b, 8, _og))
    FIN_CASES.append(_fin(_tag, 128, _s, _b, 8, 8))
for _c, _h in ((128, 32), (256, 16), (256, 8), (256, 4), (128, 16)):
    for _og in (0, 1):
        FIN_CASES.append(_fin("cfg3", _c, _h, 256, 4, _og))
FIN_CASES += [
    _fin("cfg3", 128, 32, 256, 4, 4),
    _fin("cfg1", 256, 4, 512, 8, 1),                  # the guidance-doubled batch: 512 images, one block each
    _fin("d32", 32, 28, 64, 8, 0),                    # gn_finalize<bf16, 4>: dim 32, C / G = 4, ragged 784-pixel maps
    _fin("d32", 32, 28, 64, 1, 0, silu=0),            # GroupNorm(1) + residual of the unfused 28x28 attention block
    _fin("d32", 32, 28, 64, 8, 8, res=False),
    _fin("f32", 128, 16, 8, 8, 8, act=F32),           # gn_finalize<float, 4>
    _fin("f32", 256, 8, 8, 8, 1, silu=0, act=F32),
]
FIN_BY_NAME = {c[0]: c for c in FIN_CASES}

# (name, C, H, B, groups, Cout, plain, act): final_proj_bf16_kernel<3 | 6 | 1>, the fp32 kernel, the plain 'conv_bn_act' form and the
# generic final_proj_kernel<bf16> (an out_dim without a staged instantiation)
PROJ_CASES = [
    ("proj_cfg1_c128_32x32_g8_o3_b256", 128, 32, 256, 8, 3, 0, BF),
    ("proj_cfg2_c128_64x64_g8_o6_b128", 128, 64, 128, 8, 6, 0, BF),
    ("proj_cfg3_c128_32x32_g4_o3_b256", 128, 32, 256, 4, 3, 0, BF),
    ("proj_d32_c32_28x28_g8_o1_b256", 32, 28, 256, 8, 1, 0, BF),
    ("proj_plain_c128_32x32_o3_b16", 128, 32, 16, 0, 3, 1, BF),
    ("proj_f32_c128_16x16_g8_o3_b8", 128, 16, 8, 8, 3, 0, F32),
    ("proj_generic_c64_16x16_g8_o4_b8", 64, 16, 8, 8, 4, 0, BF),
]
PROJ_BY_NAME = {c[0]: c for c in PROJ_CASES}

# (name, C, H, B, groups, Cout): final_proj_ddpm_kernel<3> at the benchmark shape and <1> at 28x28 (ragged last 128-pixel block)
TAIL_CASES = [
    ("tail_cfg1_c128_32x32_o3_b256", 128, 32, 256, 8, 3),
    ("tail_cfg3_c128_32x32_g4_o3_b256", 128, 32, 256, 4, 3),
    ("tail_d32_c32_28x28_o1_b256", 32, 28, 256, 8, 1),
]
TAIL_BY_NAME = {c[0]: c for c in TAIL_CASES}
T_STEPS = 1000
TS = [T_STEPS - 1, T_STEPS // 2, 1, 0]         # coefficient rows 0..3; row 4 = the t = T/2 row as pred_x0
SEED, SID = 1234, 5
RESULTS = {}        # case name -> (keys, slack)


def _g(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _grouped(b, c, hw, groups, seed, act):
    """Activations [B][C][HW] with a scale 0.5 .. 2 and a mean of -8 .. 8 scales per (sample, group)."""
    g = _g(seed)
    gi = torch.arange(c, device=DEV) // (c // groups)
    bi = torch.arange(b, device=DEV)[:, None]
    scale = 2.0 ** (((bi * 5 + gi[None] * 3) % 9).float() / 4 - 1)
    mean = scale * (((bi * 7 + gi[None]) % 9).float() - 4) * 2
    v = torch.randn(b, c, hw, device=DEV, generator=g) * scale[:, :, None] + mean[:, :, None]
    return T.bf16(v) if act == BF else v


def _affine(c, seed):
    g = _g(seed)
    return 1 + 0.1 * torch.randn(c, device=DEV, generator=g), 0.1 * torch.randn(c, device=DEV, generator=g)


def run_fin_case(case, seed=0):
    name, c, h, b, groups, og, silu, res, act = case
    hw = h * h
    raw = _grouped(b, c, hw, groups, seed, act)
    rs = (T.bf16(torch.randn(b, c, hw, device=DEV, generator=_g(seed + 1))) if act == BF else
          torch.randn(b, c, hw, device=DEV, generator=_g(seed + 1))) if res else None
    gamma, beta = _affine(c, seed + 2)
    stats = T.fixed_stats(raw, groups)
    y, ost = gn_finalize_forward(raw, stats, gamma, beta, res=rs, silu=bool(silu), ogroups=og, act=act)
    o, d, bound = T.finalize_ref(raw, rs, stats, groups, gamma, beta, bool(silu), act == BF)
    nv, ratio = T.check_bound(y, o, bound)
    assert nv == 0, f"{name}: {nv} elements over the bound (max err / bound {ratio:.3g})"
    slack = {"y": ratio}
    if og:
        _, bpi, per_thread, n_at = T.finalize_geometry(b, hw, c, groups, act == BF, og)
        S, Q, dS, dQ = T.out_stats_ref(o, d, og, per_thread, n_at)
        nv, rS, rQ = T.check_out_stats(ost, S, Q, dS, dQ)
        assert nv == 0, f"{name}: output statistics outside the bound (sums {rS:.3g}, squares {rQ:.3g} of the bound)"
        y2, ost2 = gn_finalize_forward(raw, stats, gamma, beta, res=rs, silu=bool(silu), ogroups=og, act=act)
        assert torch.equal(ost, ost2) and torch.equal(y, y2), f"{name}: two runs differ"
        slack.update(sums=rS, squares=rQ, blocks=bpi)
    return {("finalize", c, hw, groups, og, silu, int(res), act)}, slack


def _proj_inputs(c, h, b, groups, cout, act, seed):
    y = _grouped(b, c, h * h, max(groups, 1), seed, act)
    gamma, beta = _affine(c, seed + 1)
    g = _g(seed + 2)
    w = torch.randn(cout, c, device=DEV, generator=g) / c ** 0.5
    bias = 0.1 * torch.randn(cout, device=DEV, generator=g)
    stats = T.fixed_stats(y, groups) if groups else None
    return y, gamma, beta, w, bias, stats


def run_proj_case(case, seed=0):
    name, c, h, b, groups, cout, plain, act = case
    y, gamma, beta, w, bias, stats = _proj_inputs(c, h, b, groups, cout, act, seed)
    eps = final_proj_forward(y, w, bias, stats=stats, gamma=gamma, beta=beta, plain=bool(plain), act=act)
    staged = act == BF and c % 8 == 0 and cout in (1, 3, 6)      # final_proj_bf16_kernel (silu_fast); else final_proj_kernel (silu_f)
    r, bound = T.proj_ref(y, stats, groups, gamma, beta, w, bias, bool(plain), fast=staged)
    nv, ratio = T.check_bound(eps, r, bound)
    assert nv == 0, f"{name}: {nv} elements over the bound (max err / bound {ratio:.3g})"
    return {("finalproj", c, h * h, groups, cout, plain, act)}, {"eps": ratio}


def _coef_table():
    s = M.GaussianDiffusion(T_STEPS, "linear")
    ts = torch.tensor(TS + [T_STEPS // 2])
    tab = torch.stack([c.reshape(-1).float() for c in s._step_rows(ts)] +
                      [torch.zeros(len(ts))] * (L.COEF_STRIDE - 6), 1)
    tab[len(TS), 5] = 1.0
    return tab.to(DEV)


def _ddpm_step(x, eps, z, coef, step):
    out = torch.empty_like(x)
    lib = L.lib()
    with torch.cuda.device(DEV):
        L.check(lib.dmn_ddpm_step(L.ptr(x), L.ptr(eps), L.ptr(z), L.ptr(out), x.numel(), L.ptr(coef), None, step, L.Rng(SEED, SID),
                                  L.stream_ptr(DEV)), "dmn_ddpm_step")
    torch.cuda.synchronize()
    return out


def check_tail(name, y, stats, gamma, beta, w, bias, x, coef, groups, slack):
    """Every coefficient row, injected and Philox noise: x_{t-1} within the bound of the mirror and equal to the unfused path."""
    b, cout, hw = x.shape
    eps_r, e_eps = T.proj_ref(y, stats, groups, gamma, beta, w, bias, False, fast=True)
    eps_k = final_proj_forward(y, w, bias, stats=stats, gamma=gamma, beta=beta)
    zin = torch.randn(x.shape, device=DEV, generator=_g(99))
    for step in range(coef.shape[0]):
        row = coef[step].cpu()
        for noise in ("z", "philox"):
            z = zin if noise == "z" else None
            out = final_proj_forward(y, w, bias, stats=stats, gamma=gamma, beta=beta, x=x, coef=coef, step=step, z=z, rng=(SEED, SID))
            if noise == "z":
                zr, ez = zin, 0.0
            else:
                zr = torch.from_numpy(P.randn(SEED, SID, step, x.numel())).to(DEV).reshape(x.shape)
                ez = T.PHILOX_ABS
            o, eo = T.ddpm_ref(x, eps_r, e_eps, zr, ez, row)
            nv, ratio = T.check_bound(out, o, eo)
            assert nv == 0, f"{name} row {step} {noise}: {nv} elements over the bound (max err / bound {ratio:.3g})"
            slack[f"row{step}_{noise}"] = ratio
            ref = _ddpm_step(x, eps_k, z, coef, step)
            ndiff = int((out != ref).sum())
            assert ndiff == 0, f"{name} row {step} {noise}: the fused tail differs from final_proj + dmn_ddpm_step in {ndiff} elements"


def run_tail_case(case, seed=0):
    name, c, h, b, groups, cout = case
    y, gamma, beta, w, bias, stats = _proj_inputs(c, h, b, groups, cout, BF, seed)
    x = torch.randn(b, cout, h * h, device=DEV, generator=_g(seed + 3))
    slack = {}
    check_tail(name, y, stats, gamma, beta, w, bias, x, _coef_table(), groups, slack)
    return {("tail", c, h * h, groups, cout)}, slack


@pytest.mark.parametrize("name", [c[0] for c in FIN_CASES])
def test_finalize_case(name):
    RESULTS[name] = run_fin_case(FIN_BY_NAME[name])


@pytest.mark.parametrize("name", [c[0] for c in PROJ_CASES])
def test_final_proj_case(name):
    RESULTS[name] = run_proj_case(PROJ_BY_NAME[name])


@pytest.mark.parametrize("name", [c[0] for c in TAIL_CASES])
def test_fused_tail_case(name):
    RESULTS[name] = run_tail_case(TAIL_BY_NAME[name])


def test_production_handoff_finalize_to_fused_tail():
    """final_conv.0's gn_finalize with ogroups = G hands y and its fixed-point statistics to the fused tail (configs[1], B = 256)."""
    c, h, b, groups, cout = 128, 32, 256, 8, 3
    raw = _grouped(b, c, h * h, groups, 7, BF)
    rs = T.bf16(torch.randn(b, c, h * h, device=DEV, generator=_g(8)))
    g1, b1 = _affine(c, 9)
    stats = T.fixed_stats(raw, groups)
    y, ost = gn_finalize_forward(raw, stats, g1, b1, res=rs, silu=True, ogroups=groups)
    o, d, bound = T.finalize_ref(raw, rs, stats, groups, g1, b1, True, True)
    assert T.check_bound(y, o, bound)[0] == 0
    _, _, per_thread, n_at = T.finalize_geometry(b, h * h, c, groups, True, groups)
    assert T.check_out_stats(ost, *T.out_stats_ref(o, d, groups, per_thread, n_at))[0] == 0
    g2, b2 = _affine(c, 10)
    w = torch.randn(cout, c, device=DEV, generator=_g(11)) / c ** 0.5
    bias = 0.1 * torch.randn(cout, device=DEV, generator=_g(12))
    x = torch.randn(b, cout, h * h, device=DEV, generator=_g(13))
    slack = {}
    check_tail("handoff", y, ost, g2, b2, w, bias, x, _coef_table(), groups, slack)
    RESULTS["handoff"] = (set(), slack)


OP_FINALIZE, OP_FINALPROJ = 3, 6      # plan.cu OpKind


def _expected_tail_ops(cfg, size):
    """name -> key of every gn_finalize / final projection launch of the U-Net (plan.cu: resblock, attn_block, build), with the fused
    linear attention blocks (no attention finalize): ResnetBlock finalizes (C, HW, G, ogroups, silu 1, residual 1) and the tail
    (C, HW, G, out_dim, plain 0)."""
    G, dim = cfg["groups"], cfg["dim"]
    dims = [dim] + [dim * m for m in cfg["dim_mults"]]
    n = len(cfg["dim_mults"])
    hs = [size >> i for i in range(n)]
    fin = lambda c, h, og: ("finalize", c, h * h, G, og, 1, 1, BF)        # noqa: E731
    out = {}
    for i in range(n):
        out[f"downs.{i}.0.finalize"] = fin(dims[i + 1], hs[i], 0)
        out[f"downs.{i}.1.finalize"] = fin(dims[i + 1], hs[i], 1)
    out["mid_block1.finalize"] = fin(dims[n], hs[n - 1], 1)
    out["mid_block2.finalize"] = fin(dims[n], hs[n - 1], 0)
    for j in range(n - 1):
        lvl, hu = n - 1 - j, hs[n - 1] << j
        out[f"ups.{j}.0.finalize"] = fin(dims[lvl], hu, 0)
        out[f"ups.{j}.1.finalize"] = fin(dims[lvl], hu, 1)
    out["final_conv.0.finalize"] = fin(dim, size, G)
    cout = cfg["channels"] * (2 if cfg.get("learned_variance") else 1)
    out["final_conv.tail"] = ("finalproj", dim, size * size, G, cout, 0, BF)
    return out


def _bytes(key):
    """plan.cu dmn_plan_op_info, bf16 activations: gn_finalize reads raw and residual and writes y; the projection reads y, writes eps."""
    if key[0] == "finalize":
        return 2.0 * key[2] * key[1] * 3.0
    return 2.0 * key[2] * key[1] + 4.0 * key[2] * key[4]


def test_cases_cover_every_production_finalize_and_tail():
    """Every gn_finalize and final-projection launch of a production plan is named and sized as derived from its config, and every key
    is run by some case (the fused DDPM tail runs the configs[1] / [3] projection shape in the DDPM loop).  Prints the slack per case."""
    c1 = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
    plans = {"configs[1] B=256": (c1, 32, 256), "configs[1] B=512": (dict(c1, num_classes=10), 32, 512),
             "configs[2] B=128": (dict(c1, learned_variance=True), 64, 128), "configs[3] B=256": (dict(c1, groups=4), 32, 256)}
    need = {}
    for pname, (cfg, size, batch) in plans.items():
        u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
        ops = {o[0]: o for o in u.plan(size, batch, DEV).op_table() if o[1] in (OP_FINALIZE, OP_FINALPROJ)}
        expect = _expected_tail_ops(cfg, size)
        assert set(ops) == set(expect), (pname, sorted(set(ops) ^ set(expect)))
        for name, key in expect.items():
            assert ops[name][1] == (OP_FINALIZE if key[0] == "finalize" else OP_FINALPROJ), (pname, name)
            assert ops[name][4] == _bytes(key), (pname, name, ops[name][4], _bytes(key))
            need.setdefault(key, set()).add(pname)
            if key[0] == "finalproj" and key[4] == cfg["channels"]:          # the DDPM loop fuses this projection with the update
                need.setdefault(("tail", key[1], key[2], key[3], key[4]), set()).add(pname)
    runners = [(c, run_fin_case) for c in FIN_CASES] + [(c, run_proj_case) for c in PROJ_CASES] + [(c, run_tail_case) for c in TAIL_CASES]
    have = {}
    for case, run in runners:
        if case[0] not in RESULTS:
            RESULTS[case[0]] = run(case)
        for k in RESULTS[case[0]][0]:
            have.setdefault(k, case[0])
    print("\nproduction keys -> covering case:")
    missing = []
    for k, pl in sorted(need.items(), key=str):
        print(f"  {k} [{', '.join(sorted(pl))}] -> {have.get(k)}")
        if k not in have:
            missing.append(k)
    print("slack per case (max err / bound):")
    for n, (_, s) in RESULTS.items():
        print(f"  {n}: " + ", ".join(f"{a} {v:.3g}" for a, v in s.items()))
    assert not missing, f"production launches no case covers: {missing}"

"""Every production instantiation of the tcgen05 convolution engine, element by element, at the tile counts the sampler runs it.

The per-layer tests elsewhere use small batches: one tile per CTA, one accumulator per tile.  At the benchmark batch the engine runs
two 128-row accumulators per tile (mt = 2), mixed 256 / 128-row tiling, several tiles per CTA (both TMEM accumulator buffers and the
hand-over between tiles), 256-row windows across several small images, and the two-source (concat) operand of the up path.  Each case
below is one distinct conv launch of a production plan -- configs[1] (3x32x32, dim 128, mults 1,2,2,2, groups 8) at B = 256 and at
the guidance-doubled B = 512, configs[2] (64x64) at B = 128, the GroupNorm-4 convs of configs[3] at B = 256 -- plus ragged batches
that end in a partial 128-row tile.  Per case (tests/conv_ref.py):

  * probe weights: bit equality with the shifted input (every input channel, every tap, both concat sources); through the GroupNorm
    prologue the fp64 prologue bound instead, and exactly the bias wherever the tap reads padding;
  * random weights: the element bound against an fp64 convolution, and the share of elements that differ from bf16_RN(fp64);
  * GroupNorm output statistics against their derived bound, where the production conv has them;
  * the launch log (dmn_debug_conv_log) shows the tiling regime the case claims: (mt, mixed 256 / 128-row tiling, tiles > CTAs).

The reference runs on the GPU in float64.  Production defaults: no DMN_CONV_* switch is set.
"""
import math

import pytest
import torch

from diffusion_model_nemo_b200 import _lib as L
from conftest import make_unet
from gpu_helpers import conv_forward, conv_log
from oracle import ref_port as O
import conv_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# share of random-weight outputs allowed to differ from bf16_RN(fp64) with a plain operand: at most 2.5e-3 measured on a B200
# (DESIGN.md section 4), gated at four times that
FRAC_GATE = 0.01

# (name, mode, ksize, C1, C2, Cout, H, B, prologue GroupNorm groups (0: none), temb, out_groups, claimed (mt, mixed, tiles > CTAs))
# mode 0: 3x3 / 1x1 same, 1: k4s2 down, 2: transposed k4s2 up; C2 > 0: concat source (dmn_conv_forward_cat).  The claims follow
# fill_params' tiling arithmetic for 148 SMs.
CASES = [
    ("cfg1_l0_c3_b256", 0, 3, 128, 0, 128, 32, 256, 0, 0, 8, (2, True, True)),
    ("cfg1_l0_c3_pro_b256", 0, 3, 128, 0, 128, 32, 256, 8, 1, 8, (2, True, True)),
    ("cfg1_l0_down_b256", 1, 4, 128, 0, 128, 32, 256, 0, 0, 0, (2, False, True)),
    ("cfg1_l1_c3_in_b256", 0, 3, 128, 0, 256, 16, 256, 0, 0, 8, (2, False, True)),
    ("cfg1_l1_res_b256", 0, 1, 128, 0, 256, 16, 256, 0, 0, 0, (2, True, True)),
    ("cfg1_l1_c3_b256", 0, 3, 256, 0, 256, 16, 256, 0, 0, 8, (2, False, True)),
    ("cfg1_l1_c3_pro_b256", 0, 3, 256, 0, 256, 16, 256, 8, 1, 8, (2, False, True)),
    ("cfg1_l1_down_b256", 1, 4, 256, 0, 256, 16, 256, 0, 0, 0, (2, True, True)),
    ("cfg1_l2_c3_b256", 0, 3, 256, 0, 256, 8, 256, 0, 0, 8, (2, True, True)),
    ("cfg1_l2_c3_pro_b256", 0, 3, 256, 0, 256, 8, 256, 8, 1, 8, (2, True, True)),
    ("cfg1_l2_down_b256", 1, 4, 256, 0, 256, 8, 256, 0, 0, 0, (1, False, False)),
    ("cfg1_l3_c3_b256", 0, 3, 256, 0, 256, 4, 256, 0, 0, 8, (1, False, False)),
    ("cfg1_l3_c3_pro_b256", 0, 3, 256, 0, 256, 4, 256, 8, 1, 8, (1, False, False)),
    ("cfg1_u0_cat_b256", 0, 3, 256, 256, 256, 4, 256, 0, 0, 8, (1, False, False)),
    ("cfg1_u0_res_b256", 0, 1, 256, 256, 256, 4, 256, 0, 0, 0, (1, False, False)),
    ("cfg1_u0_up_b256", 2, 4, 256, 0, 256, 4, 256, 0, 0, 0, (2, True, True)),
    ("cfg1_u1_cat_b256", 0, 3, 256, 256, 256, 8, 256, 0, 0, 8, (2, True, True)),
    ("cfg1_u1_res_b256", 0, 1, 256, 256, 256, 8, 256, 0, 0, 0, (1, False, True)),
    ("cfg1_u1_up_b256", 2, 4, 256, 0, 256, 8, 256, 0, 0, 0, (2, True, True)),
    ("cfg1_u2_cat_b256", 0, 3, 256, 256, 128, 16, 256, 0, 0, 8, (2, False, True)),
    ("cfg1_u2_res_b256", 0, 1, 256, 256, 128, 16, 256, 0, 0, 0, (2, False, True)),
    ("cfg1_u2_c3_b256", 0, 3, 128, 0, 128, 16, 256, 0, 0, 8, (2, False, True)),
    ("cfg1_u2_c3_pro_b256", 0, 3, 128, 0, 128, 16, 256, 8, 1, 8, (2, False, True)),
    ("cfg1_u2_up_b256", 2, 4, 128, 0, 128, 16, 256, 0, 0, 0, (2, False, True)),
    ("cfg1_final_pro_b256", 0, 3, 128, 0, 128, 32, 256, 8, 0, 8, (2, True, True)),
    ("cfg1_l0_c3_b512", 0, 3, 128, 0, 128, 32, 512, 0, 0, 8, (2, False, True)),
    ("cfg1_l0_c3_pro_b512", 0, 3, 128, 0, 128, 32, 512, 8, 1, 8, (2, False, True)),
    ("cfg1_l0_down_b512", 1, 4, 128, 0, 128, 32, 512, 0, 0, 0, (2, False, True)),
    ("cfg1_l1_c3_in_b512", 0, 3, 128, 0, 256, 16, 512, 0, 0, 8, (2, False, True)),
    ("cfg1_l1_res_b512", 0, 1, 128, 0, 256, 16, 512, 0, 0, 0, (2, False, True)),
    ("cfg1_l1_c3_b512", 0, 3, 256, 0, 256, 16, 512, 0, 0, 8, (2, False, True)),
    ("cfg1_l1_c3_pro_b512", 0, 3, 256, 0, 256, 16, 512, 8, 1, 8, (2, False, True)),
    ("cfg1_l1_down_b512", 1, 4, 256, 0, 256, 16, 512, 0, 0, 0, (2, True, True)),
    ("cfg1_l2_c3_b512", 0, 3, 256, 0, 256, 8, 512, 0, 0, 8, (2, True, True)),
    ("cfg1_l2_c3_pro_b512", 0, 3, 256, 0, 256, 8, 512, 8, 1, 8, (2, True, True)),
    ("cfg1_l2_down_b512", 1, 4, 256, 0, 256, 8, 512, 0, 0, 0, (1, False, True)),
    ("cfg1_l3_c3_b512", 0, 3, 256, 0, 256, 4, 512, 0, 0, 8, (1, False, True)),
    ("cfg1_l3_c3_pro_b512", 0, 3, 256, 0, 256, 4, 512, 8, 1, 8, (1, False, True)),
    ("cfg1_u0_cat_b512", 0, 3, 256, 256, 256, 4, 512, 0, 0, 8, (1, False, True)),
    ("cfg1_u0_res_b512", 0, 1, 256, 256, 256, 4, 512, 0, 0, 0, (1, False, False)),
    ("cfg1_u0_up_b512", 2, 4, 256, 0, 256, 4, 512, 0, 0, 0, (2, False, True)),
    ("cfg1_u1_cat_b512", 0, 3, 256, 256, 256, 8, 512, 0, 0, 8, (2, True, True)),
    ("cfg1_u1_res_b512", 0, 1, 256, 256, 256, 8, 512, 0, 0, 0, (2, False, True)),
    ("cfg1_u1_up_b512", 2, 4, 256, 0, 256, 8, 512, 0, 0, 0, (2, False, True)),
    ("cfg1_u2_cat_b512", 0, 3, 256, 256, 128, 16, 512, 0, 0, 8, (2, False, True)),
    ("cfg1_u2_res_b512", 0, 1, 256, 256, 128, 16, 512, 0, 0, 0, (2, True, True)),
    ("cfg1_u2_c3_b512", 0, 3, 128, 0, 128, 16, 512, 0, 0, 8, (2, False, True)),
    ("cfg1_u2_c3_pro_b512", 0, 3, 128, 0, 128, 16, 512, 8, 1, 8, (2, False, True)),
    ("cfg1_u2_up_b512", 2, 4, 128, 0, 128, 16, 512, 0, 0, 0, (2, False, True)),
    ("cfg2_l0_c3_b128", 0, 3, 128, 0, 128, 64, 128, 0, 0, 8, (2, True, True)),
    ("cfg2_l0_c3_pro_b128", 0, 3, 128, 0, 128, 64, 128, 8, 1, 8, (2, True, True)),
    ("cfg2_l0_down_b128", 1, 4, 128, 0, 128, 64, 128, 0, 0, 0, (2, False, True)),
    ("cfg2_l1_c3_in_b128", 0, 3, 128, 0, 256, 32, 128, 0, 0, 8, (2, True, True)),
    ("cfg2_l1_res_b128", 0, 1, 128, 0, 256, 32, 128, 0, 0, 0, (2, False, True)),
    ("cfg2_l1_c3_b128", 0, 3, 256, 0, 256, 32, 128, 0, 0, 8, (2, True, True)),
    ("cfg2_l1_c3_pro_b128", 0, 3, 256, 0, 256, 32, 128, 8, 1, 8, (2, True, True)),
    ("cfg2_l1_down_b128", 1, 4, 256, 0, 256, 32, 128, 0, 0, 0, (2, False, True)),
    ("cfg2_l2_c3_b128", 0, 3, 256, 0, 256, 16, 128, 0, 0, 8, (2, False, True)),
    ("cfg2_l2_c3_pro_b128", 0, 3, 256, 0, 256, 16, 128, 8, 1, 8, (2, False, True)),
    ("cfg2_l2_down_b128", 1, 4, 256, 0, 256, 16, 128, 0, 0, 0, (1, False, True)),
    ("cfg2_l3_c3_b128", 0, 3, 256, 0, 256, 8, 128, 0, 0, 8, (1, False, True)),
    ("cfg2_l3_c3_pro_b128", 0, 3, 256, 0, 256, 8, 128, 8, 1, 8, (1, False, True)),
    ("cfg2_u0_cat_b128", 0, 3, 256, 256, 256, 8, 128, 0, 0, 8, (1, False, True)),
    ("cfg2_u0_res_b128", 0, 1, 256, 256, 256, 8, 128, 0, 0, 0, (1, False, False)),
    ("cfg2_u0_up_b128", 2, 4, 256, 0, 256, 8, 128, 0, 0, 0, (2, True, True)),
    ("cfg2_u1_cat_b128", 0, 3, 256, 256, 256, 16, 128, 0, 0, 8, (2, False, True)),
    ("cfg2_u1_res_b128", 0, 1, 256, 256, 256, 16, 128, 0, 0, 0, (2, False, True)),
    ("cfg2_u1_up_b128", 2, 4, 256, 0, 256, 16, 128, 0, 0, 0, (2, False, True)),
    ("cfg2_u2_cat_b128", 0, 3, 256, 256, 128, 32, 128, 0, 0, 8, (2, False, True)),
    ("cfg2_u2_res_b128", 0, 1, 256, 256, 128, 32, 128, 0, 0, 0, (2, True, True)),
    ("cfg2_u2_c3_b128", 0, 3, 128, 0, 128, 32, 128, 0, 0, 8, (2, False, True)),
    ("cfg2_u2_c3_pro_b128", 0, 3, 128, 0, 128, 32, 128, 8, 1, 8, (2, False, True)),
    ("cfg2_u2_up_b128", 2, 4, 128, 0, 128, 32, 128, 0, 0, 0, (2, False, True)),
    ("cfg3_l0_c3_b256", 0, 3, 128, 0, 128, 32, 256, 0, 0, 4, (2, True, True)),
    ("cfg3_l0_c3_pro_b256", 0, 3, 128, 0, 128, 32, 256, 4, 1, 4, (2, True, True)),
    ("cfg3_l1_c3_in_b256", 0, 3, 128, 0, 256, 16, 256, 0, 0, 4, (2, False, True)),
    ("cfg3_l1_c3_pro_b256", 0, 3, 256, 0, 256, 16, 256, 4, 1, 4, (2, False, True)),
    ("cfg3_l2_c3_pro_b256", 0, 3, 256, 0, 256, 8, 256, 4, 1, 4, (2, True, True)),
    ("cfg3_l3_c3_pro_b256", 0, 3, 256, 0, 256, 4, 256, 4, 1, 4, (1, False, False)),
    ("cfg3_u0_cat_b256", 0, 3, 256, 256, 256, 4, 256, 0, 0, 4, (1, False, False)),
    ("cfg3_u2_cat_b256", 0, 3, 256, 256, 128, 16, 256, 0, 0, 4, (2, False, True)),
    ("cfg3_u2_c3_pro_b256", 0, 3, 128, 0, 128, 16, 256, 4, 1, 4, (2, False, True)),
    ("rag_l0_c3_b37", 0, 3, 128, 0, 128, 32, 37, 0, 0, 8, (2, True, True)),
    ("rag_l0_c3_pro_b37", 0, 3, 128, 0, 128, 32, 37, 8, 1, 8, (2, True, True)),
    ("rag_l1_c3_b37", 0, 3, 256, 0, 256, 16, 37, 0, 0, 8, (1, False, True)),
    ("rag_l3_c3_pro_b37", 0, 3, 256, 0, 256, 4, 37, 8, 1, 8, (1, False, False)),
    ("rag_u0_cat_b37", 0, 3, 256, 256, 256, 4, 37, 0, 0, 8, (1, False, False)),
    ("rag_u2_up_b37", 2, 4, 128, 0, 128, 16, 37, 0, 0, 0, (2, True, True)),
    ("rag_l2_c3_b131", 0, 3, 256, 0, 256, 8, 131, 0, 0, 8, (1, False, True)),
    ("rag_u0_up_b131", 2, 4, 256, 0, 256, 4, 131, 0, 0, 0, (1, False, True)),
    ("rag_u1_up_b131", 2, 4, 256, 0, 256, 8, 131, 0, 0, 0, (2, True, True)),
    ("rag_u2_cat_b131", 0, 3, 256, 256, 128, 16, 131, 0, 0, 8, (2, False, False)),
    ("rag_l0_c3_b255", 0, 3, 128, 0, 128, 32, 255, 0, 0, 8, (2, True, True)),
    ("rag_l0_c3_pro_b255", 0, 3, 128, 0, 128, 32, 255, 8, 1, 8, (2, True, True)),
    ("rag_l1_down_b255", 1, 4, 256, 0, 256, 16, 255, 0, 0, 0, (2, True, True)),
    ("rag_l2_c3_pro_b255", 0, 3, 256, 0, 256, 8, 255, 8, 1, 8, (2, True, True)),
    ("rag_l3_c3_pro_b255", 0, 3, 256, 0, 256, 4, 255, 8, 1, 8, (1, False, False)),
    ("rag_u0_res_b255", 0, 1, 256, 256, 256, 4, 255, 0, 0, 0, (1, False, False)),
    ("rag_u0_up_b255", 2, 4, 256, 0, 256, 4, 255, 0, 0, 0, (2, True, True)),
    ("rag_u1_cat_b255", 0, 3, 256, 256, 256, 8, 255, 0, 0, 8, (2, True, True)),
    ("rag_u1_up_b255", 2, 4, 256, 0, 256, 8, 255, 0, 0, 0, (2, True, True)),
]
CASE_BY_NAME = {c[0]: c for c in CASES}
# the 7x7 stem (GEO_INIT, init_conv_tcgen05) has no layer entry point; it stays outside this coverage (class-embedding epilogue)
EXCLUDED_GEO = {3: "7x7 stem (GEO_INIT)"}
CASE_KEYS = {}      # case name -> set of launch keys it produced
SLACK = {}          # case name -> measured slack (printed by the coverage test)


def _g(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _key(rec):
    return (rec["name"], rec["mt"], rec["mixed"], rec["multi"])


def _inputs(case, seed):
    name, mode, k, c1, c2, cout, h, b, pg, temb, og, _ = case
    g = _g(seed)
    if pg:
        x = R.bf16(torch.randn(b, c1, h, h, device=DEV, generator=g) * 2 + 0.5)
    else:
        x = R.bf16(torch.randn(b, c1, h, h, device=DEV, generator=g))
    x2 = R.bf16(torch.randn(b, c2, h, h, device=DEV, generator=g)) if c2 else None
    bias = torch.randn(cout, device=DEV, generator=g) * 0.1
    gn = None
    te = None
    if pg:
        gn = (pg, 1 + 0.1 * torch.randn(c1, device=DEV, generator=g), 0.1 * torch.randn(c1, device=DEV, generator=g))
        if temb:
            te = torch.randn(b, c1, device=DEV, generator=g)
    return x, x2, bias, gn, te


def _conv(case, x, x2, w, bias, gn, te):
    name, mode, k, c1, c2, cout, h, b, pg, temb, og, _ = case
    conv_log()
    y, st = conv_forward(x, w, bias, mode=mode, ksize=k, gn=gn, silu=bool(pg), temb=te, out_groups=og, act=L.ACT_BF16,
                         engine=L.CONV_TCGEN05, x2=x2)
    recs = conv_log()
    assert len(recs) == 1, recs
    return y, st, recs[0]


def _check_regime(case, rec):
    name, mode, k, c1, c2, cout, h, b, pg, temb, og, (mt, mixed, multi) = case
    assert (rec["geo"], rec["ksize"], rec["C1"], rec["C2"], rec["Cout"], rec["H"], rec["B"]) == (mode, k, c1, c2, cout, h, b), rec
    assert (rec["mt"], rec["mixed"], rec["multi"]) == (mt, mixed, multi), (name, rec)
    if mixed:      # both tile sizes present: whole rounds of 256-row tiles, then 128-row tiles from row big_rows on
        assert rec["big_rows"] == 256 * rec["n_big_tiles"] // rec["n_tiles_n"] and rec["big_rows"] < rec["total_flat"]
    assert rec["atma"] == 1, f"{name}: the production shapes take the TMA operand feed"


def _prologue(x, gn, te):
    a, t, scale = R.prologue_ref(x, gn[0], gn[1], gn[2], te, silu=True)
    e = R.prologue_error(a, t, scale, te, silu=True)
    return a, e


def run_case(case, seed=0):
    name, mode, k, c1, c2, cout, h, b, pg, temb, og, _ = case
    cin, nt = c1 + c2, R.taps(mode, k)
    x, x2, bias, gn, te = _inputs(case, seed)
    keys, slack = set(), {}
    src = (x, x2) if c2 else x
    if pg:
        a, e = _prologue(x, gn, te)
    # ---- probes: every input channel (both sources) and every tap ----
    for j in range(R.probe_channels_count(cin, cout)):
        w = R.probe_weights(cin, cout, mode, k, j).to(DEV)
        y, st, rec = _conv(case, x, x2, w, bias, gn, te)
        _check_regime(case, rec)
        keys.add(_key(rec))
        if not pg:
            r0, _ = R.probe_ref(src, cin, cout, mode, k, j)
            exp = R.probe_expected(r0, bias)
            nbad, where = R.check_probe(y, exp)
            assert nbad == 0, f"{name} probe {j}: {nbad} elements differ, first at (b, o, y, x) {where}"
            r = r0 + bias.double()[None, :, None, None]
            delta = R.U32 * r.abs()
        else:
            a_s, pad = R.probe_ref(a, cin, cout, mode, k, j)
            e_s, _ = R.probe_ref(e, cin, cout, mode, k, j)
            r = a_s + bias.double()[None, :, None, None]
            bound = R.probe_prologue_bound(a_s, e_s, bias)
            err = (y.double() - r).abs()
            viol = (err > bound) & ~pad
            assert int(viol.sum()) == 0, f"{name} probe {j}: {int(viol.sum())} over the prologue bound, first {viol.nonzero()[:8].tolist()}"
            padv = R.probe_expected(torch.zeros_like(a_s), bias)
            npad = int((y.float() != padv.float())[pad].sum())
            assert npad == 0, f"{name} probe {j}: {npad} padding reads are not exactly the bias"
            slack["probe_pro"] = max(slack.get("probe_pro", 0.0), float((err / bound)[~pad].max()))
            delta = R.operand_bound(a_s, e_s) + R.U32 * r.abs()
        if og:
            nv, sm, sr = R.check_stats(st, r, delta, og)
            assert nv == 0, f"{name} probe {j}: statistics outside the bound (mean {sm:.3g}, rstd {sr:.3g} of the bound)"
            slack["stats_probe"] = max(slack.get("stats_probe", 0.0), sm, sr)
    # ---- random weights ----
    g = _g(seed + 1)
    wshape = (cin, cout, 4, 4) if mode == 2 else (cout, cin, k, k)
    w = R.bf16(torch.randn(*wshape, device=DEV, generator=g) / math.sqrt(cin * nt))
    y, st, rec = _conv(case, x, x2, w, bias, gn, te)
    _check_regime(case, rec)
    keys.add(_key(rec))
    opnd = a if pg else src
    r = R.conv_ref(opnd, w, bias, mode, k)
    rabs = R.conv_ref(R.cat_sources(opnd).abs() if not pg else a.abs(), w.abs(), None, mode, k)
    extra = R.K_SIGMA * R.prologue_sigma(R.operand_bound(a, e), w, mode, k) if pg else None
    bound = R.element_bound(r, rabs, cin * nt, extra)
    nv, ratio, frac = R.check_bound(y, r, bound)
    assert nv == 0, f"{name} random: {nv} elements over the bound (max err / bound {ratio:.3g})"
    slack["rand"], slack["frac"] = ratio, frac
    if not pg:
        assert frac <= FRAC_GATE, f"{name} random: {frac:.4f} of the elements differ from bf16_RN(fp64)"
    if og:
        delta = R.acc_delta(r, rabs, cin * nt) + (extra if pg else 0.0)
        nv, sm, sr = R.check_stats(st, r, delta, og)
        assert nv == 0, f"{name} random: statistics outside the bound (mean {sm:.3g}, rstd {sr:.3g} of the bound)"
        slack["stats"] = max(sm, sr)
    return keys, slack


@pytest.mark.parametrize("name", [c[0] for c in CASES])
def test_conv_tile_case(name):
    keys, slack = run_case(CASE_BY_NAME[name])
    CASE_KEYS[name] = keys
    SLACK[name] = slack


def _plan_keys(cfg, size, batch):
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="bf16", engine="tcgen05", device=DEV)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(batch, cfg["channels"], size, size, generator=g).to(DEV)
    t = torch.randint(0, 1000, (batch,), generator=g).to(DEV)
    conv_log()
    u(x, t)
    torch.cuda.synchronize()
    recs = conv_log()
    assert recs, "the plan launched no tcgen05 conv"
    return recs


def test_cases_cover_every_production_instantiation():
    """Every (kernel instantiation, mt, mixed tiling, several tiles per CTA) key that a plain forward of a production plan launches is
    launched by some case of CASES.  The SM count is the device's (the tiling rule depends on it)."""
    nsm = torch.cuda.get_device_properties(DEV).multi_processor_count
    c1 = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
    plans = {"configs[1] B=256": (c1, 32, 256), "configs[1] B=512": (c1, 32, 512),
             "configs[2] B=128": (dict(c1, learned_variance=True), 64, 128), "configs[3] B=256": (dict(c1, groups=4), 32, 256)}
    need = {}
    for pname, (cfg, size, batch) in plans.items():
        for rec in _plan_keys(cfg, size, batch):
            if rec["geo"] in EXCLUDED_GEO:
                need.setdefault(("excluded", EXCLUDED_GEO[rec["geo"]]), set()).add(pname)
                continue
            need.setdefault(_key(rec), set()).add(pname)
    have = {}
    for case in CASES:
        if case[0] not in CASE_KEYS:
            CASE_KEYS[case[0]], SLACK[case[0]] = run_case(case)
        for kk in CASE_KEYS[case[0]]:
            have.setdefault(kk, case[0])
    print(f"\n{nsm} SMs; production keys (kernel, mt, mixed, tiles > CTAs) -> covering case:")
    missing = []
    for kk, pl in sorted(need.items(), key=str):
        cov = "EXCLUDED" if kk[0] == "excluded" else have.get(kk)
        print(f"  {kk} [{', '.join(sorted(pl))}] -> {cov}")
        if cov is None:
            missing.append(kk)
    print("slack per case (max err / bound; fraction of elements != bf16_RN(fp64)):")
    for n, s in SLACK.items():
        print(f"  {n}: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(s.items())))
    regimes = {(c[11][0], c[11][1], c[11][2]) for c in CASES}
    assert (2, True, True) in regimes and any(c[4] and c[11][2] for c in CASES)
    assert not missing, f"production launches no case covers: {missing}"

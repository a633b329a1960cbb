"""The checkers of tests/tail_ref.py on the CPU: the stem probes cover every (input channel, ky, kx) tap, the mirrors accept the
correctly rounded results, and each checker rejects a small injected defect of the kind a kernel could have.  Each defect also
records whether the whole-U-Net gate (rel-L2 <= 2e-2 of the output) would accept it: the rel-L2 of the defect at the production
output size (B = 256; the defect's own elements exactly, the norm of the output scaled from the test tensor's rms to the production
element count)."""
import math

import pytest
import torch

import conv_ref as R
import tail_ref as T

GATE = 2e-2


def _rand(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


def _prod_rel_l2(delta, y, n_prod):
    """rel-L2 of the defect delta against an output of n_prod elements with y's rms."""
    return float(delta.double().norm() / (y.double().pow(2).mean().sqrt() * math.sqrt(n_prod)))


# ---- stem ----------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cin,cout", [(3, 128), (1, 32)])
def test_stem_probes_cover_every_tap_and_corner(cin, cout):
    seen = set()
    for j in range(R.probe_count(cin, cout, 0, 7)):
        tap, ci = R.probe_assign(cin, cout, 0, 7, j)
        seen |= set(zip(tap.tolist(), ci.tolist()))
    assert seen == {(t, c) for t in range(49) for c in range(cin)}
    assert {0, 6, 42, 48} <= {t for t, _ in seen}


def _stem_case(b=4, cin=3, cout=16, s=8, j=0):
    x = _rand(b, cin, s, s, seed=1).float()
    bias = (_rand(cout, seed=2) * 0.1).float()
    cls_w = _rand(11, cout, seed=3).float()
    rows = cls_w[torch.tensor([3, 7, 1, 10][:b])]
    w = R.probe_weights(cin, cout, 0, 7, j)
    xo, _ = T.stem_operands(x, w, True)
    exp = T.stem_epilogue(R.probe_ref(xo, cin, cout, 0, 7, j)[0], bias, rows, True)
    return x, xo, w, bias, rows, exp


def test_stem_probe_accepts_the_mirror_and_the_conv_reference():
    x, xo, w, bias, rows, exp = _stem_case()
    assert R.check_probe(exp.clone(), exp)[0] == 0
    acc = R.conv_ref(xo, w.double(), None, 0, 7)                  # exact: one product per output
    assert R.check_probe(T.stem_epilogue(acc, bias, rows, True), exp)[0] == 0


def test_stem_probe_rejects_a_tap_shifted_by_one_column():
    x, xo, w, bias, rows, exp = _stem_case()
    o = 5
    ci, ky, kx = (int(v) for v in (w[o] != 0).nonzero()[0])
    wb = w.clone()
    wb[o, ci, ky, kx] = 0
    wb[o, ci, ky, kx + 1 if kx < 6 else kx - 1] = 1
    bad = T.stem_epilogue(R.conv_ref(xo, wb.double(), None, 0, 7), bias, rows, True)
    n, _ = R.check_probe(bad, exp)
    assert n > 0
    # one output channel of the 128 reads its neighbour column (production: 128 channels over the test's positions)
    rel = _prod_rel_l2((bad - exp)[:, o], exp, 128 * exp[:, o].numel())
    assert rel > GATE             # a whole output channel moves: the rel-L2 gate rejects it (about 8e-2)


def test_stem_probe_rejects_a_leak_across_the_shared_zero_rows():
    """The stacked images share 3 zero rows; a stem whose top taps read the previous image's bottom rows instead."""
    x, xo, w, bias, rows, exp = _stem_case()
    b, cin, s, _ = xo.shape
    tall = xo.permute(1, 0, 2, 3).reshape(1, cin, b * s, s)       # images stacked with no zero rows between them
    acc = R.conv_ref(tall, w.double(), None, 0, 7).reshape(-1, b, s, s).permute(1, 0, 2, 3)
    bad = T.stem_epilogue(acc, bias, rows, True)
    n, where = R.check_probe(bad, exp)
    assert n > 0 and all(p[2] in (0, 1, 2, s - 3, s - 2, s - 1) for p in where)
    # every probe channel whose tap row reads across the boundary: rows 0..2 and S-3..S-1 of each 8-row test image, 6 of 32 rows at
    # 32 x 32 -- the rel-L2 gate rejects this one (about 0.2 at 32 x 32)
    assert _prod_rel_l2(bad - exp, exp, exp.numel()) * math.sqrt(8 / 32) > GATE


def test_stem_probe_rejects_the_class_row_of_the_wrong_sample():
    x, xo, w, bias, rows, exp = _stem_case()
    bad = T.stem_epilogue(R.probe_ref(xo, 3, 16, 0, 7, 0)[0], bias, rows.roll(1, 0), True)
    assert R.check_probe(bad, exp)[0] > 0
    one = exp.clone()
    one[1] = bad[1]                                                  # only sample 1 takes sample 0's row
    assert R.check_probe(one, exp)[0] > 0
    # one sample of 256 with the wrong class row (rows of unit scale against outputs of unit scale): the gate rejects it (0.07)
    assert _prod_rel_l2(one - exp, exp, exp[0].numel() * 256) > GATE


def test_stem_random_bound_accepts_rn():
    x = _rand(2, 3, 8, 8, seed=4).float()
    w = (_rand(16, 3, 7, 7, seed=5) / math.sqrt(147)).float()
    bias = (_rand(16, seed=6) * 0.1).float()
    rows = _rand(2, 16, seed=7).float()
    r, rabs = T.stem_ref(x, w, bias, rows, True)
    nv, ratio, frac = R.check_bound(R.bf16(r), r, T.stem_bound(r, rabs, 3))
    assert nv == 0 and frac == 0.0


# ---- gn_finalize -------------------------------------------------------------------------------------------------------------------
def _fin_case(b=6, c=32, hw=64, groups=4, og=4):
    gi = torch.arange(c) // (c // groups)
    bi = torch.arange(b)[:, None]
    scale = 2.0 ** (((bi * 5 + gi[None] * 3) % 9).double() / 4 - 1)
    mean = scale * (((bi * 7 + gi[None]) % 9).double() - 4) * 2
    raw = R.bf16(_rand(b, c, hw, seed=1) * scale[:, :, None] + mean[:, :, None])
    res = R.bf16(_rand(b, c, hw, seed=2))
    gamma, beta = 1 + 0.1 * _rand(c, seed=3), 0.1 * _rand(c, seed=4)
    stats = T.fixed_stats(raw, groups)
    o, d, bound = T.finalize_ref(raw, res, stats, groups, gamma, beta, True, True)
    return raw, res, gamma, beta, stats, o, d, bound


def test_finalize_mirror_accepts_rn_and_matches_torch_group_norm():
    raw, res, gamma, beta, stats, o, d, bound = _fin_case()
    assert T.check_bound(R.bf16(o), o, bound)[0] == 0
    gn = torch.nn.functional.group_norm(raw, 4, gamma, beta, eps=R.GN_EPS)
    ref = torch.nn.functional.silu(gn) + res
    assert float((ref - o).abs().max()) <= 1e-5 * float(o.abs().max())


def test_finalize_rejects_statistics_of_the_wrong_sample_or_group_for_one_channel_vector():
    raw, res, gamma, beta, stats, o, d, bound = _fin_case()
    for wrong in ("sample", "group"):
        ob, _, _ = T.finalize_ref(raw, res, stats.roll(1, 0 if wrong == "sample" else 1), 4, gamma, beta, True, True)
        y = R.bf16(o).clone()
        y[3, 8:16] = R.bf16(ob)[3, 8:16]                                  # one 8-channel vector of sample 3
        assert T.check_bound(y, o, bound)[0] > 0
        if wrong == "sample":
            # the same defect in one channel vector of one sample of a configs[1] level-0 output (256 x 128 x 32 x 32, 16 times the
            # test's 64 positions): the rel-L2 gate accepts it (about 1e-2)
            assert _prod_rel_l2((y - R.bf16(o))[3, 8:16], o, 256 * 128 * 1024 / 16) <= GATE


def test_output_statistics_bound_accepts_and_rejects_a_missing_block_atomic():
    raw, res, gamma, beta, stats, o, d, bound = _fin_case()
    _, bpi, per_thread, n_at = T.finalize_geometry(6, 64, 32, 4, True, 4)
    S, Q, dS, dQ = T.out_stats_ref(o, d, 4, per_thread, n_at)
    st = torch.stack([S.round(), Q.round()], -1).to(torch.int64)
    assert T.check_out_stats(st, S, Q, dS, dQ)[0] == 0
    # one warp's atomic of sample 2, group 1 missing: the 8-channel vectors of 32 of the 64 pixels
    g = o.reshape(6, 4, 8, 64)[2, 1, :, :32]
    bad = st.clone()
    bad[2, 1, 0] -= int(round(float(g.sum()) * T.STAT_SUM))
    bad[2, 1, 1] -= int(round(float((g * g).sum()) * T.STAT_SQ))
    assert T.check_out_stats(bad, S, Q, dS, dQ)[0] >= 1


# ---- final projection and fused tail ------------------------------------------------------------------------------------------------
def _ddpm_row(t, T_=1000):
    """{c0, c1, c2, c3, c4, 0} of the linear schedule (gaussian_diffusion.py) in fp64, rounded to fp32."""
    betas = torch.linspace(1e-4, 0.02, T_, dtype=torch.float64)
    ac = torch.cumprod(1 - betas, 0)
    acp = torch.cat([torch.ones(1, dtype=torch.float64), ac[:-1]])
    pv = betas * (1 - acp) / (1 - ac)
    plv = torch.log(torch.cat([pv[1:2], pv[1:]]))
    row = [(1 / ac[t]).sqrt(), (1 / ac[t] - 1).sqrt(), betas[t] * acp[t].sqrt() / (1 - ac[t]),
           (1 - acp[t]) * (1 - betas[t]).sqrt() / (1 - ac[t]), (0.5 * plv[t]).exp() if t > 0 else torch.tensor(0.0), torch.tensor(0.0)]
    return torch.tensor([float(v) for v in row], dtype=torch.float32)


def _tail_case(b=4, c=32, hw=784, groups=8, cout=1, t=500, xs=1.0):
    y = R.bf16(_rand(b, c, hw, seed=1) * 1.5 + 0.3 * torch.arange(b, dtype=torch.float64)[:, None, None])
    gamma, beta = 1 + 0.1 * _rand(c, seed=2), 0.1 * _rand(c, seed=3)
    w, bias = _rand(cout, c, seed=4) / math.sqrt(c), 0.1 * _rand(cout, seed=5)
    stats = T.fixed_stats(y, groups)
    eps, e_eps = T.proj_ref(y, stats, groups, gamma, beta, w, bias, False, True)
    x = _rand(b, cout, hw, seed=6) * xs
    z = _rand(b, cout, hw, seed=7)
    row = _ddpm_row(t)
    o, eo = T.ddpm_ref(x, eps, e_eps, z, 0.0, row)
    return y, gamma, beta, w, bias, stats, eps, e_eps, x, z, row, o, eo


def test_projection_mirror_matches_torch_and_tail_accepts_fp32_evaluation():
    y, gamma, beta, w, bias, stats, eps, e_eps, x, z, row, o, eo = _tail_case()
    a = torch.nn.functional.silu(torch.nn.functional.group_norm(y, 8, gamma, beta, eps=R.GN_EPS))
    ref = torch.einsum("bcp,oc->bop", a, w) + bias[None, :, None]
    assert float((ref - eps).abs().max()) <= 1e-5 * float(eps.abs().max())
    # the kernel's fp32 expression on the mirror's eps
    c = row.float()
    x32, e32 = x.float(), eps.float()
    x0 = (c[0] * x32 - c[1] * e32).clamp(-1, 1)
    out = c[2] * x0 + c[3] * x32 + c[4] * z.float()
    assert T.check_bound(out, o, eo)[0] == 0


def test_tail_rejects_the_neighbouring_pixels_eps_in_the_ragged_last_block():
    # t = 1 and |x| of a few tenths: x0 = c0 x - c1 eps is mostly inside (-1, 1), where eps reaches the output
    y, gamma, beta, w, bias, stats, eps, e_eps, x, z, row, o, eo = _tail_case(t=1, xs=0.3)
    eb = eps.clone()
    eb[2, 0, 770] = eps[2, 0, 771]                     # block 6 holds pixels 768..783 of a 784-pixel map
    ob, _ = T.ddpm_ref(x, eb, e_eps, z, 0.0, row)
    assert T.check_bound(ob, o, eo)[0] == 1
    assert _prod_rel_l2(ob - o, o, 256 * 784) <= GATE


def test_tail_rejects_sample_0_statistics_for_every_sample():
    y, gamma, beta, w, bias, stats, eps, e_eps, x, z, row, o, eo = _tail_case()
    eb, _ = T.proj_ref(y, stats[:1].expand_as(stats), 8, gamma, beta, w, bias, False, True)
    ob, _ = T.ddpm_ref(x, eb, e_eps, z, 0.0, row)
    nv, _ = T.check_bound(ob, o, eo)
    assert nv > 0
    # every sample affected: the eps of the tail is 25 % off, which the per-eps gate rejects (x_{t-1} moves by 5e-4 rel-L2 only)
    assert float((eb - eps).norm() / eps.norm()) > GATE
    assert _prod_rel_l2(ob - o, o, o.numel()) <= GATE


def test_tail_clamp_interval():
    """Where x0 is clamped beyond the bound the element is exact; within the bound of +-1 the interval is one-sided."""
    x = torch.tensor([[[0.0, 0.0, 0.0]]], dtype=torch.float64)
    eps = torch.tensor([[[-5.0, -1.0, 0.0]]], dtype=torch.float64)
    row = torch.tensor([1.0, 1.0, 1.0, 0.0, 0.0, 0.0])
    o, eo = T.ddpm_ref(x, eps, 1e-3, None, 0.0, row)
    assert o.tolist() == [[[1.0, 1.0, 0.0]]]
    assert float(eo[0, 0, 0]) < 1e-6 and 1e-3 <= float(eo[0, 0, 1]) < 2e-3

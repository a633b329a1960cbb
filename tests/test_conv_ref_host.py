"""The conv checker of tests/conv_ref.py on the CPU: its fp64 reference equals torch's convolutions, its probes cover every
(tap, input channel) pair, it accepts the correctly rounded result and rejects small injected faults -- faults that the rel-L2 /
statistics gates of the per-layer tests accept at the production output size."""
import math

import pytest
import torch
import torch.nn.functional as F

import conv_ref as R

CPU = torch.device("cpu")


def _rand(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


def _rel_l2(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm())


SHAPES = [(0, 3, 32, 32, 6), (0, 1, 64, 32, 5), (0, 3, 32, 64, 4), (1, 4, 32, 32, 8), (2, 4, 32, 64, 4), (2, 4, 64, 32, 3)]


@pytest.mark.parametrize("mode,k,cin,cout,h", SHAPES)
def test_reference_equals_torch_fp64(mode, k, cin, cout, h):
    x = _rand(2, cin, h, h, seed=1)
    w = _rand(*((cin, cout, 4, 4) if mode == 2 else (cout, cin, k, k)), seed=2)
    b = _rand(cout, seed=3)
    if mode == 0:
        ref = F.conv2d(x, w, b, padding=k // 2)
    elif mode == 1:
        ref = F.conv2d(x, w, b, stride=2, padding=1)
    else:
        ref = F.conv_transpose2d(x, w, b, stride=2, padding=1)
    got = R.conv_ref(x, w, b, mode, k)
    assert got.shape == ref.shape
    assert float((got - ref).abs().max()) <= 1e-12 * float(ref.abs().max())


def test_reference_concat_equals_torch_fp64():
    x1, x2 = _rand(2, 32, 5, 5, seed=1), _rand(2, 64, 5, 5, seed=2)
    w, b = _rand(32, 96, 3, 3, seed=3), _rand(32, seed=4)
    ref = F.conv2d(torch.cat([x1, x2], 1), w, b, padding=1)
    assert float((R.conv_ref((x1, x2), w, b, 0, 3) - ref).abs().max()) <= 1e-12 * float(ref.abs().max())


@pytest.mark.parametrize("mode,k,cin,cout", [(0, 3, 128, 128), (0, 3, 512, 128), (0, 1, 512, 256), (0, 3, 128, 256), (1, 4, 256, 256),
                                             (2, 4, 128, 128), (0, 3, 96, 64)])
def test_probes_cover_every_tap_and_channel(mode, k, cin, cout):
    nt = R.taps(mode, k)
    seen = torch.zeros(nt, cin, dtype=torch.int64)
    for j in range(R.probe_count(cin, cout, mode, k)):
        w = R.probe_weights(cin, cout, mode, k, j)
        wo = w.transpose(0, 1) if mode == 2 else w           # [cout][cin][k][k]
        assert torch.equal((wo != 0).flatten(1).sum(1), torch.ones(cout, dtype=torch.int64))     # one weight per output channel
        assert set(w.unique().tolist()) == {0.0, 1.0}
        seen += (wo != 0).sum(0).flatten(1).T.long()
        tap, _ = R.probe_assign(cin, cout, mode, k, j)
        assert len(set(tap.tolist())) == min(nt, cout)       # t(o) cycles over the taps
    assert int(seen.min()) >= 1, "some (tap, channel) pair is never probed"
    # the first probe_channels_count probes already use every input channel (both sources of a concat)
    used = set()
    for j in range(R.probe_channels_count(cin, cout)):
        used |= set(R.probe_assign(cin, cout, mode, k, j)[1].tolist())
    assert used == set(range(cin))


@pytest.mark.parametrize("mode,k", [(0, 3), (0, 1), (1, 4), (2, 4)])
def test_probe_gather_equals_probe_convolution(mode, k):
    cin, cout = 64, 32
    x1, x2 = R.bf16(_rand(3, 32, 6, 6, seed=1)), R.bf16(_rand(3, 32, 6, 6, seed=2))
    for j in range(R.probe_count(cin, cout, mode, k)):
        w = R.probe_weights(cin, cout, mode, k, j).double()
        r, pad = R.probe_ref((x1, x2), cin, cout, mode, k, j)
        assert torch.equal(r, R.conv_ref((x1, x2), w, None, mode, k))
        ones = R.conv_ref(torch.ones(3, cin, 6, 6, dtype=torch.float64), w, None, mode, k)
        assert torch.equal(pad, ones == 0)


def _probe_case(mode=0, k=3, cin=64, cout=64, b=3, h=8, j=1):
    x = R.bf16(_rand(b, cin, h, h, seed=5)).float()
    bias = _rand(cout, seed=6).float() * 0.1
    r0, pad = R.probe_ref(x, cin, cout, mode, k, j)
    return x, bias, r0, pad, R.probe_expected(r0, bias)


def test_probe_check_accepts_exact_and_rejects_one_ulp():
    _, _, _, _, exp = _probe_case()
    assert R.check_probe(exp.clone(), exp)[0] == 0
    y = exp.clone()
    v = y[1, 7, 3, 4]
    y[1, 7, 3, 4] = v + float(R.ulp_bf16(v))                   # the next bf16 number
    assert R.bf16(y)[1, 7, 3, 4] == y[1, 7, 3, 4]
    assert R.check_probe(y, exp)[0] == 1


def test_probe_check_rejects_a_shifted_128_row_block():
    """One 128-position block of the flat (image, row, col) order shifted by one position, in every output channel."""
    _, _, _, _, exp = _probe_case(b=4, h=16)
    y = exp.clone()
    flat = y.permute(0, 2, 3, 1).reshape(-1, y.shape[1])         # [positions][channels] (the engine's NHWC rows)
    blk = slice(3 * 128, 4 * 128)
    flat[blk] = torch.roll(flat[blk], 1, 0)
    y = flat.reshape(4, 16, 16, -1).permute(0, 3, 1, 2)
    assert R.check_probe(y, exp)[0] > 100


def test_prologue_probe_rejects_a_nonzero_padding_read():
    """Through the prologue the padding must read exactly zero (+ bias), although SiLU(GroupNorm(0)) + temb is not zero."""
    b, cin, cout, h, j = 2, 64, 64, 8, 0
    x = R.bf16(_rand(b, cin, h, h, seed=1) * 2 + 0.5)
    gamma, beta, temb = 1 + 0.1 * _rand(cin, seed=2), 0.1 * _rand(cin, seed=3), _rand(b, cin, seed=4)
    bias = (_rand(cout, seed=5) * 0.1).float()
    a, t, scale = R.prologue_ref(x, 8, gamma, beta, temb)
    e = R.prologue_error(a, t, scale, temb)
    a_s, pad = R.probe_ref(a, cin, cout, 0, 3, j)
    e_s, _ = R.probe_ref(e, cin, cout, 0, 3, j)
    bound = R.probe_prologue_bound(a_s, e_s, bias)
    y = R.probe_expected(R.bf16(a_s), bias)                       # the engine's exact result for a correctly rounded operand
    assert bool(((y.double() - (a_s + bias.double()[None, :, None, None])).abs() <= bound).all())
    padv = R.probe_expected(torch.zeros_like(a_s), bias)
    assert bool((y == padv)[pad].all()) and int(pad.sum()) > 0
    # fault: one padding position reads the transformed zero (the prologue applied to a pad)
    i = pad.nonzero()[0].tolist()
    y2 = y.clone()
    z = R.prologue_ref(torch.zeros(b, cin, 1, 1, dtype=torch.float64) + x.mean(), 8, gamma, beta, temb)[0]
    y2[tuple(i)] = y2[tuple(i)] + float(z[i[0], 3, 0, 0])
    assert int((y2 != padv)[pad].sum()) == 1


def test_random_weight_bound_accepts_rn_and_rejects_a_dropped_pass():
    b, cin, cout, h, k = 2, 128, 32, 8, 3
    x = R.bf16(_rand(b, cin, h, h, seed=1))
    w = R.bf16(_rand(cout, cin, k, k, seed=2) / math.sqrt(cin * 9))
    bias = _rand(cout, seed=3) * 0.1
    r = R.conv_ref(x, w, bias, 0, k)
    rabs = R.conv_ref(x.abs(), w.abs(), None, 0, k)
    bound = R.element_bound(r, rabs, cin * 9)
    nv, ratio, frac = R.check_bound(R.bf16(r), r, bound)
    assert nv == 0 and ratio <= 1.0 and frac == 0.0
    # fault: one output element misses the 32-channel pass of one tap (channels 64..95, tap (1, 2))
    wd = w.clone()
    wd[:, 64:96, 1, 2] = 0
    rd = R.conv_ref(x, wd, bias, 0, k)
    y = R.bf16(r).clone()
    y[1, 5, 4, 4] = R.bf16(rd)[1, 5, 4, 4]
    assert R.check_bound(y, r, bound)[0] == 1


def test_statistics_bound_accepts_and_rejects_a_missing_block():
    b, c, h, groups = 2, 64, 16, 8
    r = _rand(b, c, h, h, seed=1) + 0.3
    mean, rstd = R.stats_ref(r, groups)
    st = torch.stack([mean.float(), rstd.float()], -1)
    delta = R.U32 * r.abs()
    nv, sm, sr = R.check_stats(st, r, delta, groups)
    assert nv == 0 and sm < 1 and sr < 1
    # fault: the statistics miss one 16-position block of one channel
    rm = r.clone()
    rm[1, 9, 3, 0:16] = 0
    g = rm.reshape(b, groups, -1)
    n = g.shape[-1]
    s, q = g.sum(-1), (g * g).sum(-1)
    m = s / n
    st_bad = torch.stack([m.float(), ((q / n - m * m) + R.GN_EPS).rsqrt().float()], -1)
    assert R.check_stats(st_bad, r, delta, groups)[0] >= 1


# ---- the same faults at production size against the gates of the per-layer tests (rel-L2 4e-3, stats atol 2e-3 / rtol 5e-3) ----
B, C, H = 256, 128, 32         # configs[1] level-0 conv output at the benchmark batch: 33.5 M elements


@pytest.fixture(scope="module")
def production_output():
    """A synthetic conv output of production size, spatially smooth as a U-Net activation is (a 5x5 box blur of white noise, fp32:
    only the fault's size against the whole tensor matters here)."""
    g = torch.Generator().manual_seed(0)
    z = torch.randn(B * C, 1, H + 4, H + 4, generator=g)
    y = F.avg_pool2d(z, 5, stride=1) * 5.0
    return y.reshape(B, C, H, H) + 0.1


def test_today_gates_accept_a_shifted_128_row_block(production_output):
    """One 128-row block shifted by one position: in one 16-byte store column (8 channels) the per-layer gate passes it; across
    all 128 channels the whole-U-Net gate (rel-L2 2e-2) still does.  The probe check rejects either (test above)."""
    y = production_output
    blk = slice(1000 * 128, 1001 * 128)
    for chans, gate in ((slice(40, 48), 4e-3), (slice(0, C), 2e-2)):
        bad = y.permute(0, 2, 3, 1).reshape(-1, C).clone()
        bad[blk, chans] = torch.roll(bad[blk, chans], 1, 0)
        bad = bad.reshape(B, H, H, C).permute(0, 3, 1, 2)
        assert int((bad != y).sum()) >= 1000
        assert _rel_l2(bad, y) <= gate


def test_today_gates_accept_a_dropped_pass_tile(production_output):
    """One 128-row tile in which one tap's 32-channel pass (32 of the 1152 products of a 3x3 128-channel conv) is missing."""
    y = production_output
    g = torch.Generator().manual_seed(1)
    flat = y.permute(0, 2, 3, 1).reshape(-1, C).clone()
    blk = slice(2000 * 128, 2001 * 128)
    # the missing partial sum: 32 of 1152 i.i.d. products of the output's spread
    flat[blk] -= torch.randn(128, C, generator=g) * float(y.std()) * math.sqrt(32 / 1152)
    bad = flat.reshape(B, H, H, C).permute(0, 3, 1, 2)
    assert _rel_l2(bad, y) <= 4e-3


def test_today_gates_accept_missing_statistics_block(production_output):
    y = production_output.double()
    groups = 8
    g = y.reshape(B, groups, -1)
    mean, rstd = g.mean(-1), (g.var(-1, unbiased=False) + R.GN_EPS).rsqrt()
    ym = y.clone()
    ym[7, 3, 5, 0:16] = 0                               # one 16-position block of one channel missing from the sums
    gm = ym.reshape(B, groups, -1)
    n = gm.shape[-1]
    m2 = gm.sum(-1) / n
    r2 = ((gm * gm).sum(-1) / n - m2 * m2 + R.GN_EPS).rsqrt()
    assert torch.allclose(m2, mean, atol=2e-3) and torch.allclose(r2, rstd, rtol=5e-3)
    st_bad = torch.stack([m2.float(), r2.float()], -1)
    assert R.check_stats(st_bad, y, R.U32 * y.abs(), groups)[0] >= 1

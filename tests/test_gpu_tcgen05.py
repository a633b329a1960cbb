"""The tcgen05/TMEM implicit-GEMM engine on the GPU: descriptor self-test, per-layer checks against the fp64 reference and
element bounds of tests/conv_ref.py, and whole-U-Net parity in bf16 mode (<= 2e-2 rel-L2)."""
import pytest
import torch
import torch.nn.functional as F

from diffusion_model_nemo_b200 import _lib as L
from conftest import CFGS, make_unet, rel_l2
from gpu_helpers import conv_forward
from oracle import ref_port as O
import conv_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rand(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def _bf(t):
    return t.to(torch.bfloat16).float()


@pytest.mark.parametrize("M_,N,K", [(256, 128, 32), (512, 128, 64), (1000, 64, 128), (4096, 384, 256), (300, 32, 32)])
def test_umma_gemm_selftest(M_, N, K):
    lib = L.lib()
    a, b = _bf(_rand(M_, K, seed=1)), _bf(_rand(N, K, seed=2))
    d = torch.empty(M_, N, device=DEV)
    ad, bd = a.to(DEV, torch.bfloat16).contiguous(), b.to(DEV, torch.bfloat16).contiguous()
    L.check(lib.dmn_selftest_umma_gemm(L.ptr(ad), L.ptr(bd), L.ptr(d), M_, N, K, L.stream_ptr(DEV)), "selftest")
    ref = a @ b.T
    assert rel_l2(d.cpu(), ref) <= 4e-3       # output is rounded to bf16 by the engine's epilogue


def _check_plain(y, st, x, w, bias, mode, k, og):
    """Element bound against the fp64 convolution (tests/conv_ref.py) and, with og groups, the statistics bound."""
    cin = x.shape[1]
    K = cin * R.taps(mode, k)
    r = R.conv_ref(x, w, bias, mode, k)
    rabs = R.conv_ref(x.abs(), w.abs(), None, mode, k)
    nv, ratio, frac = R.check_bound(y.cpu(), r, R.element_bound(r, rabs, K))
    assert nv == 0, f"{nv} elements over the bound (max err / bound {ratio:.3g})"
    assert frac <= 0.01, frac
    if og:
        nv, sm, sr = R.check_stats(st.cpu(), r, R.acc_delta(r, rabs, K), og)
        assert nv == 0, (sm, sr)


@pytest.mark.parametrize("k,cin,cout,h,b", [(3, 32, 32, 4, 5), (3, 64, 64, 8, 3), (3, 128, 128, 16, 2), (3, 128, 128, 32, 2),
                                            (3, 256, 256, 8, 4), (1, 128, 384, 16, 2), (1, 128, 256, 4, 7), (3, 64, 128, 7, 3)])
def test_conv_tcgen05_vs_torch(k, cin, cout, h, b):
    x = _bf(_rand(b, cin, h, h, seed=1))
    w = _bf(_rand(cout, cin, k, k, seed=2) / (cin * k * k) ** 0.5)
    bias = _rand(cout, seed=3) * 0.1
    og = cout // 32 if cout >= 64 else 0       # 32 channels per statistics group; fused statistics need an N tile >= 64
    y, st = conv_forward(x.to(DEV), w.to(DEV), bias.to(DEV), ksize=k, out_groups=og, act=L.ACT_BF16, engine=L.CONV_TCGEN05)
    assert y.shape == (b, cout, h, h)
    _check_plain(y, st, x, w, bias, 0, k, og)


@pytest.mark.parametrize("mode,cin,cout,h,b", [(1, 32, 32, 8, 3), (1, 128, 128, 32, 2), (1, 256, 256, 16, 3), (1, 64, 64, 14, 2),
                                               (2, 32, 32, 4, 5), (2, 256, 256, 8, 2), (2, 128, 128, 16, 2), (2, 64, 64, 7, 3)])
def test_conv_tcgen05_down_up_vs_torch(mode, cin, cout, h, b):
    """Downsample (Conv k4 s2 p1 as a 2x2 conv over the space-to-depth image) and Upsample (ConvTranspose k4 s2 p1 as four
    sub-pixel phases) on the tensor-core engine (reference utils.py:77-82)."""
    x = _bf(_rand(b, cin, h, h, seed=1))
    w = _bf(_rand(*((cin, cout, 4, 4) if mode == 2 else (cout, cin, 4, 4)), seed=2) / (cin * 8) ** 0.5)
    bias = _rand(cout, seed=3) * 0.1
    ref = F.conv2d(x, w, bias, stride=2, padding=1) if mode == 1 else F.conv_transpose2d(x, w, bias, stride=2, padding=1)
    y, _ = conv_forward(x.to(DEV), w.to(DEV), bias.to(DEV), mode=mode, ksize=4, act=L.ACT_BF16, engine=L.CONV_TCGEN05)
    assert y.shape == ref.shape
    _check_plain(y, None, x, w, bias, mode, 4, 0)


def _check_prologue(y, st, x, w, bias, k, groups, gamma, beta, temb, silu, og):
    """Prologue cases: the fp64 SiLU(GroupNorm(x)) + temb operand, its error bound propagated statistically (conv_ref.py)."""
    a, t, scale = R.prologue_ref(x, groups, gamma, beta, temb, silu=silu)
    e_op = R.operand_bound(a, R.prologue_error(a, t, scale, temb, silu=silu))
    K = x.shape[1] * k * k
    r = R.conv_ref(a, w, bias, 0, k)
    rabs = R.conv_ref(a.abs(), w.abs(), None, 0, k)
    extra = R.K_SIGMA * R.prologue_sigma(e_op, w, 0, k)
    nv, ratio, _ = R.check_bound(y.cpu(), r, R.element_bound(r, rabs, K, extra))
    assert nv == 0, f"{nv} elements over the bound (max err / bound {ratio:.3g})"
    if og:
        nv, sm, sr = R.check_stats(st.cpu(), r, R.acc_delta(r, rabs, K) + extra, og)
        assert nv == 0, (sm, sr)


def test_conv_tcgen05_prologue_and_gn1_stats():
    b, c, h = 4, 128, 16
    x = _bf(_rand(b, c, h, h, seed=1) * 2 + 0.5)
    w = _bf(_rand(128, c, 3, 3, seed=2) / (c * 9) ** 0.5)
    bias, gamma, beta, temb = _rand(128, seed=3) * 0.1, 1 + 0.1 * _rand(c, seed=4), 0.1 * _rand(c, seed=5), _rand(b, c, seed=6)
    y, st = conv_forward(x.to(DEV), w.to(DEV), bias.to(DEV), gn=(8, gamma.to(DEV), beta.to(DEV)), silu=True, temb=temb.to(DEV),
                         out_groups=1, act=L.ACT_BF16, engine=L.CONV_TCGEN05)
    _check_prologue(y, st, x, w, bias, 3, 8, gamma, beta, temb, True, 1)
    w1 = _bf(_rand(384, c, 1, 1, seed=7) / c ** 0.5)
    y, _ = conv_forward(x.to(DEV), w1.to(DEV), None, ksize=1, gn=(1, gamma.to(DEV), beta.to(DEV)), act=L.ACT_BF16, engine=L.CONV_TCGEN05)
    _check_prologue(y, None, x, w1, None, 1, 1, gamma, beta, None, False, 0)


@pytest.mark.parametrize("name", ["cfg2", "tiny", "cfg1", "tiny_g4"])
def test_unet_bf16_tcgen05_vs_reference_golden(golden, name):
    cfg, size, b = CFGS[name]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="bf16", engine="tcgen05", device=DEV)
    x = torch.from_numpy(golden["unet"][f"{name}/x"]).to(DEV)
    for tname in ("int", "float"):
        t = torch.from_numpy(golden["unet"][f"{name}/{tname}/t"]).to(DEV)
        y = u(x, t)
        assert rel_l2(y.cpu(), torch.from_numpy(golden["unet"][f"{name}/{tname}/y"])) <= 2e-2, (name, tname)


def test_teacher_forced_eps_cfg2_tcgen05(golden):
    cfg, size, b = CFGS["cfg2"]
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="bf16", engine="tcgen05", device=DEV)
    x = torch.from_numpy(golden["step"]["cfg2/x"]).to(DEV)
    for ti in (999, 500, 1, 0):
        eps = u(x, torch.full((b,), ti, device=DEV))
        assert rel_l2(eps.cpu(), torch.from_numpy(golden["step"][f"cfg2/t{ti}/eps"])) <= 2e-2, ti

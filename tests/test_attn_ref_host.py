"""CPU checks of tests/attn_ref.py, the fp64 references of the fused attention blocks: the unrounded mirror (the kernel's tiled online
k softmax) is the exact block, the exact block is the oracle's restatement of parts/mha.py, and the rounding points alone keep the
mirror within a derived distance of the exact block."""
import pytest
import torch

from oracle import ref_port as O
import attn_ref as A


def _sd(c, seed, softmax, qkv_gain, bias_shift=0.0):
    g = torch.Generator().manual_seed(seed)
    u = lambda *s, fan: (torch.rand(*s, generator=g) * 2 - 1) / fan ** 0.5      # noqa: E731
    p = "blk"
    sd = {p + ".fn.norm.weight": 1 + 0.1 * torch.randn(c, generator=g), p + ".fn.norm.bias": 0.1 * torch.randn(c, generator=g),
          p + ".fn.fn.to_qkv.weight": u(384, c, 1, 1, fan=c) * qkv_gain}
    out = p + (".fn.fn.to_out" if softmax else ".fn.fn.to_out.0")
    sd[out + ".weight"] = u(c, 128, 1, 1, fan=128)
    sd[out + ".bias"] = 0.05 * torch.randn(c, generator=g) + bias_shift
    if not softmax:
        sd[p + ".fn.fn.to_out.1.weight"] = 1 + 0.1 * torch.randn(c, generator=g)
        sd[p + ".fn.fn.to_out.1.bias"] = 0.1 * torch.randn(c, generator=g)
    return p, sd


def _x(b, c, h, seed):
    """Per-image scale and offset, and a token ramp that moves the k maximum across tiles."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(b, c, h, h, generator=g)
    ramp = torch.linspace(-1.5, 1.5, h * h).reshape(1, 1, h, h)
    sc = torch.tensor([0.5, 2.0, 1.0])[torch.arange(b) % 3].reshape(b, 1, 1, 1)
    off = torch.tensor([-1.0, 0.5, 1.0])[torch.arange(b) % 3].reshape(b, 1, 1, 1)
    sign = torch.tensor([1.0, -1.0, 0.0])[torch.arange(b) % 3].reshape(b, 1, 1, 1)
    return A.bf16(x * sc + off + sign * ramp)


CASES = [(False, 4, 256), (False, 8, 256), (False, 8, 128), (False, 16, 128), (False, 16, 256), (False, 32, 128),
         (True, 4, 256), (True, 8, 256), (True, 8, 128)]


@pytest.mark.parametrize("softmax,h,c", CASES)
def test_exact_is_the_oracle_block_and_unrounded_mirror_is_exact(softmax, h, c):
    """N = 16 and 64 (one zero-padded tile in the kernel), 256 and 1024 (2 and 8 tiles of the online k softmax)."""
    p, sd = _sd(c, 3 + h, softmax, qkv_gain=6.0 if not softmax else 3.0)
    x = _x(3, c, h, seed=h + c).double()
    sd64 = {k: v.double() for k, v in sd.items()}
    fn = O.attention_fwd if softmax else O.linear_attention_fwd
    ref = A.to_tokens(O.residual_prenorm_fwd(sd64, p, x, fn))
    ops = A.operands(x, sd, p, softmax, kernel_rounding=False)
    ex = A.exact(ops, softmax)
    mir = A.mirror(ops, softmax, rounding=False)
    scale = (ref - ops.x).abs().max()
    assert float((ex - ref).abs().max() / scale) <= 1e-12
    assert float((mir - ex).abs().max() / scale) <= 1e-12


def test_online_tiles_see_the_running_max_move():
    """The ramped inputs make the k maximum move after tile 0 in the up-ramped image and stay in the down-ramped one: the rescale
    2^(m_t - m_T) of the mirror is exercised, not a no-op."""
    p, sd = _sd(128, 5, False, qkv_gain=6.0)
    ops = A.operands(_x(3, 128, 32, seed=1), sd, p)
    st = {}
    A.linear_mirror(ops, stats=st)
    moved = (st["kmax"][:, 1:] > st["kmax"][:, :-1]).double().mean((1, 2))
    assert st["kmax"].shape == (3, 8, 128)
    assert float(moved[0]) > float(moved[1]) and float(moved[0]) > 0.3


@pytest.mark.parametrize("softmax,h,c,bias_shift", [cs + (0.0,) for cs in CASES] + [cs + (8.0,) for cs in CASES if not cs[0]])
def test_rounded_mirror_within_derived_bound_of_exact(softmax, h, c, bias_shift):
    """With its bf16 rounding points the mirror departs from the exact block by at most mirror_branch_bound (per image, L2 over the
    image).  bias_shift moves the mean of y far from zero (linear block): the parked bf16 y then costs rms(y) / std(y) more."""
    p, sd = _sd(c, 3 + h, softmax, qkv_gain=6.0 if not softmax else 3.0, bias_shift=bias_shift)
    ops = A.operands(_x(3, c, h, seed=h + c), sd, p, softmax)
    ex = A.exact(ops, softmax)
    mir = A.mirror(ops, softmax)
    err = (mir - ex).reshape(3, -1).norm(dim=1)
    bound = A.mirror_branch_bound(ops, softmax)
    assert bool((err > 0).all()), "rounding on must change the result"
    assert bool((err <= bound).all()), (err / bound).tolist()

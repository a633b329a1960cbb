"""fp64 references of the two fused attention blocks of csrc/attn_fused.cu (plain torch, any device, no engine imports).

Both blocks are Residual(PreNorm(dim, fn)) with fn = LinearAttention (linattn_fused_kernel) or the bottleneck softmax Attention
(attn_softmax_fused_kernel), heads 4 x dim_head 32.  The layer entry dmn_linear_attention_block (csrc/api_layers.cu) hands the kernel
x rounded to bf16, W_qkv * gamma rounded to bf16 with the fold vectors s1 = sum_c bf16(W gamma), s2 = sum_c W beta (fp64 sums stored
as fp32), W_o in bf16 and the PreNorm statistics of the bf16 x; `operands` builds the same.  The projection of a token is then
rstd (W_b x - mean s1) + s2, which is W (gamma x_hat + beta) up to the rounding of the folded weight.

  * `*_exact`: the block with no intermediate rounding (parts/mha.py as restated in oracle/ref_port.py), on those operands;
  * `*_mirror`: the same computation with bf16 round-to-nearest (through fp32, as the kernel converts fp32 values) at every point
    where the kernel rounds.  The linear mirror follows the kernel's 128-token tiling of the online k softmax: the P operand of tile t
    is bf16(2^(l - m_t)) against the running maximum m_t of tiles 0..t, and tile t's share of the context and of the column sums
    (sums of the ROUNDED P) is rescaled by 2^(m_t - m_T).  With rounding=False it is the exact function in another order.

The mirrors return the output before its final bf16 rounding (the kernel rounds it once more when it stores it).
Tensors are token-major: x [B][N][C] with token n = row * W + column, as the kernel reads NHWC.
"""
import math
from typing import NamedTuple, Optional

import torch

HEADS, DH, HID = 4, 32, 128
SCALE = DH ** -0.5
LOG2E = math.log2(math.e)
GN_EPS = 1e-5
TILE = 128


class Operands(NamedTuple):
    x: torch.Tensor            # [B][N][C] float64
    wqkv: torch.Tensor         # [384][C]  (PreNorm gamma folded in)
    s1: torch.Tensor           # [384]
    s2: torch.Tensor           # [384]
    wo: torch.Tensor           # [C][128]
    bo: torch.Tensor           # [C]
    go: Optional[torch.Tensor]     # [C] to_out.1 (GroupNorm(1)) weight; None for the softmax block
    beo: Optional[torch.Tensor]
    mean: torch.Tensor         # [B] PreNorm GroupNorm(1) statistics of x
    rstd: torch.Tensor


def bf16(t):
    """bf16 round-to-nearest-even of the fp32 value of t (the kernel rounds fp32 values), keeping the dtype."""
    return t.float().bfloat16().to(t.dtype)


def _ident(t):
    return t


def to_tokens(x):
    """NCHW -> [B][H*W][C]."""
    b, c = x.shape[:2]
    return x.reshape(b, c, -1).transpose(1, 2)


def to_nchw(t, h):
    b, n, c = t.shape
    return t.transpose(1, 2).reshape(b, c, h, n // h)


def operands(x, sd, prefix, softmax=False, kernel_rounding=True):
    """The kernel's operands of Residual(PreNorm(...)) for x (NCHW) and the reference parameter names under `prefix` (as
    gpu_helpers.linear_attention_block takes them), in float64 on x's device.  kernel_rounding=False keeps everything unrounded
    (x, W gamma, W_o and the fold sums in fp64): the block of the reference itself."""
    dev = x.device
    g = lambda k: sd[prefix + k].to(dev)      # noqa: E731
    c = x.shape[1]
    w = g(".fn.fn.to_qkv.weight").reshape(3 * HID, c)
    gam, bet = g(".fn.norm.weight"), g(".fn.norm.bias")
    out = ".fn.fn.to_out" if softmax else ".fn.fn.to_out.0"
    wo, bo = g(out + ".weight").reshape(c, HID), g(out + ".bias")
    if kernel_rounding:
        xt = bf16(to_tokens(x).float()).double()
        wq = bf16(w.float() * gam.float()).double()            # __float2bfloat16_rn(wq * g) in fp32
        s1 = wq.sum(1).float().double()
        s2 = (w.float().double() @ bet.float().double()).float().double()
        wo = bf16(wo.float()).double()
    else:
        xt = to_tokens(x).double()
        wq = w.double() * gam.double()
        s1 = wq.sum(1)
        s2 = w.double() @ bet.double()
        wo = wo.double()
    f32 = (lambda t: t.float().double()) if kernel_rounding else (lambda t: t.double())     # noqa: E731
    go = beo = None
    if not softmax:
        go, beo = f32(g(".fn.fn.to_out.1.weight")), f32(g(".fn.fn.to_out.1.bias"))
    mean = xt.mean((1, 2))
    rstd = (xt.var((1, 2), unbiased=False) + GN_EPS).rsqrt()
    return Operands(xt, wq, s1, s2, wo, f32(bo), go, beo, mean, rstd)


def _proj(ops, r0):
    """Rows [r0, r0 + 128) of to_qkv applied to the PreNorm output: [B][N][128]."""
    w = ops.wqkv[r0:r0 + HID]
    return ops.rstd[:, None, None] * (ops.x @ w.T - ops.mean[:, None, None] * ops.s1[r0:r0 + HID]) + ops.s2[r0:r0 + HID]


def _heads(t):
    return t.reshape(t.shape[0], t.shape[1], HEADS, DH)


def _y_stats(y):
    """Per-image mean and rstd of GroupNorm(1), [B][1][1] each."""
    mu = y.mean((1, 2), keepdim=True)
    var = (y * y).mean((1, 2), keepdim=True) - mu * mu
    return mu, (var.clamp_min(0) + GN_EPS).rsqrt()


def _out_groupnorm(ops, y, y_stat):
    """GroupNorm(1)(y) * go + beo + x with the statistics of y_stat (the kernel sums the fp32 y and normalises the parked bf16 y)."""
    mu, rs = _y_stats(y_stat)
    return (y - mu) * rs * ops.go + ops.beo + ops.x


# ---- LinearAttention block (linattn_fused_kernel) ------------------------------------------------------------------------------
def linear_exact_y(ops):
    """to_out.0 output y [B][N][C] (before GroupNorm(1)) of the exact block."""
    q, k, v = (_heads(_proj(ops, r)) for r in (0, HID, 2 * HID))
    q = q.softmax(-1) * SCALE                     # over the 32 channels of a head
    k = k.softmax(1)                              # over the tokens
    ctx = torch.einsum("bnhd,bnhe->bhde", k, v)
    o = torch.einsum("bhde,bnhd->bnhe", ctx, q)
    return o.reshape(o.shape[0], o.shape[1], HID) @ ops.wo.T + ops.bo


def linear_exact(ops):
    y = linear_exact_y(ops)
    return _out_groupnorm(ops, y, y)


def linear_mirror(ops, rounding=True, stats=None):
    """The kernel's arithmetic with bf16 rounding at its rounding points (rounding=False: none).  stats, if a dict, receives the
    running maxima [B][T][128] of the k logits (log2 domain) per tile ("kmax") and the magnitude |y| rstd_y |go| at which the parked
    y reaches the output ("y_scale", [B][N][C]): one bf16 ulp of y there is the output's sensitivity to a rounding flip of y."""
    R = bf16 if rounding else _ident
    B, N, _ = ops.x.shape
    tile = min(N, TILE)
    T = N // tile
    k2 = (_proj(ops, HID) * LOG2E).reshape(B, T, tile, HID)
    v = R(_proj(ops, 2 * HID))
    m = k2.amax(2).cummax(1).values                              # running max after tile t, per channel
    P = R(torch.exp2(k2 - m[:, :, None, :]))                     # the P operand of tile t
    w = torch.exp2(m - m[:, -1:, :])                              # 2^(m_t - m_T): rescales that tile's share up to the last tile
    colsum = (P.sum(2) * w).sum(1)                                # sums of the rounded P
    Pw = (P * w[:, :, None, :]).reshape(B, N, HEADS, DH)
    ctx = torch.einsum("bnhd,bnhe->bhde", Pw, _heads(v))
    ctx_op = R(ctx * SCALE / colsum.reshape(B, HEADS, DH, 1))
    q2 = _heads(_proj(ops, 0) * LOG2E)
    eq = torch.exp2(q2 - q2.amax(-1, keepdim=True))
    sq = R(eq / eq.sum(-1, keepdim=True))
    o = R(torch.einsum("bnhd,bhde->bnhe", sq, ctx_op)).reshape(B, N, HID)
    y = o @ ops.wo.T + ops.bo                                     # fp32 accumulator + bias: the statistics are taken here
    if isinstance(stats, dict):
        stats["kmax"] = m
        stats["y_scale"] = y.abs() * _y_stats(y)[1] * ops.go.abs()
    return _out_groupnorm(ops, R(y), y)                           # the raw y is parked in bf16 before phase C


# ---- softmax Attention block (attn_softmax_fused_kernel) -----------------------------------------------------------------------
def softmax_exact(ops):
    q, k, v = (_heads(_proj(ops, r)) for r in (0, HID, 2 * HID))
    s = torch.einsum("bihd,bjhd->bhij", q * SCALE, k)
    o = torch.einsum("bhij,bjhe->bihe", s.softmax(-1), v)
    return o.reshape(o.shape[0], o.shape[1], HID) @ ops.wo.T + ops.bo + ops.x


def softmax_mirror(ops, rounding=True):
    R = bf16 if rounding else _ident
    q = _heads(R(_proj(ops, 0) * (SCALE * LOG2E)))               # q * scale in the log2 domain
    k, v = (_heads(R(_proj(ops, r))) for r in (HID, 2 * HID))
    s = torch.einsum("bihd,bjhd->bhij", q, k)
    e = torch.exp2(s - s.amax(-1, keepdim=True))
    p = R(e / e.sum(-1, keepdim=True))
    o = R(torch.einsum("bhij,bjhe->bihe", p, v))
    return o.reshape(o.shape[0], o.shape[1], HID) @ ops.wo.T + ops.bo + ops.x


def exact(ops, softmax):
    return softmax_exact(ops) if softmax else linear_exact(ops)


def mirror(ops, softmax, rounding=True):
    return softmax_mirror(ops, rounding) if softmax else linear_mirror(ops, rounding)


# ---- bounds ------------------------------------------------------------------------------------------------------------------------
U_BF16 = 2.0 ** -9          # unit roundoff of bf16 round-to-nearest
# rounding points before the output of each block: linear P, v, ctx, softmax(q), o (the parked y is counted apart); softmax q, k, v, P, o
ROUND_POINTS = 5


def ulp_bf16(a):
    """Spacing of the bf16 numbers at |a| (8 significant bits; the bf16 subnormal spacing below 2^-126)."""
    _, e = torch.frexp(a.double().abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(a, dtype=torch.float64), e - 8)


def mirror_branch_bound(ops, softmax, ex=None, y=None):
    """Per-image bound on ||mirror - exact|| (L2 over the image, before the output rounding) of the attention branch.

    Each rounding point moves its values by at most U_BF16 relative; between the points the block forms softmax-weighted averages,
    normalised sums and products whose relative error is at most the sum of their operands' (the k softmax counts P twice: numerator
    and column sum; the q . k logits of the softmax block count q and k once more each, scaled by the logit magnitude).  After the
    linear block's GroupNorm(1) a relative error of y becomes rms(y) / std(y) times larger relative to the normalised branch, and
    the parked y adds U_BF16 rms(y) / std(y) of its own.  The bound takes twice the first-order sum."""
    B = ops.x.shape[0]
    ex = exact(ops, softmax) if ex is None else ex
    br = (ex - ops.x).reshape(B, -1).norm(dim=1)
    if softmax:
        q, k = (_heads(_proj(ops, r)) for r in (0, HID))
        logit = (torch.einsum("bihd,bjhd->bhij", q.abs() * SCALE, k.abs())).reshape(B, -1).amax(1)
        rel = U_BF16 * (ROUND_POINTS + 1 + 2 * logit)
    else:
        y = linear_exact_y(ops) if y is None else y
        amp = (y * y).mean((1, 2)).sqrt() / y.std((1, 2), unbiased=False)
        rel = U_BF16 * ((ROUND_POINTS + 1) * amp + amp)
    return 2.0 * rel * br

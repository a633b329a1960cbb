"""fp64 reference and element-wise checker for the tensor-core convolution engine (plain torch, any device, no engine imports).

The engine rounds its operands to bf16, multiplies them exactly (a bf16 x bf16 product has 16 significant bits) and accumulates in
fp32 on the tensor core; the epilogue adds the fp32 bias and rounds to bf16.  So against an fp64 convolution of the same bf16 values:

  * probe weights (one weight 1.0 per output channel) make the engine's output an exact shifted copy of one input channel plus the bias:
    the gate is bit equality, which pins every tap offset, halo, pad row / column, image boundary and tile of the addressing;
  * random weights: every element obeys |y - r| <= 1/2 ulp_bf16(|r| + d) + d,  d = K 2^-23 sum|x w| + 2^-24 |r|, K = Cin * taps,
    which allows truncating fp32 adds in any order (the tensor core's add order and rounding are not documented);
  * the GroupNorm prologue (SiLU through tanh.approx.f32) and the fixed-point output statistics get bounds derived below.
"""
import math

import torch
import torch.nn.functional as F

U32 = 2.0 ** -24          # fp32 unit roundoff (round to nearest)
# PTX ISA, tanh: tanh.approx.f32 has a maximum relative error of 2^-11 over its whole range.  The engine's SiLU is h + h tanh(h) with
# h = t / 2, so the tanh error reaches the operand as |h| |tanh h| 2^-11 <= |h| 2^-11 (large against the result for t << 0).
TANH_REL = 2.0 ** -11
GN_EPS = 1e-5


def bf16(t):
    """Round to bf16 values (round to nearest even), keeping the dtype."""
    return t.to(torch.bfloat16).to(t.dtype)


def ulp_bf16(a):
    """Spacing of the bf16 numbers at |a| (8 significant bits; the bf16 subnormal spacing below 2^-126)."""
    _, e = torch.frexp(a.double().abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(a, dtype=torch.float64), e - 8)


def taps(mode, ksize):
    return ksize * ksize if mode == 0 else 16


def _padded(x, mode, ksize):
    """Every mode as a stride-s correlation over a padded input: returns (xp, stride, Ho, Wo).  The transposed k4s2 conv is the
    zero-inserted input (stride 2 -> 1) padded by k - 1 - p = 2, correlated with the flipped, transposed kernel (see _corr_weight)."""
    B, C, H, W = x.shape
    if mode == 0:
        p = ksize // 2
        return F.pad(x, (p, p, p, p)), 1, H, W
    if mode == 1:
        return F.pad(x, (1, 1, 1, 1)), 2, H // 2, W // 2
    xu = x.new_zeros(B, C, 2 * H - 1, 2 * W - 1)
    xu[:, :, ::2, ::2] = x
    return F.pad(xu, (2, 2, 2, 2)), 1, 2 * H, 2 * W


def _corr_weight(w, mode):
    """torch-layout weight -> [Cout][Cin][k][k] correlation weight of _padded's form."""
    return w.flip(2, 3).transpose(0, 1) if mode == 2 else w


def _tap_view(xp, ky, kx, stride, Ho, Wo):
    return xp[:, :, ky:ky + stride * (Ho - 1) + 1:stride, kx:kx + stride * (Wo - 1) + 1:stride]


def cat_sources(x):
    return torch.cat(list(x), 1) if isinstance(x, (list, tuple)) else x


def conv_ref(x, w, bias=None, mode=0, ksize=3):
    """fp64 y = conv(x, w) + bias as an explicit sum over taps.  mode 0: k x k stride 1 same padding (k = 1, 3); 1: k4 s2 p1;
    2: ConvTranspose2d k4 s2 p1.  x: [B, Cin, H, W] or a tuple of sources concatenated along channels; w in torch layout
    ([Cout][Cin][k][k], transposed conv [Cin][Cout][4][4])."""
    x = cat_sources(x).double()
    wc = _corr_weight(w.double(), mode)
    xp, s, Ho, Wo = _padded(x, mode, ksize)
    k = wc.shape[-1]
    out = x.new_zeros(x.shape[0], wc.shape[0], Ho, Wo)
    for ky in range(k):
        for kx in range(k):
            out += torch.einsum("bchw,oc->bohw", _tap_view(xp, ky, kx, s, Ho, Wo), wc[:, :, ky, kx])
    if bias is not None:
        out += bias.double()[None, :, None, None]
    return out


# ---- probe weights ---------------------------------------------------------------------------------------------------------------
def _coprime_mult(cin):
    return next(a for a in (5, 7, 11, 13, 17, 19, 23, 29, 31) if math.gcd(a, cin) == 1)


def probe_count(cin, cout, mode, ksize):
    """Probes until every (tap, input channel) pair has been used once."""
    return -(-cin * taps(mode, ksize) // cout)


def probe_channels_count(cin, cout):
    """Probes until every input channel (of both concat sources) has been used once: the first ceil(cin / cout), at least two."""
    return max(2, -(-cin // cout))


def probe_assign(cin, cout, mode, ksize, j):
    """(tap, input channel) of every output channel in probe j.  Pair k = j * cout + o (mod cin * taps) maps to
    ci = a k mod cin (a coprime to cin: a permutation over any cin consecutive k) and tap = (k // cin + ci) mod taps, so the
    pairs of consecutive probes are distinct until all cin * taps are used, c(o) is a permutation within cin consecutive outputs and
    t(o) cycles over the taps.  Taps are numbered ky * k + kx of the torch-layout weight."""
    nt = taps(mode, ksize)
    k = (j * cout + torch.arange(cout)) % (cin * nt)
    ci = (_coprime_mult(cin) * k) % cin
    tap = (k // cin + ci) % nt
    return tap, ci


def probe_weights(cin, cout, mode, ksize, j):
    """torch-layout fp32 weight of probe j: exactly one 1.0 per output channel."""
    tap, ci = probe_assign(cin, cout, mode, ksize, j)
    k = ksize if mode == 0 else 4
    o = torch.arange(cout)
    if mode == 2:
        w = torch.zeros(cin, cout, k, k)
        w[ci, o, tap // k, tap % k] = 1.0
    else:
        w = torch.zeros(cout, cin, k, k)
        w[o, ci, tap // k, tap % k] = 1.0
    return w


def probe_ref(x, cin, cout, mode, ksize, j):
    """The probe output without bias in fp64: a gather of the input (zero where the tap reads padding).  Also returns the mask of
    elements that read padding (or, transposed, that receive no product)."""
    x = cat_sources(x).double()
    tap, ci = probe_assign(cin, cout, mode, ksize, j)
    k = ksize if mode == 0 else 4
    xp, s, Ho, Wo = _padded(x, mode, ksize)
    ones = _padded(torch.ones_like(x[:, :1]), mode, ksize)[0]
    out = x.new_zeros(x.shape[0], cout, Ho, Wo)
    pad = torch.zeros(x.shape[0], cout, Ho, Wo, dtype=torch.bool, device=x.device)
    tap, ci = tap.to(x.device), ci.to(x.device)
    for t in range(taps(mode, ksize)):
        sel = (tap == t).nonzero().flatten()
        if sel.numel() == 0:
            continue
        ky, kx = divmod(t, k)
        if mode == 2:          # the correlation form reads the flipped kernel
            ky, kx = k - 1 - ky, k - 1 - kx
        out[:, sel] = _tap_view(xp, ky, kx, s, Ho, Wo)[:, ci[sel]]
        pad[:, sel] = (_tap_view(ones, ky, kx, s, Ho, Wo) == 0).expand(-1, sel.numel(), -1, -1)
    return out, pad


def probe_expected(r_nobias, bias):
    """Engine result of an exact accumulator: bf16_RN(float32(acc) + float32(bias))."""
    b = torch.zeros(r_nobias.shape[1], device=r_nobias.device) if bias is None else bias.float()
    return bf16(r_nobias.float() + b[None, :, None, None])


def check_probe(y, expected):
    """Bit equality; returns the number of differing elements (and the first few positions for the message)."""
    bad = y.float() != expected.float()
    return int(bad.sum()), bad.nonzero()[:8].tolist()


# ---- random weights ----------------------------------------------------------------------------------------------------------------
def acc_delta(r, rabs, K):
    """Bound on |acc + bias - r| for K fp32-accumulated exact products: K 2^-23 sum|x w| + 2^-24 |r|."""
    return K * 2.0 ** -23 * rabs + U32 * r.abs()


def element_bound(r, rabs, K, extra=None):
    """|y - r| <= 1/2 ulp_bf16(|r| + d) + d per element, d = acc_delta (+ extra, e.g. the propagated prologue error)."""
    d = acc_delta(r, rabs, K)
    if extra is not None:
        d = d + extra
    return 0.5 * ulp_bf16(r.abs() + d) + d


def check_bound(y, r, bound):
    """Returns (number of violations, max |y - r| / bound, fraction of elements with y != bf16_RN(r))."""
    err = (y.double() - r).abs()
    ratio = err / bound
    return int((err > bound).sum()), float(ratio.max()), float((y.double() != bf16(r)).double().mean())


# ---- GroupNorm prologue ------------------------------------------------------------------------------------------------------------
def prologue_ref(x, groups, gamma, beta, temb=None, silu=True):
    """fp64 a = SiLU(GroupNorm(x)) + temb and the quantities its error bound needs.  Zero padding is applied AFTER the prologue by
    the convolution (conv_ref pads a), as the engine does.  Returns (a, t, scale) where t = GroupNorm(x) (the SiLU argument) and
    scale = |gamma| (|x| + |mean|) rstd + |beta|, the magnitude the engine's fp32 affine works at."""
    x = x.double()
    B, C = x.shape[:2]
    g = x.reshape(B, groups, -1)
    mean = g.mean(-1, keepdim=True)
    rstd = (g.var(-1, unbiased=False, keepdim=True) + GN_EPS).rsqrt()
    xh = ((g - mean) * rstd).reshape(x.shape)
    gm, bt = gamma.double()[None, :, None, None], beta.double()[None, :, None, None]
    t = xh * gm + bt
    a = t * torch.sigmoid(t) if silu else t
    if temb is not None:
        a = a + temb.double()[:, :, None, None]
    scale = gm.abs() * (g.abs() + mean.abs()).reshape(x.shape) * rstd.expand_as(g).reshape(x.shape) + bt.abs()
    return a, t, scale


def prologue_error(a, t, scale, temb=None, silu=True):
    """Bound on |s - a| for the engine's fp32 prologue value s (before the bf16 rounding of the operand): the tanh.approx term
    |t / 2| 2^-11 plus 2^-16 of the magnitudes the fp32 affine, the fixed-point input statistics (sums of at most 2^16 fp32 values)
    and the temb add work at."""
    m = scale + a.abs() + (temb.double().abs()[:, :, None, None] if temb is not None else 0.0)
    e = 2.0 ** -16 * m
    if silu:
        e = e + 0.5 * t.abs() * TANH_REL
    return e


def operand_bound(a, e):
    """|bf16 operand - a| <= 1/2 ulp_bf16(|a| + e) + e."""
    return 0.5 * ulp_bf16(a.abs() + e) + e


K_SIGMA = 6.0


def prologue_sigma(e_op, w, mode, ksize):
    """Random weights after the prologue: the operand errors (each within e_op, signs and sizes independent of the weights)
    propagate as a sum with standard deviation at most sigma = sqrt(conv(e_op^2, w^2)); the gate adds K_SIGMA sigma per element."""
    return conv_ref(e_op * e_op, w.double() ** 2, None, mode, ksize).sqrt()


def probe_prologue_bound(a_shift, e_shift, bias):
    """Bound for a probe through the prologue: y = bf16_RN(operand + bias), so |y - (a + bias)| <= |operand - a| + 1/2 ulp."""
    b = bias.double()[None, :, None, None]
    eo = operand_bound(a_shift, e_shift)
    return eo + 0.5 * ulp_bf16((a_shift + b).abs() + eo) + U32 * (a_shift + b).abs()


# ---- output statistics -------------------------------------------------------------------------------------------------------------
def stats_ref(r, groups):
    """fp64 (mean, rstd) per (image, group) of the conv output r (bias included)."""
    g = r.reshape(r.shape[0], groups, -1)
    return g.mean(-1), (g.var(-1, unbiased=False) + GN_EPS).rsqrt()


def stats_bound(r, delta, groups):
    """Bounds on |mean - mean_ref| and |rstd - rstd_ref| of the engine's out_stats.

    The engine sums the fp32 values v = acc + bias (|v - r| <= delta) of each (image, group) in chunks: 16 positions of one channel
    summed in fp32 (the swapped-role epilogue adds up to 32 rows x 16-channel pieces through a butterfly; either way at most 32
    rounded adds on the path of any value), each chunk converted to 64-bit fixed point (sum x 2^24, sum of squares x 2^20, round to
    nearest) and added exactly.  gn_mean_rstd then forms m = S / n and q = Q / n in fp64, var = q - m^2, mean -> fp32 and
    rstd = rsqrtf(float(var) + eps) (2 ulp)."""
    B = r.shape[0]
    g = r.reshape(B, groups, -1)
    d = delta.expand_as(r).reshape(B, groups, -1) if torch.is_tensor(delta) else torch.full_like(g, float(delta))
    n = g.shape[-1]
    chunks = 2 * (-(-n // 16)) + 2
    a1, a2 = (g.abs() + d).sum(-1), ((g.abs() + d) ** 2).sum(-1)
    mean, rstd = stats_ref(r, groups)
    dm = (d.sum(-1) + 32 * U32 * a1 + chunks * 0.5 * 2.0 ** -24) / n + 2 * U32 * mean.abs()
    dq = ((2 * g.abs() * d + d * d).sum(-1) + 34 * U32 * a2 + chunks * 0.5 * 2.0 ** -20) / n
    var = g.var(-1, unbiased=False)
    dv = dq + 2 * mean.abs() * dm + dm * dm
    lo = (var - dv).clamp_min(0) + GN_EPS
    drstd = (lo.rsqrt() - rstd).abs() + (var + dv + GN_EPS).rsqrt().sub(rstd).abs() + 6 * U32 * lo.rsqrt()
    return mean, rstd, dm, drstd


def check_stats(st, r, delta, groups):
    """st: engine out_stats [B][groups][2] (mean, rstd).  Returns (violations, max err/bound of mean, of rstd)."""
    mean, rstd, dm, dr = stats_bound(r, delta, groups)
    em = (st[..., 0].double() - mean).abs()
    er = (st[..., 1].double() - rstd).abs()
    return int((em > dm).sum() + (er > dr).sum()), float((em / dm).max()), float((er / dr).max())

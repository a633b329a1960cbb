"""fp64 references and element-wise checkers for the launches of a DDPM step outside the 3x3 / 1x1 / k4s2 convolutions and the fused
attention blocks: the 7x7 stem, the GroupNorm finalize and the final_conv tail with and without the fused DDPM update (plain torch,
any device, no engine imports).  Each mirror rounds where the kernel rounds and each bound is derived from the kernel's arithmetic:

  * stem (conv_tcgen05_kernel<GEO_INIT>): the producer rounds the fp32 state to bf16 (pack8), the weights are bf16, the tensor core
    accumulates exact products in fp32, the epilogue adds the bias, then the class row, in fp32 and rounds once to bf16.  The CUDA-core
    stem (init_conv_kernel) multiplies the fp32 state and fp32 weights in a sequential fmaf chain and adds (bias + class row) at once;
  * gn_finalize_kernel: mean / rstd from the fixed-point sums exactly as gn_mean_rstd, t = fmaf(v, rstd gamma, beta - mean rstd gamma),
    SiLU (silu_fast: tanh.approx, or silu_f: __expf and an IEEE divide), + residual, one rounding to the activation type; the output
    statistics are per-thread fp32 sums of the values before that rounding, one fixed-point integer atomic per warp class;
  * final_proj*_kernel: the same affine and SiLU per channel, then a sequential per-pixel fmaf chain over the C channels, + bias;
  * final_proj_ddpm_kernel: that eps (never stored), x0 = clamp(c0 x - c1 eps), x_{t-1} = c2 x0 + c3 x + c4 z in fp32.
"""
import torch

from conv_ref import GN_EPS, TANH_REL, U32, acc_delta, bf16, conv_ref, element_bound, ulp_bf16

STAT_SUM, STAT_SQ = 2.0 ** 24, 2.0 ** 20       # common.cuh kStatScaleSum / kStatScaleSq
# rstd = rsqrtf(float(var) + eps): rsqrtf is within 2 ulp (CUDA C Programming Guide, single-precision intrinsics table), and a fused
# q - m*m may move float(var) by one ulp against the mirror's unfused double expression: 2 * 2^-23 + 2^-24 <= 2^-21 relative.
RSQRT_REL = 2.0 ** -21
# the kernel's Philox normals against tests/philox_ref.py (fast-math log / sincos): the gate tests/test_gpu_philox.py holds them to
PHILOX_ABS = 1e-3


def f32(t):
    return t.float().double()


# ---- 7x7 stem ---------------------------------------------------------------------------------------------------------------------
def stem_operands(x, w, tc):
    """(operand, weights) the stem multiplies: bf16-rounded on the tensor-core stem, as given on the CUDA-core stem."""
    return (bf16(x.float()).double(), bf16(w.float()).double()) if tc else (x.double(), w.double())


def stem_epilogue(acc, bias, cls, tc, out_bf16=True):
    """The stem's output from an fp32 accumulator value acc [B][Cout][S][S] (fp32-representable): tensor core (acc + bias) + cls,
    CUDA cores acc + (bias + cls), each add in fp32, then bf16_RN.  cls: [B][Cout] class rows per sample, or None."""
    a = acc.float()
    b = torch.zeros(acc.shape[1], device=acc.device) if bias is None else bias.float()
    if tc:
        v = a + b[None, :, None, None]
        if cls is not None:
            v = v + cls.float()[:, :, None, None]
    else:
        base = b[None, :] + cls.float() if cls is not None else b[None, :].expand(acc.shape[0], -1)
        v = a + base[:, :, None, None]
    return bf16(v) if out_bf16 else v


def stem_ref(x, w, bias, cls, tc):
    """fp64 y = conv7x7(operands) + bias + cls and sum |x w| (for the accumulation bound)."""
    xo, wo = stem_operands(x, w, tc)
    r = conv_ref(xo, wo, bias, 0, 7)
    if cls is not None:
        r = r + cls.double()[:, :, None, None]
    return r, conv_ref(xo.abs(), wo.abs(), None, 0, 7)


def stem_bound(r, rabs, cin):
    """Random weights: K = 49 Cin exact products accumulated in fp32 (conv_ref.acc_delta covers the bias add), one more fp32 add for
    the class row, one bf16 rounding."""
    return element_bound(r, rabs, 49 * cin, U32 * r.abs())


# ---- GroupNorm statistics in the engine's fixed-point format ----------------------------------------------------------------------
def fixed_stats(x, groups):
    """int64 [B][groups][2] = {round(sum 2^24), round(sum of squares 2^20)} of x [B][C][...] per (sample, group): what the engine's
    integer atomics would hold with no fp32 rounding at all."""
    g = x.double().reshape(x.shape[0], groups, -1)
    return torch.stack([torch.round(g.sum(-1) * STAT_SUM), torch.round((g * g).sum(-1) * STAT_SQ)], -1).to(torch.int64)


def mean_rstd(stats, count):
    """gn_mean_rstd: m = S 2^-24 inv, q = Q 2^-20 inv in double with inv = 1.f / count in fp32, var = max(q - m^2, 0),
    mean = float(m), rstd = rsqrt(float(var) + eps) (here exact on the fp32 argument; RSQRT_REL covers rsqrtf)."""
    inv = float(torch.tensor(1.0, dtype=torch.float32) / torch.tensor(float(count), dtype=torch.float32))
    m = stats[..., 0].double() * (1.0 / STAT_SUM) * inv
    q = stats[..., 1].double() * (1.0 / STAT_SQ) * inv
    var = (q - m * m).clamp_min(0)
    arg = var.float() + torch.tensor(GN_EPS, dtype=torch.float32)
    return f32(m), arg.double().rsqrt()


def _per_channel(v, C):
    """[B][G] -> [B][C][1] (channel c belongs to group c // (C / G))."""
    return v.repeat_interleave(C // v.shape[1], dim=1)[:, :, None]


def norm_silu(v, stats, groups, gamma, beta, silu, fast):
    """fp64 a = act(GroupNorm(v) gamma + beta) of v [B][C][HW] from the kernel's own statistics, and the bound on |a_kernel - a| for
    the kernel's fp32 evaluation (before any later rounding).  fast: silu_fast (bf16 kernels) or silu_f (fp32 kernels)."""
    B, C, HW = v.shape
    mean, rstd = mean_rstd(stats, HW * (C // groups))
    mean, rstd = _per_channel(mean, C), _per_channel(rstd, C)
    sc = rstd * gamma.double()[None, :, None]
    bt = beta.double()[None, :, None]
    v = v.double()
    t = (v - mean) * sc + bt
    # sc = fl(rstd gamma) (RSQRT_REL + u), sh = beta - mean sc (one or two roundings), t = fmaf(v, sc, sh) (one rounding)
    e_t = (RSQRT_REL + 2 * U32) * (v - mean).abs() * sc.abs() + 2 * U32 * (bt.abs() + (mean * sc).abs()) + 2 * U32 * t.abs()
    if not silu:
        return t, e_t
    a = t * torch.sigmoid(t)
    # |silu'| <= 1.1 carries e_t; silu_fast = fmaf(h, tanh.approx(h), h), h = t / 2: |h tanh h| 2^-11 + one rounding;
    # silu_f = t / (1 + __expf(-t)): __expf within 2 + floor(1.173 |t|) ulp, one add, one IEEE divide
    if fast:
        e = 1.1 * e_t + 0.5 * t.abs() * TANH_REL + U32 * a.abs()
    else:
        e = 1.1 * e_t + ((3.0 + 1.2 * t.abs()) * 2.0 ** -23 + 3 * U32) * a.abs()
    return a, e


# ---- gn_finalize ------------------------------------------------------------------------------------------------------------------
def finalize_ref(raw, res, stats, groups, gamma, beta, silu, bf16_out):
    """fp64 mirror o [B][C][HW] of gn_finalize, the bound d on |fp32 value - o| before the store, and the element bound of the
    stored value (bf16: + 1/2 ulp at |o| + d; fp32: the residual add is the last rounding and is in d)."""
    a, e = norm_silu(raw, stats, groups, gamma, beta, silu, fast=bf16_out)
    o = a + (res.double() if res is not None else 0.0)
    d = e + (U32 * (o.abs() + e) if res is not None else 0.0)
    bound = 0.5 * ulp_bf16(o.abs() + d) + d if bf16_out else d
    return o, d, bound


def finalize_geometry(B, HW, C, groups, act_bf16, ogroups):
    """gn_finalize's launch: vector width V, blocks per image, the most fp32 terms one thread sums and the most integer atomics per
    (sample, output group) -- one per warp class per block (8 warps)."""
    V = 8 if act_bf16 else 4
    if V == 8 and ((C // groups) % 8 or (ogroups and (C // ogroups) % 8) or 256 % (C // 8)):
        V = 4
    items = HW * (C // V)
    bpi = min(max(-(-items // (256 * 8)), 1), 64)
    per_thread = V * -(-items // (bpi * 256))
    return V, bpi, per_thread, 8 * bpi


def out_stats_ref(o, d, ogroups, per_thread, n_atomics):
    """Expected fixed-point output sums (S, Q) per (sample, output group) in the engine's units and their bounds: the fp32 values
    differ from o by at most d; a thread adds up to per_thread of them in fp32 and a warp butterfly adds 5 more levels
    ((per_thread + 5) u per term, one more u for the square); each atomic rounds its scaled sum to an integer (1/2 unit)."""
    B = o.shape[0]
    g, dg = o.reshape(B, ogroups, -1), d.expand_as(o).reshape(B, ogroups, -1)
    ab = g.abs() + dg
    S = g.sum(-1) * STAT_SUM
    Q = (g * g).sum(-1) * STAT_SQ
    k = per_thread + 5
    dS = STAT_SUM * (dg.sum(-1) + k * U32 * ab.sum(-1)) + 0.5 * n_atomics
    dQ = STAT_SQ * ((2 * g.abs() * dg + dg * dg).sum(-1) + (k + 1) * U32 * (ab * ab).sum(-1)) + 0.5 * n_atomics
    return S, Q, dS, dQ


def check_out_stats(st, S, Q, dS, dQ):
    """st: int64 [B][G][2] kernel sums.  Returns (violations, max err / bound of the sums, of the sums of squares)."""
    eS = (st[..., 0].double() - S).abs()
    eQ = (st[..., 1].double() - Q).abs()
    return int((eS > dS).sum() + (eQ > dQ).sum()), float((eS / dS).max()), float((eQ / dQ).max())


# ---- final projection -------------------------------------------------------------------------------------------------------------
def proj_ref(y, stats, groups, gamma, beta, w, bias, plain, fast):
    """fp64 eps [B][Cout][HW] of final_proj from y [B][C][HW] and the bound on |eps_kernel - eps|: the sequential fmaf chain over
    K = C channels (conv_ref.acc_delta, which also covers the bias add) plus the propagated affine / SiLU error sum_c |w| e_a."""
    if plain:
        a, e = y.double(), torch.zeros_like(y, dtype=torch.float64)
    else:
        a, e = norm_silu(y, stats, groups, gamma, beta, True, fast)
    wd = w.double()
    eps = torch.einsum("bcp,oc->bop", a, wd)
    if bias is not None:
        eps = eps + bias.double()[None, :, None]
    rabs = torch.einsum("bcp,oc->bop", a.abs() + e, wd.abs())
    return eps, acc_delta(eps, rabs, y.shape[1]) + torch.einsum("bcp,oc->bop", e, wd.abs())


# ---- fused DDPM tail --------------------------------------------------------------------------------------------------------------
def ddpm_ref(x, eps, e_eps, z, e_z, row):
    """fp64 x_{t-1} of ddpm_step_kernel / final_proj_ddpm_kernel and its bound.  row: the fp32 coefficient row {c0, c1, c2, c3, c4,
    pred_x0}.  Each fp32 expression a p + b q rounds once or twice (FMA contraction), 2u |terms|; the clamp is monotone: an x0 within
    e of the mirror's clamps into [clamp(x0 - e), clamp(x0 + e)] (0 error where both ends clamp)."""
    c0, c1, c2, c3, c4, flag = (float(v) for v in row[:6])
    x, eps = x.double(), eps.double()
    if flag != 0.0:
        x0, e0 = eps, e_eps
    else:
        x0 = c0 * x - c1 * eps
        e0 = abs(c1) * e_eps + 2 * U32 * ((c0 * x).abs() + (c1 * eps).abs())
    x0c = x0.clamp(-1, 1)
    ec = torch.maximum((x0 + e0).clamp(-1, 1) - x0c, x0c - (x0 - e0).clamp(-1, 1))
    mean = c2 * x0c + c3 * x
    em = abs(c2) * ec + 2 * U32 * ((c2 * x0c).abs() + (c3 * x).abs()) + U32 * abs(c2) * ec
    zt = torch.zeros_like(x) if z is None else z.double()
    o = mean + c4 * zt
    eo = em + abs(c4) * e_z + 2 * U32 * (mean.abs() + em + (c4 * zt).abs())
    return o, eo


def check_bound(y, r, bound):
    """(violations, max |y - r| / bound)."""
    ratio = (y.double() - r).abs() / bound
    return int((ratio > 1).sum()), float(ratio.max())

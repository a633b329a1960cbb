"""fp64 mirror of the time-embedding table and of the FiLM positional-encoding table, with an element-wise bound derived from the
kernels' fp32 arithmetic (plain torch, any device, no engine imports).

  * time_table (kernels_simt.cu): sinusoid_kernel takes the fp32 product times[r] * freqs[k] -- the same rounding the reference's
    torch ops make -- then sinf | cosf of it; three rows_linear_kernel launches follow, each a sequential fmaf chain over K inputs
    from 0, + bias in fp32, then GELU(erf) (time_mlp.1), SiLU (time_mlp.3, the SiLU the blocks' mlp starts with) or nothing (all
    ResnetBlock mlp.1 projections side by side, one fp32 row of sumC columns per time value);
  * film_pe_kernel: a = (5000 * level) * freq with a rounding after each product, then sinf or cosf per the column's is_cos flag.

The bound of a layer output is carried from its inputs: a K-term fmaf chain is within gamma_K sum |a_k w_kn| of the exact sum of its
fp32 operands, the input error enters as sum |w_kn| e_k, the bias add rounds once, GELU and SiLU pass an input error on with their
Lipschitz constants and add their own evaluation error (erff / expf / sinf / cosf within the documented ulp maxima of the CUDA C
Programming Guide's single-precision function table, IEEE divide).
"""
import math

import torch

U32 = 2.0 ** -24          # fp32 unit roundoff
SINCOS_ULP = 2            # sinf, cosf: 2 ulp over the whole range
ERF_ULP = 2               # erff
EXP_ULP = 2               # expf
GELU_LIP = 1.13           # max |GELU'(x)| = 1.1289 (x = sqrt(2))
SILU_LIP = 1.1            # max |SiLU'(x)| = 1.0998 (x = 2.3994)
FILM_SCALE = 5000.0       # parts/film.py: FILM_LINEAR_SCALE


def gamma(k):
    return k * U32 / (1 - k * U32)


def ulp32(v):
    """Spacing of the fp32 numbers at |v| (the subnormal spacing below 2^-126)."""
    _, e = torch.frexp(v.double().abs().clamp_min(2.0 ** -126))
    return torch.ldexp(torch.ones_like(v, dtype=torch.float64), e - 24)


def _sincos_bound(v):
    # SINCOS_ULP ulp of the exact value, + 1/2 ulp so the bound also holds at a power of two the result rounds onto
    return (SINCOS_ULP + 0.5) * ulp32(v)


# ---- time embedding ---------------------------------------------------------------------------------------------------------------
def sinusoid(times, freqs):
    """[R][dim] = [sin | cos](fp32(times[r] * freqs[k])) in fp64, and the bound of sinf / cosf."""
    a = (times.float()[:, None] * freqs.float()[None, :]).double()
    e = torch.cat([a.sin(), a.cos()], 1)
    return e, _sincos_bound(e)


def linear(a, ea, w, b):
    """rows_linear_kernel without activation: fp64 y = a w^T + b for w [N][K] (torch layout) and the bound on the kernel's fp32 y
    when its inputs are within ea of a."""
    wd, wa = w.double(), w.double().abs()
    y = a @ wd.T + b.double()
    d = ea @ wa.T + gamma(w.shape[1]) * ((a.abs() + ea) @ wa.T)     # input error + the K roundings of the fmaf chain
    return y, d + U32 * (y.abs() + d)                                # + bias, one rounding


def gelu(h, eh):
    """acc = 0.5f * acc * (1 + erff(acc * 0.70710678f)): the argument rounds twice (the constant and the product), erff within
    ERF_ULP ulp of a value below 1, the add and the last product round once each; 0.5 * acc is exact."""
    z = h / math.sqrt(2.0)
    er = torch.erf(z)
    g = 0.5 * h * (1 + er)
    ha = h.abs() + eh
    e_one = (2 / math.sqrt(math.pi)) * 2 * U32 * ha / math.sqrt(2.0) + ERF_ULP * 2.0 ** -23 + U32 * (1 + er.abs())
    return g, GELU_LIP * eh + 0.5 * ha * e_one + U32 * (g.abs() + GELU_LIP * eh)


def silu(t, et):
    """acc / (1 + expf(-acc)): expf within EXP_ULP ulp, one rounding for the add, one for the IEEE divide."""
    s = t * torch.sigmoid(t)
    return s, SILU_LIP * et + (EXP_ULP * 2.0 ** -23 + 3 * U32) * (s.abs() + SILU_LIP * et)


def block_projection(sd, cols, sum_c):
    """The [sumC][4 dim] weight and [sumC] bias of the concatenated ResnetBlock mlp.1 projections: cols maps each block prefix
    ('downs.0.0', ...) to its first table column."""
    td = sd["time_mlp.3.weight"].shape[0]
    w = torch.full((sum_c, td), float("nan"))
    b = torch.full((sum_c,), float("nan"))
    for p, c in cols.items():
        wb = sd[p + ".mlp.1.weight"]
        w[c:c + wb.shape[0]] = wb
        b[c:c + wb.shape[0]] = sd[p + ".mlp.1.bias"]
    assert not torch.isnan(w).any(), "the block slices do not tile [0, sumC)"
    return w, b


def time_table_ref(times, freqs, sd, cols, sum_c):
    """fp64 table [R][sumC] of time_table for the fp32 times [R] and the element bound of the kernel's fp32 table."""
    e, ee = sinusoid(times, freqs)
    h, eh = linear(e, ee, sd["time_mlp.1.weight"], sd["time_mlp.1.bias"])
    g, eg = gelu(h, eh)
    t, et = linear(g, eg, sd["time_mlp.3.weight"], sd["time_mlp.3.bias"])
    s, es = silu(t, et)
    w, b = block_projection(sd, cols, sum_c)
    return linear(s, es, w, b)


# ---- FiLM positional encoding -----------------------------------------------------------------------------------------------------
def film_columns(channels):
    """Per-column (freq, is_cos) of the FiLM table: for each layer of C channels [exponents | exponents] with
    exponents = 1e-4 ** (arange(C/2) / (C/2)) in fp32 (parts/film.py:19-21), sin in the first half, cos in the second."""
    freq, is_cos = [], []
    for c in channels:
        half = c // 2
        ex = 1e-4 ** (torch.arange(half, dtype=torch.float32) / float(half))
        freq += [ex, ex]
        is_cos += [torch.zeros(half, dtype=torch.bool), torch.ones(half, dtype=torch.bool)]
    return torch.cat(freq), torch.cat(is_cos)


def film_table_ref(levels, freq, is_cos):
    """fp64 [R][sumC] of film_pe_kernel for fp32 noise levels [R] and the bound of sinf / cosf."""
    a = ((torch.tensor(FILM_SCALE, dtype=torch.float32) * levels.float())[:, None] * freq.float()[None, :]).double()
    v = torch.where(is_cos[None, :], a.cos(), a.sin())
    return v, _sincos_bound(v)


def check_bound(y, r, bound):
    """(violations, max |y - r| / bound)."""
    ratio = (y.double() - r).abs() / bound
    return int((ratio > 1).sum()), float(ratio.max())

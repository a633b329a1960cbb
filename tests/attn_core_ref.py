"""Reference and error bound of the bf16 softmax-attention core above 64 tokens (attn_flash_kernel, csrc/attn_fused.cu), plus a
float32 CPU model of that kernel with switchable defects for the host tests of the checker.

Layout: qkv [B][N][384] (channel = which * 128 + head * 32 + d), o [B][N][128] (channel = head * 32 + e), as attn_core sees them.

Bound of one output element o[b][i][h][e] (derived from the kernel's rounding points; w_j = exact softmax weights of row i):
  * each weight the kernel uses is p~_j = p_j (1 + delta_j) with
      |delta_j| <= 2^-9                              bf16 rounding of P (l sums the ROUNDED P, so numerator and denominator agree)
                 + (T + 1) 2^-21                     ex2.approx of P and of the T rescale factors
                 + ln 2 * dz_j                       the exponent argument z_j = s_j * scale * log2 e - m:
      dz_j <= 2 * 32 * 2^-24 * c * sum_d |q_d k_d|   fp32 K = 32 product of the tensor core (with a factor 2 for its internal order)
              + 4 * 2^-24 * (|z_j| + |m|)            fp32 roundings of the scale, of the running max and of the fmaf
    then sum_j (w~_j - w_j) v_j = sum_j w_j (delta_j - delta_bar) / (1 + delta_bar) (v_j - o_i), which is bounded by
      [sum_j w_j (|delta_j| + delta_max) (|v_j| + |o_i|)] / (1 - delta_max);
  * fp32 accumulation of O over N keys and of l, the T rescales and the final 1 / l: (N + 2T + 4) 2^-23 sum_j w_j |v_j|;
  * the bf16 store: half an ulp, at most 2^-8 (|o| + the error before rounding).
"""
import math

import torch

LOG2E = 1.0 / math.log(2.0)
SCALE = 32 ** -0.5
U24 = 2.0 ** -24


def bf16(t):
    return t.to(torch.bfloat16).to(t.dtype)


def split(qkv):
    """[B][N][384] -> q, k, v as [B][4][N][32]."""
    b, n, _ = qkv.shape
    return [qkv[..., w * 128:(w + 1) * 128].reshape(b, n, 4, 32).permute(0, 2, 1, 3) for w in range(3)]


def merge(o):
    """[B][4][N][32] -> [B][N][128]."""
    b, _, n, _ = o.shape
    return o.permute(0, 2, 1, 3).reshape(b, n, 128)


def exact_and_bound(qkv, chunk_elems=1 << 26):
    """float64 exact core output and the per-element bound (both [B][N][128]) on qkv's device, images in chunks."""
    outs, bounds = [], []
    b, n, _ = qkv.shape
    T = (n + 127) // 128
    c = SCALE * LOG2E
    step = max(1, chunk_elems // (4 * n * n))
    for b0 in range(0, b, step):
        q, k, v = [t.double() for t in split(qkv[b0:b0 + step])]
        s = q @ k.transpose(-1, -2)                                          # [b][4][N][N]
        z = s * c
        m = z.amax(-1, keepdim=True)
        w = torch.exp2(z - m)
        w = w / w.sum(-1, keepdim=True)
        o = w @ v
        dz = 2 * 32 * U24 * c * (q.abs() @ k.abs().transpose(-1, -2)) + 4 * U24 * (z.abs() + m.abs())
        delta = 2.0 ** -9 + (T + 1) * 2.0 ** -21 + math.log(2.0) * dz
        dmax = delta.amax(-1, keepdim=True)
        wd = w * (delta + dmax)
        err = (wd @ v.abs() + o.abs() * wd.sum(-1, keepdim=True)) / (1 - dmax)
        err = err + (n + 2 * T + 4) * 2.0 ** -23 * (w @ v.abs())
        bound = err + 2.0 ** -8 * (o.abs() + err)
        outs.append(merge(o))
        bounds.append(merge(bound))
        del s, z, w, dz, delta, wd
    return torch.cat(outs), torch.cat(bounds)


def check(got, exact, bound):
    """(max |got - exact| / bound, index of the worst element) over [B][N][128]."""
    r = (got.double() - exact).abs() / bound
    i = int(r.argmax())
    return float(r.flatten()[i]), i


def make_inputs(b, n, negative=False, seed=0, device="cpu"):
    """bf16-valued qkv [B][N][384] that make defects of the core visible:
      * every image has its own scale (0.5 .. 2) of q;
      * logits of several units;
      * a key ramp along a direction u that q sees positively: the logits grow along the tokens, so the running max moves on
        later tiles (the rescale path);
      * head 2 has three times the logit scale of the others (and its own direction), so a head mix-up is visible;
      * negative=True: every real logit is strongly negative (about -12 natural units), so an unmasked zero-padded key of a ragged
        tile (logit 0) would take almost all of the weight."""
    g = torch.Generator(device=device).manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, device=device)      # noqa: E731
    q, k, v = r(b, 4, n, 32), r(b, 4, n, 32), r(b, 4, n, 32)
    u = r(4, 32)
    u = u / u.norm(dim=-1, keepdim=True)
    ramp = torch.linspace(0, 3, n, device=device)
    if negative:
        q = 0.3 * q + 4.0 * u[None, :, None, :]          # q . k about -72, times 32^-0.5: about -12.7
        k = 0.3 * k - 18.0 * u[None, :, None, :]
    else:
        q = q + 1.5 * u[None, :, None, :]
        k = k + ramp[None, None, :, None] * u[None, :, None, :]
    img = torch.arange(b, device=device)
    q = q * (2.0 ** (((img * 5) % 9).float() / 4 - 1))[:, None, None, None]
    q[:, 2] = q[:, 2] * 3.0
    qkv = torch.cat([merge(q), merge(k), merge(v)], -1)
    return bf16(qkv.float())


def model_flash(qkv, defect=None):
    """float32 CPU model of attn_flash_kernel's arithmetic (128-key tiles, running max in the log2 domain, bf16 P, rescale of O
    when the max moves, l over the rounded P).  defect: None | "unmasked_pad" (padded keys of the last tile take part with logit 0
    and v = 0) | "skip_rescale" (O is not rescaled when the max moves) | "neighbour_row" (query row 0 of every image but the last
    uses the next image's q) | "swap_heads" (heads 0 and 1 of the output exchanged)."""
    q, k, v = [t.float() for t in split(qkv)]
    b, _, n, _ = q.shape
    if defect == "neighbour_row" and b > 1:
        q = q.clone()
        q[:-1, :, 0] = q[1:, :, 0]
    c = torch.tensor(SCALE * LOG2E, dtype=torch.float32)
    T = (n + 127) // 128
    m = torch.full((b, 4, n, 1), -math.inf)
    l = torch.zeros(b, 4, n, 1)
    o = torch.zeros(b, 4, n, 32)
    for j in range(T):
        kj, vj = k[:, :, j * 128:(j + 1) * 128], v[:, :, j * 128:(j + 1) * 128]
        nv = kj.shape[2]
        s = q @ kj.transpose(-1, -2)
        if defect == "unmasked_pad" and nv < 128:
            s = torch.cat([s, s.new_zeros(b, 4, n, 128 - nv)], -1)
            vj = torch.cat([vj, vj.new_zeros(b, 4, 128 - nv, 32)], 2)
        m_new = torch.maximum(m, s.amax(-1, keepdim=True) * c)
        corr = torch.exp2(m - m_new)
        p = bf16(torch.exp2(s * c - m_new))
        l = l * corr + p.sum(-1, keepdim=True)
        o = (o if defect == "skip_rescale" else o * corr) + p @ vj
        m = m_new
    o = o / l
    if defect == "swap_heads":
        o = o[:, [1, 0, 2, 3]]
    return bf16(merge(o))

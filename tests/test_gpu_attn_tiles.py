"""Both fused attention kernels of csrc/attn_fused.cu, element by element, at every (softmax, tokens, channels) shape and images-per-CTA
regime the production plans launch.

tests/test_gpu_attn_fused.py compares the blocks with the fp32 oracle at rel-L2 <= 2e-2 on small batches.  Here each case is one
fused-attention launch of a production plan -- configs[1] (3x32x32, dim 128, mults 1,2,2,2) at B = 256 and at the guidance-doubled
B = 512 (2 to 4 images per CTA), configs[2] (64x64, learned variance) at B = 128 (linear attention at N = 4096: 32 tiles of the online
k softmax) -- plus edge batches: one image, fewer images than SMs, exactly one CTA with two images (B = 149), 300 images at 4x4.
The inputs are built to make kernel defects visible (tests/attn_ref.py holds the references):

  * every image has its own scale and offset, so its PreNorm statistics differ from every other image's;
  * to_qkv is scaled (k logits of several units) and a token ramp along one input direction that only the k rows see moves the
    running k maximum on most tiles (ramp up), on none after tile 0 (ramp down), or in one head only (the per-warp rescale);
  * one case shifts to_out.0.bias so that mean / std of y is about 8 (the bf16 parking of y in front of GroupNorm(1) matters).

Checks per case, image by image: the largest |kernel - mirror| in bf16 ulps (at the element's magnitude, or the image's attention
branch rms where that is larger), the share of elements that differ from bf16_RN(mirror), and the attention branch out - x against
the exact block within the bound derived from the mirror's rounding points.  Padded token rows and columns of the 4x4 and 8x8 maps
(one zero-padded 128-token tile per image) must not reach any image's output or statistics, which the per-image comparison sees.
The references run on the GPU in float64.  Production defaults: no DMN_* switch is set.
"""
import pytest
import torch

from conftest import make_unet
from gpu_helpers import linear_attention_block
from oracle import ref_port as O
import attn_ref as A

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Gates per kernel (False: linear, True: softmax), at twice the largest value measured over all cases on a B200 (the per-case values
# are printed by the coverage test): linear 5.06 ulps and a share of 0.079, softmax 6.94 ulps and a share of 0.19.  The remaining
# differences from the mirror are fp32 accumulation order, ex2.approx and rounding-boundary flips of the bf16 intermediates (the
# softmax kernel's P and o flip more often: its logits of several units come out of a K = 32 fp32 product).
ULP_GATE = {False: 10.0, True: 14.0}     # max |kernel - mirror| / ulp_bf16(magnitude of the element, see run_case)
FRAC_GATE = {False: 0.16, True: 0.38}    # share of an image's elements != bf16_RN(mirror)

# (name, softmax, H, C, B, inputs): "mixed" = per-image scale / offset and ramps cycling up, down, none; "head" = the k maximum
# moves in one head only; "shift" = mixed, with mean / std of y about 8
CASES = [
    ("cfg1_lin_1024x128_b256", False, 32, 128, 256, "mixed"),
    ("cfg1_lin_256x256_b256", False, 16, 256, 256, "mixed"),
    ("cfg1_lin_64x256_b256", False, 8, 256, 256, "mixed"),
    ("cfg1_lin_16x256_b256", False, 4, 256, 256, "mixed"),
    ("cfg1_lin_256x128_b256", False, 16, 128, 256, "mixed"),
    ("cfg1_soft_16x256_b256", True, 4, 256, 256, "mixed"),
    ("cfg1_lin_1024x128_b512", False, 32, 128, 512, "mixed"),
    ("cfg1_lin_256x256_b512", False, 16, 256, 512, "mixed"),
    ("cfg1_lin_64x256_b512", False, 8, 256, 512, "mixed"),
    ("cfg1_lin_16x256_b512", False, 4, 256, 512, "mixed"),
    ("cfg1_lin_256x128_b512", False, 16, 128, 512, "mixed"),
    ("cfg1_soft_16x256_b512", True, 4, 256, 512, "mixed"),
    ("cfg2_lin_4096x128_b128", False, 64, 128, 128, "mixed"),
    ("cfg2_lin_1024x256_b128", False, 32, 256, 128, "mixed"),
    ("cfg2_lin_256x256_b128", False, 16, 256, 128, "mixed"),
    ("cfg2_lin_64x256_b128", False, 8, 256, 128, "mixed"),
    ("cfg2_lin_1024x128_b128", False, 32, 128, 128, "mixed"),
    ("cfg2_soft_64x256_b128", True, 8, 256, 128, "mixed"),
    ("edge_lin_4096x128_b1", False, 64, 128, 1, "mixed"),
    ("edge_lin_16x256_b1", False, 4, 256, 1, "mixed"),
    ("edge_soft_16x256_b1", True, 4, 256, 1, "mixed"),
    ("edge_lin_1024x128_b37", False, 32, 128, 37, "mixed"),
    ("edge_soft_64x256_b37", True, 8, 256, 37, "mixed"),
    ("edge_lin_256x256_b149", False, 16, 256, 149, "mixed"),
    ("edge_lin_16x256_b149", False, 4, 256, 149, "mixed"),
    ("edge_soft_16x256_b149", True, 4, 256, 149, "mixed"),
    ("edge_lin_16x256_b300", False, 4, 256, 300, "mixed"),
    ("edge_soft_16x256_b300", True, 4, 256, 300, "mixed"),
    ("head_lin_4096x128_b4", False, 64, 128, 4, "head"),
    ("head_lin_1024x256_b8", False, 32, 256, 8, "head"),
    ("shift_lin_1024x128_b16", False, 32, 128, 16, "shift"),
    ("shift_lin_64x256_b16", False, 8, 256, 16, "shift"),
]
CASE_BY_NAME = {c[0]: c for c in CASES}
RESULTS = {}        # case name -> (key, slack dict), printed by the coverage test
QKV_GAIN = {False: 6.0, True: 3.0}      # k logits of several units (linear block), q . k / sqrt(32) of order several (softmax block)
RAMP_K = 10.0       # amplitude of the token ramp in the k logits (natural units)
RAMP_HEAD = 2


def _g(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _params(c, softmax, seed):
    g = _g(seed)
    u = lambda *s, fan: (torch.rand(*s, device=DEV, generator=g) * 2 - 1) / fan ** 0.5      # noqa: E731
    p = "blk"
    sd = {p + ".fn.norm.weight": 1 + 0.1 * torch.randn(c, device=DEV, generator=g),
          p + ".fn.norm.bias": 0.1 * torch.randn(c, device=DEV, generator=g),
          p + ".fn.fn.to_qkv.weight": u(384, c, 1, 1, fan=c) * QKV_GAIN[softmax]}
    out = p + (".fn.fn.to_out" if softmax else ".fn.fn.to_out.0")
    sd[out + ".weight"] = u(c, 128, 1, 1, fan=128)
    sd[out + ".bias"] = 0.05 * torch.randn(c, device=DEV, generator=g)
    if not softmax:
        sd[p + ".fn.fn.to_out.1.weight"] = 1 + 0.1 * torch.randn(c, device=DEV, generator=g)
        sd[p + ".fn.fn.to_out.1.bias"] = 0.1 * torch.randn(c, device=DEV, generator=g)
    return p, sd


def _inputs(case, seed=0):
    """(prefix, state dict, bf16-valued x NCHW fp32, ramp sign per image)."""
    name, softmax, h, c, b, kind = case
    p, sd = _params(c, softmax, seed)
    g = _g(seed + 1)
    n = h * h
    # a unit input direction a that the k rows of to_qkv see with gain gamma_ch (+ on every channel, or + on one head and - on the
    # others): a ramp r(n) a over the tokens moves every k logit of the image by gamma_ch * beta * r(n)
    a = torch.randn(c, device=DEV, generator=g)
    a = a / a.norm()
    beta = 8.0
    gam = torch.full((128,), RAMP_K / beta, device=DEV)
    if kind == "head":
        gam = -gam
        gam[RAMP_HEAD * 32:(RAMP_HEAD + 1) * 32] *= -1
    w = sd[p + ".fn.fn.to_qkv.weight"].reshape(384, c)
    w[128:256] += gam[:, None] * a[None, :] / sd[p + ".fn.norm.weight"][None, :]
    sd[p + ".fn.fn.to_qkv.weight"] = w.reshape(384, c, 1, 1)
    idx = torch.arange(b, device=DEV)
    scale = 2.0 ** (((idx * 5) % 9).double() / 4 - 1)          # 0.5 .. 2
    offset = ((idx * 7) % 9).double() / 4 - 1                 # -1 .. 1
    sign = torch.ones(b, device=DEV) if kind == "head" else torch.tensor([1.0, -1.0, 0.0], device=DEV)[idx % 3]
    r = torch.linspace(-1, 1, n, device=DEV)
    z = torch.randn(b, c, n, device=DEV, generator=g) + beta * sign[:, None, None] * r[None, None, :] * a[None, :, None]
    x = A.bf16((z * scale[:, None, None].float() + offset[:, None, None].float()).reshape(b, c, h, h))
    if kind == "shift":      # to_out.0.bias + 8 std(y): mean / std of y about 8
        y = A.linear_exact_y(A.operands(x[:8], sd, p))
        sd[p + ".fn.fn.to_out.0.bias"] = sd[p + ".fn.fn.to_out.0.bias"] + 8.0 * float(y.std((1, 2), unbiased=False).mean())
    return p, sd, x, sign


def run_case(case, nsm):
    name, softmax, h, c, b, kind = case
    p, sd, x, sign = _inputs(case)
    out = A.to_tokens(linear_attention_block(x, sd, p, softmax=softmax)).double()
    ops = A.operands(x, sd, p, softmax)
    st = {}
    mir = A.softmax_mirror(ops) if softmax else A.linear_mirror(ops, stats=st)
    ex = A.exact(ops, softmax)
    assert torch.isfinite(out).all(), f"{name}: non-finite output"
    B = b
    # ---- against the mirror, per element and per image: ulps at the larger of the element's magnitude, the image's branch rms and
    # (linear block) the magnitude at which the parked bf16 y reaches the output ----
    br_rms = (mir - ops.x).reshape(B, -1).pow(2).mean(1).sqrt()
    mag = torch.maximum(mir.abs(), br_rms[:, None, None])
    if not softmax:
        mag = torch.maximum(mag, st["y_scale"])
    ulp = A.ulp_bf16(mag)
    ulps = ((out - mir).abs() / ulp).reshape(B, -1).amax(1)
    frac = (out != A.bf16(mir)).double().reshape(B, -1).mean(1)
    # ---- against the exact block: the attention branch within the bound of the rounding points (+ the output rounding) ----
    e_ex = (out - ex).reshape(B, -1).norm(dim=1)
    bound = A.mirror_branch_bound(ops, softmax, ex) + (0.5 * A.ulp_bf16(ex)).reshape(B, -1).norm(dim=1)
    r_ex = e_ex / bound
    bad = lambda v, gate: [(i, round(float(v[i]), 4)) for i in (v > gate).nonzero().flatten()[:8].tolist()]      # noqa: E731
    ug, fg = ULP_GATE[softmax], FRAC_GATE[softmax]
    assert not bool((ulps > ug).any()), f"{name}: images over {ug} ulps of the mirror (image, ulps): {bad(ulps, ug)}"
    assert not bool((frac > fg).any()), f"{name}: images with a share != bf16_RN(mirror) over {fg}: {bad(frac, fg)}"
    assert not bool((r_ex > 1).any()), f"{name}: attention branch outside the bound of exact (image, err / bound): {bad(r_ex, 1.0)}"
    slack = {"ulps": float(ulps.max()), "frac": float(frac.max()), "exact": float(r_ex.max()),
             "rel_exact": float((e_ex / (ex - ops.x).reshape(B, -1).norm(dim=1)).max())}
    if not softmax and h * h > 128:
        moved = (st["kmax"][:, 1:] > st["kmax"][:, :-1]).double()       # [B][T-1][128]: the running k max moved at tile t
        if kind == "head":
            in_head = moved[..., RAMP_HEAD * 32:(RAMP_HEAD + 1) * 32].mean()
            others = torch.cat([moved[..., :RAMP_HEAD * 32], moved[..., (RAMP_HEAD + 1) * 32:]], -1).mean()
            slack["moved_head"], slack["moved_other"] = float(in_head), float(others)
            assert in_head > others, f"{name}: the ramp does not move the k max in one head more than in the others"
        elif bool((sign < 0).any()):
            up, down = moved[sign > 0].mean(), moved[sign < 0].mean()
            slack["moved_up"], slack["moved_down"] = float(up), float(down)
            assert up > down, f"{name}: the ramps do not steer the running k max (up {float(up):.3f}, down {float(down):.3f})"
    if kind == "shift":
        y = A.linear_exact_y(ops)
        slack["y_mean_over_std"] = float((y.mean((1, 2)) / y.std((1, 2), unbiased=False)).abs().min())
    return (softmax, h * h, c, b > nsm), slack


@pytest.mark.parametrize("name", [c[0] for c in CASES])
def test_attn_tile_case(name):
    nsm = torch.cuda.get_device_properties(DEV).multi_processor_count
    RESULTS[name] = run_case(CASE_BY_NAME[name], nsm)
    print(f"\n{name}: " + ", ".join(f"{k} {v:.4g}" for k, v in RESULTS[name][1].items()))


OP_LINATTN, OP_ATTN, OP_ATTN_FUSED = 4, 5, 9      # plan.cu OpKind


def _expected_attn_ops(cfg, size):
    """name -> (softmax, N, C) of every attention block of the U-Net (plan.cu build order: downs.i.2, mid_attn, ups.j.2)."""
    dims = [cfg["dim"]] + [cfg["dim"] * m for m in cfg["dim_mults"]]
    n = len(cfg["dim_mults"])
    hs = [size >> i for i in range(n)]
    out = {f"downs.{i}.2.fused": (False, hs[i] ** 2, dims[i + 1]) for i in range(n)}
    out["mid_attn.fused"] = (True, hs[n - 1] ** 2, dims[n])
    for j in range(n - 1):
        out[f"ups.{j}.2.fused"] = (False, (hs[n - 1] << j) ** 2, dims[n - 1 - j])
    return out


def _fused_flops(softmax, n, c):
    """plan.cu dmn_plan_op_info, OP_ATTN_FUSED: to_qkv + both contractions + to_out per sample."""
    return 2.0 * n * (384.0 * c + (2.0 * 128.0 * n if softmax else 2.0 * 128.0 * 32.0) + 128.0 * c)


def test_cases_cover_every_production_attention_launch():
    """Every attention block of a production plan is a fused tcgen05 launch (no fallback to the round-1 cores), and every
    (softmax, N, C, more than one image per CTA) key the plans launch is run by some case.  grid = min(B, SMs): the SM count is the
    device's."""
    nsm = torch.cuda.get_device_properties(DEV).multi_processor_count
    c1 = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
    plans = {"configs[1] B=256": (c1, 32, 256), "configs[1] B=512": (c1, 32, 512),
             "configs[2] B=128": (dict(c1, learned_variance=True), 64, 128)}
    need = {}
    for pname, (cfg, size, batch) in plans.items():
        u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
        ops = u.plan(size, batch, DEV).op_table()
        assert not [o for o in ops if o[1] in (OP_LINATTN, OP_ATTN)], f"{pname}: attention fell back to the unfused cores"
        fused = {o[0]: o for o in ops if o[1] == OP_ATTN_FUSED}
        expect = _expected_attn_ops(cfg, size)
        assert set(fused) == set(expect), (pname, sorted(fused), sorted(expect))
        for name, (softmax, n, c) in expect.items():
            assert fused[name][3] == _fused_flops(softmax, n, c), (pname, name, fused[name][3])
            need.setdefault((softmax, n, c, batch > nsm), set()).add(pname)
    have = {}
    for case in CASES:
        if case[0] not in RESULTS:
            RESULTS[case[0]] = run_case(case, nsm)
        have.setdefault(RESULTS[case[0]][0], case[0])
    print(f"\n{nsm} SMs; production keys (softmax, N, C, images > CTAs) -> covering case:")
    missing = []
    for kk, pl in sorted(need.items()):
        print(f"  {kk} [{', '.join(sorted(pl))}] -> {have.get(kk)}")
        if kk not in have:
            missing.append(kk)
    print("slack per case (ulps: max |kernel - mirror| in bf16 ulps; frac: share != bf16_RN(mirror); exact: branch error / bound;"
          " rel_exact: branch rel-L2 vs exact):")
    for n, (k, s) in RESULTS.items():
        print(f"  {n} {k}: " + ", ".join(f"{a} {v:.4g}" for a, v in s.items()))
    for sm in (False, True):
        worst = {a: max(s[a] for k, s in RESULTS.values() if k[0] == sm) for a in ("ulps", "frac", "exact")}
        print(f"worst {'softmax' if sm else 'linear'}: {worst}; gates ulps {ULP_GATE[sm]}, frac {FRAC_GATE[sm]}")
    assert not missing, f"production launches no case covers: {missing}"

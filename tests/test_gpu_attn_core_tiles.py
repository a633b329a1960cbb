"""The bf16 softmax-attention core above 64 tokens (attn_flash_kernel, csrc/attn_fused.cu), element by element, against a float64
reference on the GPU, through `dmn_attention_core`.

The inputs (tests/attn_core_ref.py make_inputs) give every image its own q scale, logits of several units, a key ramp that moves the
running max on later tiles (the rescale path), one head that differs from the others, and -- in the "negative" cases -- real logits
that are all strongly negative on ragged images, where a zero-padded key that took part would get almost all of the weight.

Gate: every element within the bound derived from the kernel's rounding points (tests/attn_core_ref.py module docstring): the bf16
rounding of P, ex2.approx, the fp32 K = 32 product and the roundings of the exponent argument, fp32 accumulation of O and l, and half
an ulp of the bf16 store.  The measured slack (max error / bound per case) is printed and recorded in DESIGN.md.
"""
import pytest
import torch

from conftest import make_unet
from diffusion_model_nemo_b200 import _lib as L
from gpu_helpers import attention_core
from oracle import ref_port as O
import attn_core_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

GRID = {80: (10, 8), 144: (12, 12), 256: (16, 16), 400: (20, 20), 1024: (32, 32), 4096: (64, 64)}
# (N, B, negative): the production launches (N = 256 at B = 64 and the guidance-doubled 128), ragged last tiles (80, 144, 400),
# an odd batch, one image at 4096 tokens (32 key tiles of the running max) and many images at 400
CASES = [(80, 37, True), (144, 37, False), (144, 1, True), (256, 64, False), (256, 128, False), (256, 256, True),
         (400, 1, True), (400, 256, False), (1024, 64, False), (4096, 1, False)]
RESULTS = {}

HIRES_A = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
HIRES_B = dict(dim=64, dim_mults=[1, 2, 4, 8], channels=3, groups=8)
OP_ATTN = 5      # plan.cu OpKind


def run_core(qkv):
    """qkv [B][N][384] bf16-valued -> kernel output [B][N][128] (fp32 holding bf16 values)."""
    b, n, _ = qkv.shape
    h, w = GRID[n]
    x = qkv.permute(0, 2, 1).reshape(b, 384, h, w)
    y = attention_core(x.contiguous(), False, L.ACT_BF16)
    return y.reshape(b, 128, n).permute(0, 2, 1)


def run_case(n, b, neg):
    qkv = R.make_inputs(b, n, negative=neg, seed=n + b, device=DEV)
    got = run_core(qkv)
    assert torch.isfinite(got).all()
    ex, bound = R.exact_and_bound(qkv)
    r, i = R.check(got, ex, bound)
    rel = float((got.double() - ex).norm() / ex.norm())
    return r, i, rel


@pytest.mark.parametrize("n,b,neg", CASES)
def test_flash_core_case(n, b, neg):
    r, i, rel = run_case(n, b, neg)
    RESULTS[(n, b, neg)] = r
    print(f"\nN={n} B={b} negative={neg}: max err / bound {r:.4f}, rel-L2 vs exact {rel:.3e}")
    assert r <= 1.0, f"element {i} (flat [B][N][128]) outside the bound: err / bound = {r:.3f}"


def test_cases_cover_every_hires_softmax_attention_launch():
    """Every softmax-attention core launch of the 128x128 plans A and B at B = 64 and 128 is a case above, and runs on tcgen05."""
    cases = {(n, b) for n, b, _ in CASES}
    for cfg in (HIRES_A, HIRES_B):
        u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
        for batch in (64, 128):
            ops = u.plan(128, batch, DEV).op_table()
            core = [o for o in ops if o[1] == OP_ATTN]
            assert core, (cfg, batch, "no softmax-attention core op")
            for name, _, eng, _, _ in core:
                assert eng == 1, (cfg, batch, name, "not on tcgen05")
            assert (256, batch) in cases, (cfg, batch)

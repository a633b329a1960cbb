"""The checker of the bf16 softmax-attention core above 64 tokens (tests/attn_core_ref.py) on the CPU: a float32 model of the
kernel's arithmetic stays inside the bound, and each defect the GPU test has to catch lands outside it."""
import pytest
import torch

import attn_core_ref as R

# (B, N, negative logits): ragged last tiles (144 = 128 + 16, 200 = 128 + 72) and a whole-tile image (256)
SHAPES = [(3, 144, False), (3, 144, True), (2, 200, True), (2, 256, False)]


@pytest.mark.parametrize("b,n,neg", SHAPES)
def test_model_inside_bound(b, n, neg):
    qkv = R.make_inputs(b, n, negative=neg, seed=n)
    ex, bound = R.exact_and_bound(qkv)
    r, _ = R.check(R.model_flash(qkv), ex, bound)
    assert r <= 1.0, r


def test_inputs_move_the_running_max():
    """The key ramp moves the running max on every later tile for most query rows (the rescale path runs)."""
    qkv = R.make_inputs(2, 512, seed=1)
    q, k, _ = [t.double() for t in R.split(qkv)]
    tmax = (q @ k.transpose(-1, -2)).reshape(2, 4, 512, 4, 128).amax(-1)     # [b][h][i][tile]
    moved = (tmax[..., 1:] > tmax[..., :-1].cummax(-1).values).double().mean()
    assert moved > 0.5, float(moved)


@pytest.mark.parametrize("defect,b,n,neg", [("unmasked_pad", 2, 144, True), ("unmasked_pad", 2, 200, True),
                                            ("skip_rescale", 2, 384, False), ("neighbour_row", 3, 144, False),
                                            ("swap_heads", 2, 256, False)])
def test_checker_rejects(defect, b, n, neg):
    qkv = R.make_inputs(b, n, negative=neg, seed=n)
    ex, bound = R.exact_and_bound(qkv)
    r, _ = R.check(R.model_flash(qkv, defect=defect), ex, bound)
    assert r > 1.0, (defect, r)


def test_bound_is_tight_enough():
    """The bound stays within a small multiple of the bf16 output rounding: about 2^-7 relative to the largest |o| of a row."""
    qkv = R.make_inputs(2, 256, seed=5)
    ex, bound = R.exact_and_bound(qkv)
    rel = (bound / ex.abs().amax(-1, keepdim=True)).max()
    assert rel < 2.0 ** -5, float(rel)
    assert torch.isfinite(bound).all()

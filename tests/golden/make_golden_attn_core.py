"""Fixture of the fp32 SIMT softmax-attention core (tests/golden/attn_core_simt.npz): the outputs of `dmn_attention_core`
(compute_dtype fp32) on seeded inputs at N in {16, 64, 144, 192} tokens, taken on a B200 with the kernel that held all of K and V
in shared memory.  The streamed kernel keeps each query's key order and its fmaf / __expf chain, so it must reproduce these
outputs bit for bit (tests/test_gpu_hires.py).

    python tests/golden/make_golden_attn_core.py [out.npz]      # needs a GPU
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from gpu_helpers import attention_core  # noqa: E402

# (h, w) of the token grid: N = h * w; 192 is the most the all-in-shared-memory kernel held
SHAPES = [(4, 4), (8, 8), (12, 12), (12, 16)]
BATCH = 2


def inputs(h, w):
    """Seeded qkv [BATCH][384][h][w]; logits of several units (q.k / sqrt(32) has a standard deviation of about 4)."""
    return 2.0 * torch.randn(BATCH, 384, h, w, generator=torch.Generator().manual_seed(1000 + h * w))


def main():
    from diffusion_model_nemo_b200 import _lib as L

    out = {}
    for h, w in SHAPES:
        y = attention_core(inputs(h, w).to("cuda:0"), False, L.ACT_F32).cpu()
        out[f"n{h * w}"] = y.numpy().astype(np.float32)
        print(f"N={h * w}: |y|max {float(y.abs().max()):.4f}")
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "attn_core_simt.npz")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    np.savez_compressed(path, **out)
    print("wrote", path)


if __name__ == "__main__":
    main()

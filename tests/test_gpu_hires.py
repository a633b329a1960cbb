"""The 128x128 path end to end.  Two configurations, both with a 16x16 bottleneck of 256 tokens (the softmax attention of the
bottleneck runs on attn_flash_kernel in bf16 and on the streamed SIMT core in fp32):

  A: dim 128, dim_mults (1, 2, 2, 2)          bottleneck C = 256; fused linear attention at 16 384 tokens x 128 and 4 096 x 256
  B: dim 64,  dim_mults (1, 2, 4, 8)          the reference constructor's defaults; bottleneck C = 512; linear attention at C = 64
                                              (level 0) on the unfused path
"""
import functools
import os
import sys

import numpy as np
import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from conftest import make_unet, make_wavegrad_unet, rel_l2
from diffusion_model_nemo_b200 import _lib as L
from gpu_helpers import attention_core, conv_log
from oracle import ref_port as O

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
import make_golden_attn_core as G  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
S = 128
HIRES_A = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
HIRES_B = dict(dim=64, dim_mults=[1, 2, 4, 8], channels=3, groups=8)
CFGS = {"A": HIRES_A, "B": HIRES_B}
OP_INIT, OP_CONV = 1, 2      # plan.cu OpKind


def _x(b, seed=3):
    return torch.randn(b, 3, S, S, generator=torch.Generator().manual_seed(seed))


# ---- the fp32 SIMT core: bit-identical to the all-resident kernel up to 192 tokens ----------------------------------------------
def test_fp32_core_matches_fixture_bit_for_bit():
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "attn_core_simt.npz")
    ref = np.load(path)
    for h, w in G.SHAPES:
        got = attention_core(G.inputs(h, w).to(DEV), False, L.ACT_F32).cpu()
        assert torch.equal(got, torch.from_numpy(ref[f"n{h * w}"])), (h, w)


# ---- U-Net forward against the CPU oracle -------------------------------------------------------------------------------------
_ORACLE = {}


def _oracle(name):
    """Oracle eps for batch 2 at t in {999, 500, 1, 0} (8 rows: sample i at t_k is row 2k + i)."""
    if name not in _ORACLE:
        cfg = CFGS[name]
        sd = O.random_state_dict(cfg, seed=0)
        x = _x(2).repeat(4, 1, 1, 1)
        t = torch.tensor([999, 500, 1, 0]).repeat_interleave(2)
        _ORACLE[name] = (sd, x, t, O.unet_forward(sd, cfg, x, t.float()))
    return _ORACLE[name]


@pytest.mark.parametrize("name", ["A", "B"])
def test_unet_bf16_tcgen05_vs_oracle(name):
    sd, x, t, ref = _oracle(name)
    u = make_unet(CFGS[name], sd, dtype="bf16", engine="tcgen05", device=DEV)
    for k in range(4):
        sl = slice(2 * k, 2 * k + 2)
        eps = u(x[sl].to(DEV), t[sl].to(DEV)).cpu()
        assert torch.isfinite(eps).all()
        assert rel_l2(eps, ref[sl]) <= 2e-2, (name, int(t[2 * k]), rel_l2(eps, ref[sl]))


@pytest.mark.parametrize("name", ["A", "B"])
def test_unet_fp32_vs_oracle(name):
    sd, x, t, ref = _oracle(name)
    u = make_unet(CFGS[name], sd, dtype="fp32", engine="simt", device=DEV)
    eps = u(x[2:3].to(DEV), t[2:3].to(DEV)).cpu()          # batch 1, t = 500
    assert rel_l2(eps, ref[2:3]) <= 1e-4


def test_wavegrad_unet_vs_oracle():
    cfg = dict(HIRES_A, film=True)
    sd = O.random_state_dict(cfg, seed=0)
    x = _x(2, seed=4)
    level = torch.tensor([0.3, 0.8]).view(2, 1, 1, 1)
    ref = O.wavegrad_unet_forward(sd, cfg, x, level)
    u = make_wavegrad_unet(cfg, sd, dtype="bf16", engine="tcgen05", device=DEV)
    y = u(x.to(DEV), level.to(DEV)).cpu()
    assert rel_l2(y, ref) <= 2e-2


# ---- which convolutions of A and B run on the tensor-core engine ---------------------------------------------------------------
# The conv engine's guards (fill_params, csrc/conv_tcgen05.cu) send these convolutions to the SIMT engine at 128x128, at B = 64 and 128
# alike (measured on a B200; the engine is not widened here).  The level-0 3x3 convolutions (H = 128) trip the operand-window guard:
# a 256-row tile plus two halo rows of W + 1 pixels is P = 516 > 448 positions per producer pass.  B's level-0 1x1 convolutions
# (C = 64) and its 64-channel 3x3 convolutions of ups.2 (64x64) are outside the guards as well.
SIMT_CONVS = {
    "A": ["downs.0.0.block1.proj", "downs.0.0.block2.proj", "downs.0.1.block1.proj", "downs.0.1.block2.proj",
          "final_conv.0.block1.proj", "final_conv.0.block2.proj"],
    "B": ["downs.0.0.block1.proj", "downs.0.0.block2.proj", "downs.0.1.block1.proj", "downs.0.1.block2.proj",
          "downs.0.2.fn.fn.to_qkv", "downs.0.2.fn.fn.to_out.0", "ups.2.0.block1.proj", "ups.2.0.block2.proj",
          "ups.2.1.block1.proj", "ups.2.1.block2.proj", "final_conv.0.block1.proj", "final_conv.0.block2.proj"],
}


@pytest.mark.parametrize("name", ["A", "B"])
@pytest.mark.parametrize("batch", [64, 128])
def test_conv_engines_at_128(name, batch):
    """The op table's engine field names the SIMT fallbacks exactly (SIMT_CONVS), and the tcgen05 launch log of one forward holds
    one record per convolution the table marks tcgen05: the silent fallback is visible and pinned."""
    cfg = CFGS[name]
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
    ops = u.plan(S, batch, DEV).op_table()
    convs = [o for o in ops if o[1] == OP_CONV]
    simt = [o[0] for o in convs if o[2] != 1]
    assert simt == SIMT_CONVS[name], f"{name} B={batch}: convolutions on the SIMT engine: {simt}"
    n_tc = sum(1 for o in convs if o[2] == 1) + sum(1 for o in ops if o[1] == OP_INIT and o[2] == 1)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(batch, 3, S, S, generator=g).to(DEV)
    t = torch.randint(0, 1000, (batch,), generator=g).to(DEV)
    conv_log(1 << 16)        # drains what earlier tests recorded (the log keeps up to 65 536 records)
    u(x, t)
    torch.cuda.synchronize()
    recs = conv_log()
    assert len(recs) == n_tc, (name, batch, len(recs), n_tc)


# ---- linear attention at 16 384 and 4 096 tokens ------------------------------------------------------------------------------
@pytest.mark.parametrize("n_side,c,b", [(128, 128, 8), (64, 256, 16)])
def test_fused_linear_attention_hires(n_side, c, b):
    """The fused block of A's levels 0 and 1, element by element (the gates and references of tests/test_gpu_attn_tiles.py)."""
    import test_gpu_attn_tiles as T

    nsm = torch.cuda.get_device_properties(DEV).multi_processor_count
    key, slack = T.run_case((f"hires_lin_{n_side * n_side}x{c}_b{b}", False, n_side, c, b, "mixed"), nsm)
    print(f"\nN={n_side * n_side} C={c} B={b}: " + ", ".join(f"{k} {v:.4g}" for k, v in slack.items()))


def test_unfused_linear_attention_core_16384():
    """B's level 0 (C = 64) runs to_qkv, the linear-attention core and to_out as three launches: the bf16 core at 16 384 tokens."""
    qkv = torch.randn(2, 384, S, S, generator=torch.Generator().manual_seed(9))
    b, n = 2, S * S
    qq, kk, vv = [t.reshape(b, 4, 32, n).double() for t in qkv.chunk(3, dim=1)]
    qq = qq.softmax(dim=-2) * 32 ** -0.5
    kk = kk.softmax(dim=-1)
    ref = torch.einsum("bhde,bhdn->bhen", torch.einsum("bhdn,bhen->bhde", kk, vv), qq).reshape(b, 128, S, S)
    got = attention_core(qkv.to(DEV), True, L.ACT_BF16).cpu()
    assert rel_l2(got, ref) <= 1.5e-2


# ---- sampling loops at 128x128 on A -----------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def unet_a():
    return make_unet(HIRES_A, O.random_state_dict(HIRES_A, seed=0), dtype="bf16", engine="tcgen05", device=DEV)


def test_ddpm_loop_graph_slice_and_seed(unet_a):
    s = M.GaussianDiffusion(50, "linear")
    s.seed = 11
    a = s.sample(unet_a, [8, 3, S, S], device=DEV)[-1]
    a2 = s.sample(unet_a, [8, 3, S, S], device=DEV)[-1]
    s.use_cuda_graph = False
    c = s.sample(unet_a, [8, 3, S, S], device=DEV)[-1]
    assert torch.equal(a, a2) and torch.equal(a, c)
    assert torch.isfinite(a).all() and float(a.min()) >= 0.0 and float(a.max()) <= 1.0
    # the batch-8 slice of a batch-64 run (explicit noise, so both runs draw the same numbers)
    s.use_cuda_graph = True
    s.seed = None
    q = O.NoiseQueue(5)
    nz = torch.stack([q([64, 3, S, S]) for _ in range(51)])
    big = s.sample(unet_a, [64, 3, S, S], device=DEV, noise=nz)[-1]
    small = s.sample(unet_a, [8, 3, S, S], device=DEV, noise=nz[:, :8].contiguous())[-1]
    assert (big[:8] - small).abs().max() <= 1e-6


def test_few_step_samplers_finite_and_reproducible(unet_a):
    shape = [4, 3, S, S]
    samplers = [M.GeneralizedGaussianDiffusion(1000, "linear", ddim_timesteps=50),
                M.DPMSolverDiffusion(1000, "linear", steps=20, order=2)]
    vp = M.DPMSolverSampler(steps=20, order=2)
    vp.update_sde(M.VPSDE())
    samplers.append(vp)
    for s in samplers:
        s.seed = 21
        a = s.sample(unet_a, shape, device=DEV)[-1]
        b = s.sample(unet_a, shape, device=DEV)[-1]
        assert torch.isfinite(a).all(), type(s).__name__
        assert torch.equal(a, b), type(s).__name__


def test_classifier_free_guidance_hires():
    cfg = dict(HIRES_A, num_classes=10)
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
    shape = [4, 3, S, S]
    labels = torch.tensor([1, 3, 5, 7], device=DEV)
    q = O.NoiseQueue(8)
    nz = torch.stack([q(shape) for _ in range(11)])
    s = M.GaussianDiffusion(10, "linear", class_conditional=True)
    s.guidance_scale = 3.0
    out = s.sample(functools.partial(u.forward, classes=labels), shape, device=DEV, noise=nz)[-1]
    assert torch.isfinite(out).all()
    # w = 0: eps = eps_u, the null-label prediction of the same doubled batch
    s.guidance_scale = 0.0
    g0 = s.sample(functools.partial(u.forward, classes=labels), shape, device=DEV, noise=nz)[-1]
    null = torch.full_like(labels, cfg["num_classes"])
    g0n = s.sample(functools.partial(u.forward, classes=null), shape, device=DEV, noise=nz)[-1]
    assert (g0 - g0n).abs().max() <= 1e-6

"""BASELINE.json `configs` at their real shapes on the tensor-core engine (bf16 activations, fp32 accumulation).

The oracle (oracle/ref_port.py, pinned against the executed reference) is evaluated on the CPU inside the test at a small batch;
at the full benchmark batch the checks are size-independent properties (bit-reproducibility, independent RNG streams per rank,
batch-slice invariance).  Tolerance: per-evaluation eps rel-L2 <= 2e-2 (north_star, bf16 mode).
"""
import os

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from conftest import make_unet, rel_l2
from oracle import ref_port as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rand(*shape, seed=0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed))


def test_config3_improved_ddpm_64x64_learned_variance():
    """configs[2]: 3x64x64, dim 128, mults 1,2,2,2, learned variance (6 output channels); 250-step cosine table and DDIM-50."""
    cfg = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8, learned_variance=True)
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="bf16", engine="tcgen05", device=DEV)
    x = _rand(2, 3, 64, 64, seed=3)
    t = torch.tensor([249, 17])
    ref = O.unet_forward(sd, cfg, x, t.float())
    y = u(x.to(DEV), t.to(DEV)).cpu()
    assert y.shape == (2, 6, 64, 64)
    assert rel_l2(y, ref) <= 2e-2
    # learned-variance loop on the fresh 250-step cosine table (the reference has no respacing: SURVEY.md section 8)
    s = M.LearnedGaussianDiffusion(250, "cosine")
    s.seed = 11
    a = s.p_sample_loop(u, [2, 3, 64, 64], device=DEV)[-1]
    s.seed = 11
    b = s.p_sample_loop(u, [2, 3, 64, 64], device=DEV)[-1]
    assert torch.isfinite(a).all() and a.min() >= 0 and a.max() <= 1 and torch.equal(a, b)


def test_config3_ddim50_64x64():
    cfg = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
    d = M.GeneralizedGaussianDiffusion(1000, "cosine", eta=0.0, ddim_timesteps=50)
    d.seed = 5
    out = d.sample(u, [2, 3, 64, 64], device=DEV)[-1]
    assert out.shape == (2, 3, 64, 64) and torch.isfinite(out).all()


@pytest.mark.parametrize("kind", ["vp", "ve"])
def test_config4_score_sde_pc_32x32(kind):
    """configs[3]: 3x32x32 U-Net with groups = 4, reverse-diffusion predictor + Langevin corrector; float time input."""
    cfg = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=4)
    sd = O.random_state_dict(cfg, seed=0)
    u = make_unet(cfg, sd, dtype="bf16", engine="tcgen05", device=DEV)
    x = _rand(2, 3, 32, 32, seed=4)
    t = torch.tensor([999 * 0.731, 999 * 0.02]) if kind == "vp" else torch.tensor([12.5, 0.03])
    ref = O.unet_forward(sd, cfg, x, t)
    assert rel_l2(u(x.to(DEV), t.to(DEV)).cpu(), ref) <= 2e-2
    sde = M.VPSDE(0.1, 20, 40) if kind == "vp" else M.VESDE(0.01, 50, 40)
    pc = M.PredictorCorrectorSampler("reverse_diffusion", "langevin", snr=0.16, n_steps=1)
    pc.update_sde(sde)
    pc.seed = 3
    out = pc.sample(u, [2, 3, 32, 32], device=DEV)[-1]
    assert out.shape == (2, 3, 32, 32) and torch.isfinite(out).all()
    # seeded mode at the benchmark batch: the Langevin step size depends on batch-mean norms, which are summed in a fixed order,
    # so two graph runs and a plain-launch run give the same bits
    shape = [256, 3, 32, 32]
    a = pc.sample(u, shape, device=DEV)[-1]
    b = pc.sample(u, shape, device=DEV)[-1]
    pc.use_cuda_graph = False
    c = pc.sample(u, shape, device=DEV)[-1]
    assert torch.isfinite(a).all() and torch.equal(a, b) and torch.equal(a, c)


def test_config2_full_batch_properties():
    """configs[1] at the benchmark batch (256): bit-reproducible, rank streams independent, and a sample's trajectory does not
    depend on which other samples share its batch (no cross-sample coupling in DDPM: SURVEY.md section 8e)."""
    cfg = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
    u = make_unet(cfg, O.random_state_dict(cfg, seed=0), dtype="bf16", engine="tcgen05", device=DEV)
    s = M.GaussianDiffusion(8, "linear")
    shape = [256, 3, 32, 32]
    noise = torch.stack([_rand(*shape, seed=100 + i) for i in range(9)])
    a = s.sample(u, shape, device=DEV, noise=noise)[-1]
    b = s.sample(u, shape, device=DEV, noise=noise)[-1]
    assert torch.isfinite(a).all() and torch.equal(a, b)
    # the first 32 samples alone: same weights, same injected noise -> the same images up to the order-independent statistics
    c = s.sample(u, [32, 3, 32, 32], device=DEV, noise=noise[:, :32].contiguous())[-1]
    assert (a[:32] - c).abs().max() <= 1e-6
    # in-kernel Philox: same (seed, rank) -> identical; another rank -> different
    s.seed = 7
    r0 = s.sample(u, [64, 3, 32, 32], device=DEV)[-1]
    s.seed = 7
    r0b = s.sample(u, [64, 3, 32, 32], device=DEV)[-1]
    os.environ["RANK"] = "1"
    try:
        s.seed = 7
        r1 = s.sample(u, [64, 3, 32, 32], device=DEV)[-1]
    finally:
        os.environ.pop("RANK")
    assert torch.equal(r0, r0b) and not torch.equal(r0, r1)

"""Forward-mode JVP of the U-Net on the GPU (Unet.jvp / dmn_unet_jvp, fp32 SIMT engine) against torch.func.jvp of the fp64
oracle U-Net (tests/likelihood_oracle.py), for every op kind of the forward program: stem, ResnetBlocks, skip concat,
LinearAttention, the bottleneck softmax Attention, down / up convolutions, both tails, class-conditional and learned-variance
U-Nets, at VP labels t * 999 for t in {1e-3, 0.5, 1}.

Gates: tangent rel-L2 <= 2e-5 (measured on a B200: at most 3.9e-6, cfg2; the proposed fp32 parity gate 1e-4 was looser than
needed); the primal output equals Unet.forward bit for bit; the tangent is linear in v bit for bit (v -> 2v); two runs give the
same bits."""
import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from conftest import CFGS, make_unet, rel_l2
from oracle import ref_port as O
import likelihood_oracle as LO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 2e-5
CASES = dict(CFGS)
CASES["tiny_cba"] = (dict(dim=32, dim_mults=[1, 2], channels=3, groups=8, order="conv_bn_act"), 16, 2)


def _unet(name):
    cfg, size, _ = CASES[name]
    sd = O.random_state_dict(cfg, seed=0)
    if cfg.get("order") == "conv_bn_act":
        u = M.Unet(None, dim=cfg["dim"], dim_mults=cfg["dim_mults"], channels=cfg["channels"], use_convnext=False,
                   resnet_block_groups=cfg["groups"], resnet_block_order="conv_bn_act", compute_dtype="fp32", conv_engine="simt")
        u.load_state_dict(sd, strict=True)
        u.to(DEV)
    else:
        u = make_unet(cfg, sd, dtype="fp32", engine="simt", device=DEV)
    return cfg, size, sd, u


def _inputs(cfg, size, b=2):
    g = torch.Generator().manual_seed(7)
    x = torch.randn(b, cfg["channels"], size, size, generator=g)
    v = torch.randn(b, cfg["channels"], size, size, generator=g)
    cls = torch.tensor([3, 10][:b]) if cfg.get("num_classes") is not None else None
    return x, v, cls


@pytest.mark.parametrize("name", list(CASES))
def test_jvp_matches_fp64_oracle(name):
    cfg, size, sd, u = _unet(name)
    x, v, cls = _inputs(cfg, size)
    dcls = cls.to(DEV) if cls is not None else None
    errs = []
    for t in (1e-3, 0.5, 1.0):
        label = torch.full((2,), t * 999.0)
        out, tan = u.jvp(x.to(DEV), label.to(DEV), v.to(DEV), dcls)
        assert torch.equal(out, u(x.to(DEV), label.to(DEV), dcls))
        _, ref = LO.unet_jvp(sd, cfg, x, label, v, cls)
        assert tan.shape == ref.shape and torch.isfinite(tan).all()
        errs.append(rel_l2(tan.cpu(), ref))
    print(f"jvp {name}: tangent rel-L2 {max(errs):.3e}")
    assert max(errs) <= TOL, (name, errs)


@pytest.mark.parametrize("name", ["tiny_cls", "cfg1"])
def test_jvp_linear_and_deterministic(name):
    cfg, size, sd, u = _unet(name)
    x, v, cls = _inputs(cfg, size)
    x, v, t = x.to(DEV), v.to(DEV), torch.full((2,), 321.0, device=DEV)
    dcls = cls.to(DEV) if cls is not None else None
    o1, t1 = u.jvp(x, t, v, dcls)
    o2, t2 = u.jvp(x, t, v, dcls)
    _, t3 = u.jvp(x, t, 2 * v, dcls)
    assert torch.equal(o1, o2) and torch.equal(t1, t2)
    assert torch.equal(t3, 2 * t1)

"""The per-step host loop that samples with a model callable other than this package's Unet (modules/_runtime.py run_loop).

1. A model output of the wrong width is rejected with ValueError before any update kernel reads it, for every sampler.
2. A call through a model callable leaves torch's CPU generator where the native loop leaves it: one seed draw per call when
   `seed` is None, with and without an injected x_T.
"""
import functools

import pytest
import torch

import diffusion_model_nemo_b200.modules as M
from diffusion_model_nemo_b200.modules import _runtime as R
from conftest import CFGS, WG_CFGS, make_unet, make_wavegrad_unet
from oracle import ref_port as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture
def steps_launched(monkeypatch):
    """Counts the host loop's update kernels."""
    seen = []
    real = R.launch_step

    def spy(*args, **kw):
        seen.append(args[0])
        return real(*args, **kw)

    monkeypatch.setattr(R, "launch_step", spy)
    return seen


def _known_and_mask(shape):
    return torch.zeros(shape), torch.ones(1, 1, shape[2], shape[3])


@pytest.mark.parametrize("name", ["ddpm", "learned", "ddim", "inpaint", "inpaint_learned"])
def test_wrong_model_output_width_is_rejected_before_the_update(steps_launched, name):
    shape = [2, 3, 8, 8]
    learned = name.endswith("learned")
    s = {"ddpm": M.GaussianDiffusion(10, "linear"), "learned": M.LearnedGaussianDiffusion(10, "linear"),
         "ddim": M.GeneralizedGaussianDiffusion(100, "linear", eta=0.5, ddim_timesteps=5),
         "inpaint": M.GaussianDiffusion(10, "linear"), "inpaint_learned": M.LearnedGaussianDiffusion(10, "linear")}[name]
    # learned variance reads 2C channels, the others C: C + 1 is too wide for one and too narrow for the other, C the wrong width
    # for learned variance
    for ch in (4, 3 if learned else 6):
        def model(x, t, ch=ch):
            return torch.zeros(x.shape[0], ch, *x.shape[2:], device=x.device)

        with pytest.raises(ValueError, match="model output has shape"):
            if name.startswith("inpaint"):
                s.inpaint(model, *_known_and_mask(shape), device=DEV)
            else:
                s.sample(model, shape, device=DEV)
        assert steps_launched == []


def _rng_after(call):
    torch.manual_seed(1234)
    call()
    return torch.get_rng_state()


def _sampler(name):
    if name == "ddpm":
        return M.GaussianDiffusion(10, "linear"), "tiny"
    if name == "learned":
        return M.LearnedGaussianDiffusion(10, "linear"), "tiny_lv"
    if name == "ddim":
        return M.GeneralizedGaussianDiffusion(100, "linear", eta=0.5, ddim_timesteps=5), "tiny"
    if name == "wavegrad":
        return M.WaveGradDiffusion(10, "linear"), "wg_tiny"
    if name == "dpmpp":
        return M.DPMSolverDiffusion(100, "linear", steps=5, order=3), "tiny"
    if name == "inpaint":
        return M.GaussianDiffusion(10, "linear"), "tiny"
    s = M.DPMSolverSampler(steps=4, order=2, algorithm_type="sde-dpmsolver++" if name == "score_sde" else "dpmsolver++")
    s.update_sde(M.VESDE())
    return s, "tiny"


@pytest.mark.parametrize("name", ["ddpm", "learned", "ddim", "wavegrad", "dpmpp", "inpaint", "score_dpm", "score_sde"])
@pytest.mark.parametrize("given_x_T", [False, True])
def test_one_seed_draw_per_call_on_both_paths(name, given_x_T):
    s, fixture = _sampler(name)
    cfg, size, b = WG_CFGS[fixture] if fixture in WG_CFGS else CFGS[fixture]
    make = make_wavegrad_unet if fixture in WG_CFGS else make_unet
    u = make(cfg, O.random_state_dict(cfg, seed=0), dtype="fp32", engine="simt", device=DEV)
    shape = [b, cfg["channels"], size, size]
    g = torch.Generator().manual_seed(3)
    x_T = torch.randn([1] + shape, generator=g) if given_x_T else None
    noise = None if x_T is None else torch.cat([x_T, torch.randn([s.steps] + shape, generator=g)]) if name == "score_sde" else x_T

    def run(model):
        if name == "inpaint":
            return functools.partial(s.inpaint, model, *_known_and_mask(shape), device=DEV, noise=x_T)
        if name in ("score_dpm", "score_sde"):
            return functools.partial(s.sample, model, shape, device=DEV, noise=noise)
        return functools.partial(s.p_sample_loop, model, shape, device=DEV, img=None if x_T is None else x_T[0].to(DEV))

    native = _rng_after(run(u))
    foreign = _rng_after(run(lambda x, t: u(x, t)))
    assert torch.equal(native, foreign)
    # the seed is the one draw: a fixed seed leaves the generator untouched
    s.seed = 7
    untouched = torch.manual_seed(1234).get_state()
    assert torch.equal(_rng_after(run(lambda x, t: u(x, t))), untouched)

"""Shared host logic of the native sampling loops: model resolution, coefficient rows, loop launch, outputs."""
import ctypes as C
import functools
import os
from typing import List, Optional, Sequence, Tuple

import torch

from .. import _lib as L
from .unet import Unet


def resolve_model(model) -> Tuple[Optional[Unet], Optional[torch.Tensor]]:
    """-> (native Unet, classes) when `model` is our Unet or `functools.partial(unet[.forward], classes=...)`
    (how ConditionalDDPM passes it, reference models/conditional_ddpm.py:63); else (None, None)."""
    if isinstance(model, Unet):
        return model, None
    if isinstance(model, functools.partial) and not model.args:
        f = model.func
        owner = f if isinstance(f, Unet) else getattr(f, "__self__", None)
        if isinstance(owner, Unet) and set(model.keywords) <= {"classes"}:
            return owner, model.keywords.get("classes")
    return None, None


def default_device(model, device):
    if device is not None:
        return torch.device(device)
    return next(model.parameters()).device     # same rule as the reference (gaussian_diffusion.py:172-173)


def require_cuda(device):
    if torch.device(device).type != "cuda":
        raise L.DmnError("sampling runs on CUDA devices only: the native kernels have no CPU fallback")


def draw_seed() -> int:
    """Philox seed taken from torch's global CPU generator, so `seed_everything` / `torch.manual_seed`
    (reference examples/ddpm/eval_ddpm.py:78) keep steering the samples."""
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item())


def rank_stream_id() -> int:
    """Independent RNG stream per data-parallel rank: the process-group rank when torch.distributed is initialised (covers
    launchers that do not export RANK: mp.spawn, ddp_spawn, init_method=tcp://), else the RANK environment variable."""
    try:
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            return int(dist.get_rank())
    except Exception:
        pass
    return int(os.environ.get("RANK", "0"))


def coef_rows(cols: Sequence[torch.Tensor], device) -> torch.Tensor:
    """Stack per-step fp32 CPU columns into the [steps][8] device table the kernels index."""
    n = cols[0].shape[0]
    tab = torch.zeros(n, L.COEF_STRIDE, dtype=torch.float32)
    for j, c in enumerate(cols):
        tab[:, j] = c.reshape(-1).to(torch.float32)
    return tab.to(device)


def stable_copy(bufs: dict, name: str, src: torch.Tensor, like: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Copy `src` into bufs[name], a buffer whose address a cached CUDA graph bakes in.  The buffer takes the shape, dtype and
    device of `like` (default: `src`) and is reallocated only when that shape changes."""
    like = src if like is None else like
    buf = bufs.get(name)
    if buf is None or buf.shape != like.shape:
        buf = bufs[name] = torch.empty_like(like)
    return buf.copy_(src)


class LoopResult:
    def __init__(self, final, aux, traj):
        self.final, self.aux, self.traj = final, aux, traj


def run_native_loop(unet: Unet, *, kind: int, shape: Sequence[int], device, times: torch.Tensor, coef: torch.Tensor,
                    coef2: Optional[torch.Tensor] = None, x_init: Optional[torch.Tensor] = None,
                    noise: Optional[torch.Tensor] = None, classes: Optional[torch.Tensor] = None,
                    n_corr: int = 0, corr_kind: int = 0, snr: float = 0.0, denoise: bool = False,
                    seed: Optional[int] = None, traj_every: int = 0, use_graph: bool = True,
                    init_scale: float = 1.0, n_steps: Optional[int] = None, cfg_scale: Optional[float] = None,
                    inpaint: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None) -> LoopResult:
    """Run n_steps of (U-Net + update) natively.  noise: [1 + n_steps*draws, B, C, H, W] injected N(0,1) tensors in
    the reference's draw order (element 0 = x_T), or None for in-kernel Philox; LOOP_DPMPP draws nothing and uses only noise[0].
    cfg_scale: classifier-free guidance weight (None = off; 0.0 is a valid weight and gives the unconditional prediction).
    inpaint: (known [B, C, H, W], mask broadcasting to it, prep_coef [n_steps + 1][8] device rows) runs the loop through
    dmn_sample_loop_inpaint (in-kernel noise only)."""
    lib = L.lib()
    device = torch.device(device)
    require_cuda(device)
    b, c, h, w = (int(s) for s in shape)
    assert h == w, "square images only"
    if c != unet.channels:
        raise ValueError(f"shape has {c} channels but the U-Net was built for {unet.channels} (the reference raises a conv shape error)")
    for name, t, lead in (("x_init", x_init, 0), ("noise", noise, 1)):
        if t is not None and tuple(t.shape[lead:]) != (b, c, h, w):
            raise ValueError(f"{name} has shape {tuple(t.shape)}; expected {'[n, ' if lead else '['}{b}, {c}, {h}, {w}]")
    n_steps = int(times.shape[0]) if n_steps is None else int(n_steps)
    assert 1 <= n_steps <= times.shape[0]
    guided = cfg_scale is not None
    if guided:
        if unet.num_classes is None or classes is None:
            raise ValueError("classifier-free guidance needs a class-conditional Unet and `classes` labels")
        if kind == L.LOOP_PC:
            raise NotImplementedError("classifier-free guidance is built for the DDPM / learned-variance / DDIM / DPM-Solver++ loops")
    plan = unet.plan(h, 2 * b if guided else b, device, time_rows=int(times.shape[0]))
    n = b * c * h * w
    draws = (n_corr + 1) if kind == L.LOOP_PC else (0 if kind == L.LOOP_DPMPP else 1)
    d = L.LoopDesc()
    d.kind, d.n_steps, d.batch, d.n_corr = kind, n_steps, b, n_corr
    d.snr, d.denoise, d.use_graph, d.corr_kind = float(snr), int(denoise), int(use_graph), corr_kind
    d.cfg_scale = float(cfg_scale) if guided else 0.0
    d.cfg_on = 1 if guided else 0
    with torch.cuda.device(device):
        st = L.stream_ptr(device)
        tkey = (times.data_ptr(), int(times.shape[0]), tuple(times[:: max(1, int(times.shape[0]) // 7)].tolist()))
        if plan.time_rows_key != tkey:
            plan.time_table(times, 0)
            plan.time_rows_key = tkey
        rng = L.Rng(seed if seed is not None else draw_seed(), rank_stream_id())
        # loop buffers live with the plan so their addresses (baked into the cached CUDA graph) stay stable
        n_traj = (n_steps // traj_every) if traj_every > 0 else 0
        bkey = (kind, b, n_steps if (n_traj or kind == L.LOOP_BPD) else 0, n_traj, bool(denoise), guided)
        bufs = plan.__dict__.setdefault("_loop_bufs", {})
        if bkey not in bufs:
            bufs[bkey] = {
                "state": torch.empty((b, c, h, w), dtype=torch.float32, device=device),
                "scratch": torch.empty(lib.dmn_loop_scratch_bytes(plan.h, C.byref(d)) // 4, dtype=torch.float32, device=device),
                "aux": (torch.empty((b, c, h, w), dtype=torch.float32, device=device) if (kind == L.LOOP_PC and denoise) else
                        torch.zeros((b, n_steps), dtype=torch.float32, device=device) if kind == L.LOOP_BPD else None),
                "traj": torch.empty((n_traj, b, c, h, w), dtype=torch.float32, device=device) if n_traj > 0 else None,
            }
        state, scratch, aux, traj = (bufs[bkey][k] for k in ("state", "scratch", "aux", "traj"))
        noise_dev = None
        if x_init is not None:
            state.copy_(x_init.to(device, torch.float32))
        elif noise is not None:
            state.copy_(noise[0].to(device, torch.float32))
            if init_scale != 1.0:
                state.mul_(init_scale)
        else:
            L.check(lib.dmn_randn(L.ptr(state), n, rng, -1, st), "dmn_randn")
            if init_scale != 1.0:
                state.mul_(init_scale)
        if noise is not None and draws:
            need = n_steps * draws + (0 if x_init is not None else 1)
            assert noise.shape[0] >= need, f"need {need} injected noise tensors, got {noise.shape[0]}"
            nz = noise[(0 if x_init is not None else 1):]
            noise_dev = nz.to(device, torch.float32).contiguous()
        if classes is not None:
            classes = classes.to(device, torch.int64).reshape(-1)
            if guided:     # doubled batch: [labels ; null class] (the padding row of class_embed, reference unet.py:118-120)
                classes = torch.cat([classes, torch.full_like(classes, unet.num_classes)])
            classes = stable_copy(bufs[bkey], "classes", classes)
        d.coef_dev = coef.data_ptr()
        d.coef2_dev = coef2.data_ptr() if coef2 is not None else None
        d.classes_dev = classes.data_ptr() if classes is not None else None
        d.noise_dev = noise_dev.data_ptr() if noise_dev is not None else None
        d.rng = rng
        d.state_dev = state.data_ptr()
        d.aux_dev = aux.data_ptr() if aux is not None else None
        d.scratch_dev = scratch.data_ptr()
        d.scratch_bytes = scratch.numel() * 4
        d.traj_dev = traj.data_ptr() if traj is not None else None
        d.traj_every = traj_every if traj is not None else 0
        d.state_elems = state.numel()
        if inpaint is None:
            L.check(lib.dmn_sample_loop(plan.h, C.byref(d), st), "dmn_sample_loop")
            plan.last_loop_launches = lib.dmn_loop_launches_per_step(plan.h, C.byref(d)) * n_steps
        else:
            assert noise_dev is None, "inpainting draws its noise in-kernel"
            known, mask, prep_coef = inpaint
            kb = stable_copy(bufs[bkey], "known", known, like=state)
            mb = stable_copy(bufs[bkey], "mask", mask, like=state)      # broadcast to the state's shape
            ip = L.InpaintDesc()
            ip.known_dev, ip.mask_dev, ip.prep_coef_dev = kb.data_ptr(), mb.data_ptr(), prep_coef.data_ptr()
            L.check(lib.dmn_sample_loop_inpaint(plan.h, C.byref(d), C.byref(ip), st), "dmn_sample_loop_inpaint")
            # + one prepare kernel per event and the final composite
            plan.last_loop_launches = (lib.dmn_loop_launches_per_step(plan.h, C.byref(d)) + 1) * n_steps + 1
        # keep every buffer alive until the stream has consumed it
        torch.cuda.current_stream(device).synchronize()
    return LoopResult(state.clone(), None if aux is None else aux.clone(), traj)


def to_image_list(final: torch.Tensor, traj: Optional[torch.Tensor]) -> List[torch.Tensor]:
    """Reference return convention (gaussian_diffusion.py:187-189): list of CPU tensors mapped to [0,1]; the last
    element is the final sample.  Trajectory capture is opt-in (one D2H per kept step instead of one per step)."""
    lib = L.lib()
    outs = []
    with torch.cuda.device(final.device):
        st = L.stream_ptr(final.device)
        items = ([] if traj is None else [traj[i] for i in range(traj.shape[0])]) + [final]
        for t in items:
            o = torch.empty_like(t)
            L.check(lib.dmn_unnormalize(L.ptr(t), L.ptr(o), t.numel(), st), "dmn_unnormalize")
            outs.append(o.cpu())
    if traj is not None and len(outs) >= 2 and torch.equal(outs[-1], outs[-2]):
        outs.pop(-2)    # the last kept step IS the final state
    return outs

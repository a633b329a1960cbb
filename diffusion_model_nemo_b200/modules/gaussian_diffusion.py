"""DDPM ancestral sampler: drop-in for reference modules/gaussian_diffusion.py::GaussianDiffusion.

Hot path (`sample`, `p_sample_loop`, `p_sample`, `interpolate`) runs natively: when the model is this package's
`Unet` the whole T-step loop is a replayed CUDA graph (U-Net + one fused update kernel per step, no host sync, no
per-step D2H); for any other callable the model is called per step and only the update is the fused kernel.
Helper methods used by training / BPD code (`q_sample`, `q_posterior`, ...) keep the reference's torch semantics.
`inpaint` (RePaint, an extension) runs the same loop with one merge kernel in front of every model evaluation.
"""
import math
from typing import List, Optional, Tuple

import torch

from .. import _lib as L
from . import _runtime as R
from .diffusion_process import AbstractDiffusionProcess, SCHEDULE_FNS, gaussian_tables


def _default(val, d):
    return val if val is not None else (d() if callable(d) else d)


def repaint_schedule(k: int, jump_length: int = 1, jump_n_sample: int = 1) -> List[int]:
    """RePaint's get_schedule_jump (Lugmayr et al. 2022) with only jump_length / jump_n_sample: the state indices 0..k-1 of the
    sampler's grid in the order they are visited, ending with -1 (the output).  j = r = 1 is the plain visit order."""
    jumps = {p: jump_n_sample - 1 for p in range(0, k - jump_length, jump_length)}
    t, ts = k, []
    while t >= 1:
        t -= 1
        ts.append(t)
        if jumps.get(t, 0) > 0:
            jumps[t] -= 1
            for _ in range(jump_length):
                t += 1
                ts.append(t)
    ts.append(-1)
    return ts


def inpaint_events(ts: List[int]) -> List[Tuple[int, Optional[int]]]:
    """[(i, a)] per reverse event: one per decreasing pair (i, i - 1) of the schedule, with a = the index the forward jump into it
    starts from (a run of increasing pairs a -> i), or None when the event follows another event."""
    events, src = [], None
    for u, v in zip(ts[:-1], ts[1:]):
        if v < u:
            events.append((u, src))
            src = None
        elif src is None:
            src = u
    return events


class GaussianDiffusion(AbstractDiffusionProcess):
    def __init__(self, timesteps: int, schedule_name: str, schedule_cfg=None, objective: str = "pred_noise",
                 class_conditional: bool = False):
        super().__init__(timesteps=timesteps, schedule_name=schedule_name, schedule_cfg=schedule_cfg)
        assert schedule_name in SCHEDULE_FNS, f"Invalid schedule `{schedule_name}` provided to sampler !"
        assert objective in ["pred_noise", "pred_x0"]
        self.objective = objective
        self.use_class_conditioning = class_conditional
        # drop-in extras (not in the reference): opt-in trajectory capture, fixed Philox seed, graph switch
        self.trajectory_every = 0
        self.seed: Optional[int] = None
        self.use_cuda_graph = True
        # classifier-free guidance weight w (extension, BASELINE config 5a; the reference only TRAINS with label dropout,
        # models/conditional_ddpm.py:59-61): eps = eps_u + w (eps_c - eps_u) on a doubled batch per step.  None = off.
        self.guidance_scale: Optional[float] = None
        self.compute_constants(timesteps)

    # ---- tables ------------------------------------------------------------------------------------
    def compute_constants(self, timesteps):
        self.schedule_fn = SCHEDULE_FNS[self.schedule_name]
        self.timesteps = timesteps
        cfg = self.schedule_cfg.get(self.schedule_name, {})
        for name, tab in gaussian_tables(self.schedule_fn(timesteps=timesteps, **cfg)).items():
            setattr(self, name, tab)
        self._coef_cache = {}

    def _step_rows(self, ts: torch.Tensor):
        """Coefficient columns for the visited timesteps `ts` (int64 CPU, visiting order); kernel row layout in
        include/dmn_b200.h (dmn_ddpm_step)."""
        mask = 1 - (ts == 0).float()
        sigma = mask * torch.exp(0.5 * self.posterior_log_variance_clipped[ts])
        flag = torch.full_like(sigma, 1.0 if self.objective == "pred_x0" else 0.0)
        return [self.sqrt_recip_alphas_cumprod[ts], self.sqrt_recipm1_alphas_cumprod[ts], self.posterior_mean_coef1[ts],
                self.posterior_mean_coef2[ts], sigma, flag]

    _loop_kind = L.LOOP_DDPM

    def _loop_tables(self, ts: torch.Tensor, device):
        key = (str(device), tuple(ts[:: max(1, len(ts) // 5)].tolist()), len(ts), self.objective)
        hit = self._coef_cache.get(key)
        if hit is None:
            hit = (R.coef_rows(self._step_rows(ts), device), ts.to(torch.float32).to(device))
            self._coef_cache[key] = hit
        return hit

    # ---- reference helper API (torch semantics, any device) -------------------------------------------------
    def q_mean_variance(self, x_start, t):
        mean = x_start * self.extract(self.sqrt_alphas_cumprod, t, x_start.shape)
        variance = self.extract(1.0 - self.alphas_cumprod, t, x_start.shape)
        log_variance = self.extract(self.log_one_minus_alphas_cumprod, t, x_start.shape)
        return mean, variance, log_variance

    def q_posterior(self, x_start, x, t):
        c1 = self.extract(self.posterior_mean_coef1, t, x.shape)
        c2 = self.extract(self.posterior_mean_coef2, t, x.shape)
        return c1 * x_start + c2 * x, self.extract(self.posterior_log_variance_clipped, t, x.shape)

    def q_sample(self, x_start, t, noise=None):
        if noise is None:
            noise = torch.randn_like(x_start)
        a = self.extract(self.sqrt_alphas_cumprod, t, x_start.shape)
        b = self.extract(self.sqrt_one_minus_alphas_cumprod, t, x_start.shape)
        return a * x_start + b * noise

    def predict_start_from_noise(self, x_t, t, noise):
        assert x_t.shape == noise.shape, f"{x_t.shape} != {noise.shape}"
        a = self.extract(self.sqrt_recip_alphas_cumprod, t, x_t.shape)
        b = self.extract(self.sqrt_recipm1_alphas_cumprod, t, x_t.shape)
        return a * x_t - b * noise

    def p_mean_variance(self, model, x, t, model_output=None, return_pred_x_start: bool = False):
        model_output = _default(model_output, lambda: model(x, t))
        x_recon = self.predict_start_from_noise(x, t, model_output) if self.objective == "pred_noise" else model_output
        x_recon = x_recon.clamp(-1.0, 1.0)
        mean, logvar = self.q_posterior(x_start=x_recon, x=x, t=t)
        return (mean, None, logvar, x_recon) if return_pred_x_start else (mean, None, logvar)

    # ---- hot path -----------------------------------------------------------------------------------------
    def _uniform_t(self, t: torch.Tensor) -> int:
        tc = t.detach().cpu()
        if not bool((tc == tc[0]).all()):
            raise NotImplementedError("the fused update kernel takes one timestep per call (all entries of t equal)")
        return int(tc[0])

    def _fused_step(self, x, model_out, ts_cpu, noise=None, seed=None):
        R.require_cuda(x.device)
        lib = L.lib()
        coef, _ = self._loop_tables(ts_cpu, x.device)
        out = torch.empty_like(x, dtype=torch.float32)
        x = x.float().contiguous()
        model_out = model_out.float().contiguous()
        rng = L.Rng(seed if seed is not None else R.draw_seed(), R.rank_stream_id())
        with torch.cuda.device(x.device):
            self._launch_step(lib, x, model_out, None if noise is None else noise.float().contiguous(), out, coef, 0, rng,
                              L.stream_ptr(x.device))
        return out

    def _launch_step(self, lib, x, model_out, z, out, coef, step, rng, st):
        L.check(lib.dmn_ddpm_step(L.ptr(x), L.ptr(model_out), L.ptr(z), L.ptr(out), x.numel(), L.ptr(coef), None, step, rng, st),
                "dmn_ddpm_step")

    @torch.no_grad()
    def p_sample(self, model, x, t, noise=None):
        """x_{t-1} from x_t (reference gaussian_diffusion.py:157-167): model call + ONE fused update kernel."""
        ti = self._uniform_t(t)
        return self._fused_step(x, model(x, t), torch.tensor([ti], dtype=torch.long), noise=noise)

    def _model_arg(self, ti: int, b: int, device):
        """Second argument of the denoiser for visited timestep ti (WaveGrad overrides it with the continuous noise level)."""
        return torch.full((b,), ti, device=device, dtype=torch.long)

    def _visit_order(self, start: Optional[int] = None):
        return torch.arange((self.timesteps if start is None else start) - 1, -1, -1, dtype=torch.long)

    @torch.no_grad()
    def p_sample_loop(self, model, shape, device=None, use_tqdm=True, noise=None, img=None, start: Optional[int] = None):
        device = R.default_device(model, device)
        R.require_cuda(device)
        ts = self._visit_order(start)
        unet, classes = R.resolve_model(model)
        if unet is not None:
            coef, times = self._loop_tables(ts, device)
            res = R.run_native_loop(unet, kind=self._loop_kind, shape=shape, device=device, times=times, coef=coef,
                                    x_init=img, noise=noise, classes=classes, seed=self.seed,
                                    traj_every=self.trajectory_every, use_graph=self.use_cuda_graph,
                                    cfg_scale=float(self.guidance_scale) if (self.guidance_scale is not None and classes is not None) else None)
            return R.to_image_list(res.final, res.traj)
        # foreign model: call it per step, fuse only the update
        if self.guidance_scale is not None:
            raise NotImplementedError("guidance_scale needs this package's class-conditional Unet (doubled-batch native loop)")
        b = shape[0]
        seed = self.seed if self.seed is not None else R.draw_seed()
        lib = L.lib()
        coef, _ = self._loop_tables(ts, device)
        with torch.cuda.device(device):
            st = L.stream_ptr(device)
            x = torch.empty(tuple(shape), dtype=torch.float32, device=device)
            rng = L.Rng(seed, R.rank_stream_id())
            k = 0
            if img is not None:
                x.copy_(img)
            elif noise is not None:
                x.copy_(noise[0])
                k = 1
            else:
                L.check(lib.dmn_randn(L.ptr(x), x.numel(), rng, -1, st), "dmn_randn")
            keep = []
            for s, ti in enumerate(ts.tolist()):
                mo = model(x, self._model_arg(ti, b, device)).float().contiguous()
                z = None if noise is None else noise[k + s].to(device, torch.float32).contiguous()
                self._launch_step(lib, x, mo, z, x, coef, s, rng, st)
                if self.trajectory_every and (s + 1) % self.trajectory_every == 0:
                    keep.append(x.clone())
            traj = torch.stack(keep) if keep else None
        return R.to_image_list(x, traj)

    # ---- bits-per-dimension evaluation (SURVEY 8f rank 3) ------------------------------------------------------------
    @torch.no_grad()
    def calculate_bits_per_dimension(self, x_start, diffusion_model_fn, max_batch_size: int = 32, noise=None):
        """Drop-in for AbstractDiffusionModel.calculate_bits_per_dimension (reference models/abstract_diffusion_model.py:137-197;
        there a method of the model shell that only touches `self.sampler`, here a method of the sampler).  For every t = T-1..0:
        x_t = q_sample(x_0, t), one U-Net evaluation, and the variational-bound term (KL of the two posteriors, decoder NLL at t = 0) of
        every sample, plus the prior term.  With this package's Unet the T steps are ONE replayed CUDA graph (q_sample kernel, U-Net,
        fused term reduction); any other callable is evaluated per step and only the two kernels are native.
        `noise` ([T, *x.shape], optional) injects the q_sample draws in the reference's order.  Returns the reference's dict:
        {'total_bpd' [B], 'terms_bpd' [B, T], 'prior_bpd' [B]} on x_start's device."""
        device = x_start.device
        R.require_cuda(device)
        lib = L.lib()
        b = x_start.shape[0]
        if max_batch_size > 0:
            b = min(max_batch_size, b)
        x0 = x_start[:b].float().contiguous()
        T = self.timesteps
        ts = torch.arange(T - 1, -1, -1, dtype=torch.long)
        flag = torch.full((T,), 1.0 if self.objective == "pred_x0" else 0.0)
        coef = R.coef_rows([self.sqrt_recip_alphas_cumprod[ts], self.sqrt_recipm1_alphas_cumprod[ts], self.posterior_mean_coef1[ts],
                            self.posterior_mean_coef2[ts], self.posterior_log_variance_clipped[ts], flag, self.sqrt_alphas_cumprod[ts],
                            self.sqrt_one_minus_alphas_cumprod[ts]], device)
        coef2 = R.coef_rows([torch.log(self.betas)[ts], ts.float(), (ts == 0).float()], device)
        chw = x0[0].numel()
        unet, classes = R.resolve_model(diffusion_model_fn)
        if unet is not None:
            res = R.run_native_loop(unet, kind=L.LOOP_BPD, shape=list(x0.shape), device=device, times=ts.float().to(device), coef=coef,
                                    coef2=coef2, x_init=x0, noise=noise, classes=classes, seed=self.seed, use_graph=self.use_cuda_graph)
            terms = res.aux
        else:
            terms = torch.zeros((b, T), dtype=torch.float32, device=device)
            xt = torch.empty_like(x0)
            rng = L.Rng(self.seed if self.seed is not None else R.draw_seed(), R.rank_stream_id())
            with torch.cuda.device(device):
                st = L.stream_ptr(device)
                for s, ti in enumerate(ts.tolist()):
                    z = None if noise is None else noise[s].to(device, torch.float32).contiguous()
                    L.check(lib.dmn_bpd_qsample(L.ptr(x0), L.ptr(z), L.ptr(xt), x0.numel(), L.ptr(coef), None, s, rng, st), "dmn_bpd_qsample")
                    mo = diffusion_model_fn(xt, torch.full((b,), ti, device=device, dtype=torch.long)).float().contiguous()
                    learned = int(mo.shape[1] == 2 * x0.shape[1])
                    L.check(lib.dmn_bpd_term(L.ptr(x0), L.ptr(xt), L.ptr(mo), L.ptr(terms), b, chw, learned, T, 0, L.ptr(coef), L.ptr(coef2),
                                             None, s, st), "dmn_bpd_term")
        # prior: KL( q(x_T | x_0) || N(0, I) )  (abstract_diffusion_model.py:180-184)
        prior = torch.empty((b,), dtype=torch.float32, device=device)
        pc = R.coef_rows([torch.zeros(1)] * 6 + [self.sqrt_alphas_cumprod[T - 1:T]], device)
        pc2 = R.coef_rows([self.log_one_minus_alphas_cumprod[T - 1:T]], device)
        with torch.cuda.device(device):
            L.check(lib.dmn_bpd_term(L.ptr(x0), None, None, L.ptr(prior), b, chw, 0, 1, 1, L.ptr(pc), L.ptr(pc2), None, 0,
                                     L.stream_ptr(device)), "dmn_bpd_term(prior)")
            torch.cuda.current_stream(device).synchronize()
        return {"total_bpd": terms.sum(dim=1) + prior, "terms_bpd": terms, "prior_bpd": prior}

    # ---- RePaint inpainting (extension) -------------------------------------------------------------------------------------------
    def _inpaint_tables(self, jump_length: int, jump_n_sample: int, device):
        """-> (update rows [E][8], time labels [E], prepare rows [E + 1][8], labels list) for the E events of the schedule.  The update
        row and label of an event at grid index i are the sampler's own visit-order row for that index; prepare rows as documented at
        dmn_inpaint_prepare in include/dmn_b200.h, expanded in fp64 from the fp32 alphas_cumprod table and rounded to fp32 once."""
        ts = self._visit_order()
        coef, times = self._loop_tables(ts, device)
        key = ("inpaint", str(device), coef.data_ptr(), jump_length, jump_n_sample)
        hit = self._coef_cache.get(key)
        if hit is None:
            k = len(ts)
            events = inpaint_events(repaint_schedule(k, jump_length, jump_n_sample))
            rows = [k - 1 - i for i, _ in events]               # grid index i is visit-order row k - 1 - i
            ac = self.alphas_cumprod.double()

            def abar(i):
                return float(ac[int(ts[k - 1 - i])])

            prep = []
            for i, a in events:
                ab = abar(i)
                ratio = 1.0 if a is None else ab / abar(a)
                prep.append([math.sqrt(ratio), math.sqrt(1.0 - ratio), math.sqrt(ab), math.sqrt(1.0 - ab)])
            prep.append([1.0, 0.0, 1.0, 0.0])                      # final composite: the known pixels exactly, no draw
            prep = torch.tensor(prep, dtype=torch.float64).to(torch.float32)
            idx = torch.tensor(rows, dtype=torch.long, device=coef.device)
            hit = (coef[idx].contiguous(), times[idx].contiguous(), R.coef_rows([prep[:, c] for c in range(4)], device),
                   [int(ts[r]) for r in rows], coef, times)      # the base tables stay alive: their address is in the key
            self._coef_cache[key] = hit
        return hit[:4]

    def _check_inpaint_args(self, x_known, mask, jump_length, jump_n_sample):
        if not (isinstance(jump_length, int) and isinstance(jump_n_sample, int) and jump_length >= 1 and jump_n_sample >= 1):
            raise ValueError(f"jump_length and jump_n_sample must be integers >= 1, got {jump_length!r}, {jump_n_sample!r}")
        k = len(self._visit_order())
        if jump_n_sample > 1 and jump_length >= k:
            raise ValueError(f"jump_length={jump_length} must be smaller than the sampler's {k} grid points when jump_n_sample > 1")
        if not (torch.is_tensor(x_known) and x_known.dim() == 4):
            raise ValueError(f"x_known must be a [B, C, H, W] tensor, got {getattr(x_known, 'shape', type(x_known))}")
        if not torch.is_tensor(mask):
            raise ValueError("mask must be a tensor that broadcasts to x_known's shape")
        try:
            ok = torch.broadcast_shapes(mask.shape, x_known.shape) == x_known.shape
        except RuntimeError:
            ok = False
        if not ok:
            raise ValueError(f"mask of shape {tuple(mask.shape)} does not broadcast to x_known's shape {tuple(x_known.shape)}")
        if not bool(((mask >= 0) & (mask <= 1)).all()):
            raise ValueError("mask values must lie in [0, 1] (1 = keep the known pixel)")

    @torch.no_grad()
    def inpaint(self, model, x_known, mask, device=None, noise=None, jump_length: int = 1, jump_n_sample: int = 1):
        """RePaint inpainting (Lugmayr et al. 2022) with the trained model unchanged: keep the pixels of `x_known` ([B, C, H, W] in the
        model's data space [-1, 1]) where `mask` (broadcasts to x_known, values in [0, 1], 1 = keep) is 1 and generate the rest.

        The sampler visits its own grid in RePaint's jump schedule (`repaint_schedule`).  Every reverse event merges
        mask * q_sample(x_known, t) + (1 - mask) * x before the model at label t, then applies the sampler's own update.
        `jump_n_sample` > 1 resamples: every `jump_length` grid points the state is noised forward by `jump_length` points and
        denoised again, so that the generated region agrees with the known one.  A forward jump is one draw,
        x_b = sqrt(abar_b / abar_a) x_a + sqrt(1 - abar_b / abar_a) z, which has the distribution of RePaint's `jump_length` single-step
        undos.  After the last event the known pixels are put back exactly.

        x_T is the draw `sample()` makes for `self.seed`, or `noise[0]` (further elements are ignored).  `trajectory_every` counts
        events.  Returns the reference's list of CPU images in [0, 1], the last being the final sample."""
        device = R.default_device(model, device)
        R.require_cuda(device)
        self._check_inpaint_args(x_known, mask, jump_length, jump_n_sample)
        shape = list(x_known.shape)
        if noise is not None and tuple(noise.shape[1:]) != tuple(shape):
            raise ValueError(f"noise has shape {tuple(noise.shape)}; expected [n, {', '.join(map(str, shape))}]")
        coef, times, prep, labels = self._inpaint_tables(jump_length, jump_n_sample, device)
        unet, classes = R.resolve_model(model)
        if unet is not None:
            res = R.run_native_loop(unet, kind=self._loop_kind, shape=shape, device=device, times=times, coef=coef,
                                    x_init=None if noise is None else noise[0], classes=classes, seed=self.seed,
                                    traj_every=self.trajectory_every, use_graph=self.use_cuda_graph,
                                    cfg_scale=float(self.guidance_scale) if (self.guidance_scale is not None and classes is not None) else None,
                                    inpaint=(x_known, mask, prep))
            return R.to_image_list(res.final, res.traj)
        # foreign model: call it per event; the same kernels, rows and step words as the graph
        if self.guidance_scale is not None:
            raise NotImplementedError("guidance_scale needs this package's class-conditional Unet (doubled-batch native loop)")
        b = shape[0]
        seed = self.seed if self.seed is not None else R.draw_seed()
        lib = L.lib()
        with torch.cuda.device(device):
            st = L.stream_ptr(device)
            known = x_known.to(device, torch.float32).contiguous()
            m = torch.empty_like(known)
            m.copy_(mask)
            x = torch.empty(tuple(shape), dtype=torch.float32, device=device)
            rng = L.Rng(seed, R.rank_stream_id())
            if noise is not None:
                x.copy_(noise[0])
            else:
                L.check(lib.dmn_randn(L.ptr(x), x.numel(), rng, -1, st), "dmn_randn")
            keep = []
            for e, ti in enumerate(labels):
                L.check(lib.dmn_inpaint_prepare(L.ptr(x), L.ptr(known), L.ptr(m), L.ptr(x), x.numel(), L.ptr(prep), None, e, rng, st),
                        "dmn_inpaint_prepare")
                mo = model(x, self._model_arg(ti, b, device)).float().contiguous()
                self._launch_step(lib, x, mo, None, x, coef, e, rng, st)
                if self.trajectory_every and (e + 1) % self.trajectory_every == 0:
                    keep.append(x.clone())
            L.check(lib.dmn_inpaint_prepare(L.ptr(x), L.ptr(known), L.ptr(m), L.ptr(x), x.numel(), L.ptr(prep), None, len(labels), rng,
                                            st), "dmn_inpaint_prepare(final)")
            traj = torch.stack(keep) if keep else None
        return R.to_image_list(x, traj)

    @torch.no_grad()
    def sample(self, model, shape, device=None, noise=None):
        """Returns a list of CPU tensors in [0,1] whose LAST element is the final sample (reference contract,
        gaussian_diffusion.py:187-193).  `noise` ([T+1, *shape], element 0 = x_T) injects the N(0,1) draws."""
        return self.p_sample_loop(model, shape=shape, device=device, noise=noise)

    @torch.no_grad()
    def interpolate(self, model, x1, x2, t: Optional[int] = None, lambd: float = 0.5, noise=None):
        """q_sample both images to level t, lerp, denoise t-1 .. 0 (reference gaussian_diffusion.py:196-218)."""
        t = _default(t, self.timesteps - 1)
        if t >= self.timesteps:
            raise ValueError(f"`t` must be < {self.timesteps} during interpolation")
        assert x1.shape == x2.shape
        R.require_cuda(x1.device)
        lib = L.lib()
        a, b = float(self.sqrt_alphas_cumprod[t]), float(self.sqrt_one_minus_alphas_cumprod[t])
        k = 0
        outs = []
        with torch.cuda.device(x1.device):
            st = L.stream_ptr(x1.device)
            for x in (x1, x2):
                x = x.float().contiguous()
                if noise is not None:
                    z = noise[k].to(x.device, torch.float32).contiguous()
                    k += 1
                else:
                    z = torch.empty_like(x)
                    L.check(lib.dmn_randn(L.ptr(z), z.numel(), L.Rng(R.draw_seed(), R.rank_stream_id()), -1, st), "dmn_randn")
                o = torch.empty_like(x)
                L.check(lib.dmn_axpby(L.ptr(x), L.ptr(z), a, b, L.ptr(o), x.numel(), st), "dmn_axpby")   # q_sample
                outs.append(o)
            img = torch.empty_like(outs[0])
            L.check(lib.dmn_axpby(L.ptr(outs[0]), L.ptr(outs[1]), 1.0 - lambd, float(lambd), L.ptr(img), img.numel(), st), "lerp")
        if t == 0:
            return []
        return self.p_sample_loop(model, shape=list(x1.shape), device=x1.device, img=img, start=t,
                                  noise=None if noise is None else noise[k:])

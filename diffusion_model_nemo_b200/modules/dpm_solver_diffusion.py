"""DPM-Solver++ multistep sampler (Lu et al. 2022, "DPM-Solver++: Fast Solver for Guided Sampling of Diffusion Probabilistic
Models", Algorithm 2 and its third-order extension) for models trained with the DDPM objective.

Not in the reference: an extension, like classifier-free guidance.  It reuses the trained eps (or x0) model unchanged and visits the
DDIM grid, so a config swaps `_target_` from GeneralizedGaussianDiffusion to this class and keeps the U-Net's time labels.  Each step
is one U-Net evaluation and one elementwise update kernel (`dmn_dpmpp_step`) that keeps the last three data predictions in a device
ring; with this package's Unet the whole loop is one replayed CUDA graph (`DMN_LOOP_DPMPP`).  The solver is deterministic: only x_T
is random.
"""
import math
from typing import List, Optional

import torch

from .. import _lib as L
from . import _runtime as R
from .gaussian_diffusion import GaussianDiffusion
from .generalized_gaussian_diffusion import strided_pairs


class DPMSolverDiffusion(GaussianDiffusion):
    _loop_kind = L.LOOP_DPMPP

    def __init__(self, timesteps: int, schedule_name: str, schedule_cfg=None, objective: str = "pred_noise",
                 class_conditional: bool = False, steps: int = 20, order: int = 2):
        if not (isinstance(steps, int) and 1 <= steps <= timesteps):
            raise ValueError(f"`steps` must be an integer in [1, timesteps={timesteps}], got {steps!r}")
        if order not in (1, 2, 3):
            raise ValueError(f"`order` must be 1, 2 or 3, got {order!r}")
        super().__init__(timesteps=timesteps, schedule_name=schedule_name, schedule_cfg=schedule_cfg, objective=objective,
                         class_conditional=class_conditional)
        self.steps = steps
        self.order = order

    def timestep_pairs(self):
        """[(t_i, t_{i+1})] in visiting order: the DDIM grid with stride T // steps; the last target is -1 (alpha_bar = 1)."""
        return strided_pairs(self.timesteps, self.steps)

    def step_orders(self) -> List[int]:
        """Solver order of every step: 1 for the last step (into alpha_bar = 1 it returns the data prediction), at most 2 for the
        step before it when there are fewer than 15 steps, else min(order, steps taken so far + 1)."""
        k = len(self.timestep_pairs())
        out = []
        for i in range(k):
            if i == k - 1:
                out.append(1)
            elif k < 15 and i == k - 2:
                out.append(min(self.order, 2, i + 1))
            else:
                out.append(min(self.order, i + 1))
        return out

    def _dpm_rows(self):
        """Per-step coefficient columns (kernel row layout at dmn_dpmpp_step in include/dmn_b200.h), expanded in fp64 from the fp32
        alphas_cumprod table and rounded to fp32 once."""
        pairs = self.timestep_pairs()
        ac = self.alphas_cumprod.double()

        def abar(t):
            return 1.0 if t < 0 else float(ac[t])

        def lam(t):
            a = abar(t)
            return 0.5 * (math.log(a) - math.log1p(-a))

        rows = []
        ts = [p[0] for p in pairs]
        for i, (order, (t, tn)) in enumerate(zip(self.step_orders(), pairs)):
            kx, km = float(self.sqrt_recip_alphas_cumprod[t]), float(self.sqrt_recipm1_alphas_cumprod[t])
            flag = 1.0 if self.objective == "pred_x0" else 0.0
            slot = float(i % 3)
            if tn < 0:                       # sigma' = 0, lambda' = inf: x' = m_i
                rows.append([0.0, 1.0, 0.0, 0.0, kx, km, slot, flag])
                continue
            a_n, s_n, s_t = math.sqrt(abar(tn)), math.sqrt(1.0 - abar(tn)), math.sqrt(1.0 - abar(t))
            h = lam(tn) - lam(t)
            em = math.expm1(-h)
            A = -a_n * em
            cx, c0, c1, c2 = s_n / s_t, A, 0.0, 0.0
            if order >= 2:
                r0 = (lam(t) - lam(ts[i - 1])) / h
            if order == 2:                   # x' = cx x + A m0 + A/2 (m0 - m1)/r0
                c0 += A / (2.0 * r0)
                c1 = -A / (2.0 * r0)
            elif order == 3:                 # x' = cx x + A m0 + B1 D1 + B2 D2
                r1 = (lam(ts[i - 1]) - lam(ts[i - 2])) / h
                b1 = a_n * (em / h + 1.0)
                b2 = -a_n * ((em + h) / (h * h) - 0.5)
                q = r0 / (r0 + r1)
                a0 = b1 * (1.0 + q) + b2 / (r0 + r1)      # coefficient of D1_0 = (m0 - m1)/r0
                a1 = -b1 * q - b2 / (r0 + r1)             # coefficient of D1_1 = (m1 - m2)/r1
                c0 += a0 / r0
                c1 = -a0 / r0 + a1 / r1
                c2 = -a1 / r1
            rows.append([cx, c0, c1, c2, kx, km, slot, flag])
        return torch.tensor(rows, dtype=torch.float64).to(torch.float32)

    def _loop_tables(self, ts, device):
        key = (str(device), self.timesteps, self.steps, self.order, self.objective)
        hit = self._coef_cache.get(key)
        if hit is None:
            rows = self._dpm_rows()
            t = torch.tensor([p[0] for p in self.timestep_pairs()], dtype=torch.long)
            hit = (R.coef_rows([rows[:, j] for j in range(rows.shape[1])], device), t.to(torch.float32).to(device))
            self._coef_cache[key] = hit
        return hit

    def _visit_order(self, start=None):
        return torch.tensor([p[0] for p in self.timestep_pairs()], dtype=torch.long)

    def p_sample(self, model, x, t, noise=None):
        raise NotImplementedError("DPM-Solver++ is a multistep solver: it has no single-step API; use p_sample_loop / sample")

    def interpolate(self, model, x1, x2, t: Optional[int] = None, lambd: float = 0.5, noise=None):
        raise NotImplementedError("DPMSolverDiffusion has no interpolate(); decode a given latent with p_sample_loop(img=...)")

    def inpaint(self, model, x_known, mask, device=None, noise=None, jump_length: int = 1, jump_n_sample: int = 1):
        raise NotImplementedError("DPMSolverDiffusion has no inpaint(): its history ring would mix data predictions across merged "
                                  "states; use GaussianDiffusion, LearnedGaussianDiffusion or GeneralizedGaussianDiffusion")

    @torch.no_grad()
    def p_sample_loop(self, model, shape, device=None, use_tqdm=True, noise=None, img=None):
        """Solve from x_T (img, else noise[0], else a Philox draw with self.seed -- the draw DDIM makes for that seed) to the data
        prediction at t = 0.  Returns the reference's list of CPU images in [0, 1], the last being the final sample."""
        device = R.default_device(model, device)
        R.require_cuda(device)
        ts = self._visit_order()
        coef, times = self._loop_tables(ts, device)
        unet, classes = R.resolve_model(model)
        if unet is not None:
            res = R.run_native_loop(unet, kind=L.LOOP_DPMPP, shape=shape, device=device, times=times, coef=coef,
                                    x_init=img, noise=noise, classes=classes, seed=self.seed,
                                    traj_every=self.trajectory_every, use_graph=self.use_cuda_graph,
                                    cfg_scale=float(self.guidance_scale) if (self.guidance_scale is not None and classes is not None) else None)
            return R.to_image_list(res.final, res.traj)
        # foreign model: call it per step, the update is the native kernel with a local history ring
        if self.guidance_scale is not None:
            raise NotImplementedError("guidance_scale needs this package's class-conditional Unet (doubled-batch native loop)")
        b = shape[0]
        lib = L.lib()
        with torch.cuda.device(device):
            st = L.stream_ptr(device)
            x = torch.empty(tuple(shape), dtype=torch.float32, device=device)
            if img is not None:
                x.copy_(img)
            elif noise is not None:
                x.copy_(noise[0])
            else:
                rng = L.Rng(self.seed if self.seed is not None else R.draw_seed(), R.rank_stream_id())
                L.check(lib.dmn_randn(L.ptr(x), x.numel(), rng, -1, st), "dmn_randn")
            ring = torch.empty((3,) + tuple(shape), dtype=torch.float32, device=device)
            chw = x[0].numel()
            keep = []
            for s, ti in enumerate(ts.tolist()):
                mo = model(x, self._model_arg(ti, b, device)).float().contiguous()
                if mo.shape[0] != b or mo[0].numel() not in (chw, 2 * chw):
                    raise ValueError(f"model output has shape {tuple(mo.shape)}; expected {b} samples of C or 2C channels")
                L.check(lib.dmn_dpmpp_step(L.ptr(x), L.ptr(mo), L.ptr(ring), L.ptr(x), b, chw, mo[0].numel(), L.ptr(coef), None, s, st),
                        "dmn_dpmpp_step")
                if self.trajectory_every and (s + 1) % self.trajectory_every == 0:
                    keep.append(x.clone())
            traj = torch.stack(keep) if keep else None
        return R.to_image_list(x, traj)

    @torch.no_grad()
    def sample(self, model, shape, device=None, noise=None):
        """Returns a list of CPU tensors in [0,1] whose LAST element is the final sample.  `noise` ([n >= 1, *shape]): element 0 is x_T,
        the rest is ignored (a DDIM noise stack can be reused)."""
        return self.p_sample_loop(model, shape=shape, device=device, noise=noise)

"""float64 RePaint inpainting oracle (Lugmayr et al. 2022), independent of the rows GaussianDiffusion.inpaint builds.

Grid: the sampler's visit order as ascending labels g[0..K-1] (DDPM / learned variance: g[i] = i; DDIM: oracle.ref_port.ddim_pairs).
State index i is x at label g[i]; index -1 is the output (alpha_bar = 1).  The schedule is RePaint's get_schedule_jump with only
jump_length (j) and jump_n_sample (r).  Walking its pairs:
  - a decreasing pair (i, i - 1) is a reverse event e: merge, model at label g[i], the sampler's update (oracle.ref_port step);
  - a run of increasing pairs a -> b is one forward jump, x_b = sqrt(abar_b / abar_a) x_a + sqrt(1 - abar_b / abar_a) z, applied in
    front of the event at b.
Event e: y = jump(x) (z = draw 2), k = sqrt(abar) known + sqrt(1 - abar) z (draw 1), x = m k + (1 - m) y, then the update (draw 0).
After the last event x = m known + (1 - m) x.  Draws are the in-kernel Philox normals of step e (tests/philox_ref.py).

Also a correlated two-pixel Gaussian prior whose exact eps-model is closed form, for checking what inpainting computes.
"""
import math

import numpy as np
import torch

from oracle import ref_port as O
import philox_ref as P


def schedule(t_T, jump_length, jump_n_sample):
    """RePaint's get_schedule_jump (guided_diffusion/scheduler.py) without n_sample, jump2 / jump3 and start_resampling."""
    jumps = {}
    for j in range(0, t_T - jump_length, jump_length):
        jumps[j] = jump_n_sample - 1
    t = t_T
    ts = []
    while t >= 1:
        t = t - 1
        ts.append(t)
        if jumps.get(t, 0) > 0:
            jumps[t] = jumps[t] - 1
            for _ in range(jump_length):
                t = t + 1
                ts.append(t)
    ts.append(-1)
    return ts


def n_events(k, j, r):
    return k + (r - 1) * j * len(range(0, k - j, j))


def events(ts):
    """[(i, a)]: the reverse event at index i and the start a of the forward jump in front of it (None: no jump)."""
    out, k = [], 0
    while k < len(ts) - 1:
        a = None
        if ts[k + 1] > ts[k]:
            a = ts[k]
            while ts[k + 1] > ts[k]:
                k += 1
        out.append((ts[k], a))
        k += 1
    return out


class Grid:
    """Labels and alpha_bar (fp64 of the fp32 table, as the package reads it) of a sampler's grid."""

    def __init__(self, kind, timesteps, schedule_name="linear", ddim_timesteps=-1, eta=0.0, objective="pred_noise"):
        self.kind, self.eta, self.objective = kind, eta, objective
        self.tb = O.ddpm_tables(timesteps, schedule_name)
        self.aext = O.ddim_extended_cumprod(self.tb["betas"])
        if kind == "ddim":
            self.g = sorted(t for t, _ in O.ddim_pairs(timesteps, ddim_timesteps))
        else:
            self.g = list(range(timesteps))
        self.ac = self.tb["alphas_cumprod"].double()

    def abar(self, i):
        return 1.0 if i < 0 else float(self.ac[self.g[i]])

    def prep_row(self, i, a):
        """(a_j, g_j, a_0, s_0) of the event at index i with the jump from a (None: no jump)."""
        ab = self.abar(i)
        q = 1.0 if a is None else ab / self.abar(a)
        return math.sqrt(q), math.sqrt(1.0 - q), math.sqrt(ab), math.sqrt(1.0 - ab)

    def step(self, x, i, out, z):
        b = x.shape[0]
        t = torch.full((b,), self.g[i], dtype=torch.long)
        if self.kind == "ddpm":
            return O.ddpm_step(self.tb, x, t, out, z, self.objective)
        if self.kind == "learned":
            return O.learned_step(self.tb, x, t, out, z)
        tn = torch.full((b,), self.g[i - 1] if i > 0 else -1, dtype=torch.long)
        return O.ddim_step(self.aext, x, t, tn, out, z, self.eta)


def philox_draws(seed, sid, shape):
    """draw(step, slot) -> the first prod(shape) in-kernel normals of that step word, as fp64 [shape] (a batch prefix of a larger
    run draws the same values: the quad index is the flat element index / 4)."""
    n = int(np.prod(shape))

    def draw(step, slot):
        return torch.from_numpy(P.randn(seed, sid, step, n, draw=slot)).view(*shape)

    return draw


def run(grid, model, x_T, known, mask, ts, draw, keep_every=0):
    """The event recursion.  model(x fp64, t long[B]) -> model output.  Returns (final state, [state after every keep_every-th
    event])."""
    x = x_T.double()
    known, mask = known.double(), mask.double().expand_as(x)
    traj = []
    for e, (i, a) in enumerate(events(ts)):
        aj, gj, a0, s0 = grid.prep_row(i, a)
        if a is not None:
            x = aj * x + gj * draw(e, 2)
        x = mask * (a0 * known + s0 * draw(e, 1)) + (1.0 - mask) * x
        out = model(x, torch.full((x.shape[0],), grid.g[i], dtype=torch.long))
        x = grid.step(x, i, out, draw(e, 0))
        if keep_every and (e + 1) % keep_every == 0:
            traj.append(x)
    return mask * known + (1.0 - mask) * x, traj


def ref_unet_model(sd, cfg, classes=None):
    """The oracle.ref_port U-Net (fp32 weights) as a model callable of the fp64 recursion."""
    return lambda x, t: O.unet_forward(sd, cfg, x.float(), t.float(), classes).double()


# ---- two correlated pixels: x0 ~ N(0, s^2 [[1, rho], [rho, 1]]) ---------------------------------------------------------------
def pair_model(grid, s2, rho):
    """The exact eps-model of the two-pixel prior on images [B, 1, 1, 2]: eps = sqrt(1 - abar) C_t^-1 x_t with
    C_t = abar s^2 Sigma + (1 - abar) I.  Also returns a list that records max |x0 prediction| (the clamp must not bind)."""
    seen = [0.0]
    sig = torch.tensor([[1.0, rho], [rho, 1.0]], dtype=torch.float64)

    def model(x, t):
        ab = float(grid.ac[int(t[0])])
        ct = ab * s2 * sig + (1.0 - ab) * torch.eye(2, dtype=torch.float64)
        eps = math.sqrt(1.0 - ab) * (x.reshape(-1, 2) @ torch.linalg.inv(ct).T)
        x0 = (x.reshape(-1, 2) - math.sqrt(1.0 - ab) * eps) / math.sqrt(ab)
        seen[0] = max(seen[0], float(x0.abs().max()))
        return eps.view_as(x)

    return model, seen

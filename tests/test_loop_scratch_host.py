"""dmn_loop_scratch_bytes on unbound plans (no GPU): the scratch size of every loop kind, with and without guidance, matches the
documented layout, and invalid descriptors get 0."""
import ctypes as C

import pytest

from diffusion_model_nemo_b200 import _lib as L

CH, S = 3, 16
GUIDABLE = (L.LOOP_DDPM, L.LOOP_LEARNED, L.LOOP_DDIM, L.LOOP_DPMPP)


def _plan(out_dim):
    c = L.UnetCfg()
    c.dim, c.n_mults = 32, 2
    c.dim_mults[0], c.dim_mults[1] = 1, 2
    c.channels, c.out_dim, c.groups, c.with_time_emb, c.num_classes = CH, out_dim, 8, 1, 10
    c.image_size, c.max_batch, c.act_dtype, c.conv_engine, c.max_time_rows = S, 512, L.ACT_F32, L.CONV_SIMT, 1000
    h = C.c_void_p()
    L.check(L.lib().dmn_plan_create(C.byref(c), C.byref(h)), "dmn_plan_create")
    return h


def _desc(kind, batch, cfg_on=0):
    d = L.LoopDesc()
    d.kind, d.batch, d.cfg_on = kind, batch, cfg_on
    return d


def _expected_floats(kind, batch, out_dim, cfg_on):
    """The layout in floats: model output [n_out], x_mean [n], Langevin norms behind them, with guidance the doubled batch
    [2n] and its model output [2 n_out], and for DPM-Solver++ a 3n history ring at the next multiple of 4."""
    n, n_out = batch * CH * S * S, batch * out_dim * S * S
    common = 3 * n_out + 3 * n + 2 * batch + 36 if cfg_on else n_out + n + 2 * batch + 16
    return ((common + 3) & ~3) + 3 * n if kind == L.LOOP_DPMPP else common


CASES = [(out_dim, kind, cfg_on)
         for out_dim, kinds in ((CH, (L.LOOP_DDPM, L.LOOP_DDIM, L.LOOP_PC, L.LOOP_BPD, L.LOOP_DPMPP)),
                                (2 * CH, (L.LOOP_LEARNED, L.LOOP_BPD, L.LOOP_DPMPP)))
         for kind in kinds for cfg_on in ((0, 1) if kind in GUIDABLE else (0,))]


@pytest.mark.parametrize("out_dim,kind,cfg_on", CASES)
def test_loop_scratch_bytes_follow_the_layout(out_dim, kind, cfg_on):
    lib = L.lib()
    h = _plan(out_dim)
    try:
        for batch in (1, 3, 64, 256):
            got = lib.dmn_loop_scratch_bytes(h, C.byref(_desc(kind, batch, cfg_on)))
            assert got == 4 * _expected_floats(kind, batch, out_dim, cfg_on), (batch, got)
    finally:
        lib.dmn_plan_destroy(h)


def test_loop_scratch_bytes_is_zero_for_invalid_arguments():
    lib = L.lib()
    h = _plan(CH)
    try:
        assert lib.dmn_loop_scratch_bytes(None, C.byref(_desc(L.LOOP_DDPM, 2))) == 0
        assert lib.dmn_loop_scratch_bytes(h, None) == 0
        for kind in (-1, L.LOOP_DPMPP + 1):
            assert lib.dmn_loop_scratch_bytes(h, C.byref(_desc(kind, 2))) == 0
        for batch in (0, -3):
            assert lib.dmn_loop_scratch_bytes(h, C.byref(_desc(L.LOOP_DDPM, batch))) == 0
        assert lib.dmn_loop_scratch_bytes(h, C.byref(_desc(L.LOOP_DDPM, 2))) > 0
    finally:
        lib.dmn_plan_destroy(h)

"""The time-table mirror of tests/time_ref.py on the CPU: it agrees with the oracle's fp32 time MLP + block projections (and FiLM
encoding) within its bound, and the bound is tight enough to tell a row from its neighbours and a block's column slice from the slice
shifted by one column at every production time set -- otherwise an element-wise pin on the device could not see a loop reading the
wrong row or a block reading the wrong columns.  The column layout comes from the native plan (host-only calls of the C ABI)."""
import contextlib
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import diffusion_model_nemo_b200.modules as M
import time_ref as T
from diffusion_model_nemo_b200 import _lib as L
from diffusion_model_nemo_b200.engine import film_freqs, sinusoid_freqs
from diffusion_model_nemo_b200.modules.sde import ScoreFunction
from gpu_helpers import time_layout
from oracle import ref_port as O

CFG2 = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)
CFG1 = dict(dim=32, dim_mults=[1, 2, 4], channels=1, groups=8)
WG = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8, film=True)


@contextlib.contextmanager
def host_plan(cfg, size=32, batch=2, rows=1000):
    c = L.UnetCfg()
    c.dim, c.n_mults = cfg["dim"], len(cfg["dim_mults"])
    for i, m in enumerate(cfg["dim_mults"]):
        c.dim_mults[i] = m
    c.channels = cfg["channels"]
    c.out_dim = cfg["channels"] * (2 if cfg.get("learned_variance") else 1)
    c.groups = cfg["groups"]
    c.with_time_emb, c.film = (0, 1) if cfg.get("film") else (1, 0)
    c.num_classes = -1 if cfg.get("num_classes") is None else cfg["num_classes"]
    c.image_size, c.max_batch, c.act_dtype, c.conv_engine, c.max_time_rows = size, batch, L.ACT_F32, L.CONV_SIMT, rows
    h = C.c_void_p()
    L.check(L.lib().dmn_plan_create(C.byref(c), C.byref(h)), "dmn_plan_create")
    try:
        yield h
    finally:
        L.lib().dmn_plan_destroy(h)


def layout(cfg):
    with host_plan(cfg) as h:
        return time_layout(h)[1:]


def _ref(cfg, times, seed=0):
    sd = O.random_state_dict(cfg, seed=seed)
    sum_c, _, cols = layout(cfg)
    y, b = T.time_table_ref(times.float(), sinusoid_freqs(cfg["dim"]), sd, cols, sum_c)
    return sd, cols, y, b


# ---- the production time sets -------------------------------------------------------------------------------------------------------
def loop_times(kind):
    """fp32 times in the order the loop passes them: the DDPM (T = 1000 and configs[2]'s 250-step cosine) and DDIM-50 table rows, the
    configs[3] VP labels t (N - 1) and VE sigma(t) over N = 1000 steps."""
    if kind == "ddpm1000":
        return torch.arange(999, -1, -1).float()
    if kind == "cosine250":
        return torch.arange(249, -1, -1).float()
    if kind == "ddim50":
        return M.GeneralizedGaussianDiffusion(1000, "cosine", eta=0.0, ddim_timesteps=50)._loop_tables(None, "cpu")[1]
    sde = M.VPSDE(0.1, 20.0, 1000) if kind == "vp" else M.VESDE(0.01, 50.0, 1000)
    s = M.PredictorCorrectorSampler("reverse_diffusion", "langevin", snr=0.16)
    s.update_sde(sde)
    return ScoreFunction(None, sde, True).labels(s.timesteps()).float()


# ---- agreement with the oracle --------------------------------------------------------------------------------------------------------
def test_sinusoid_freqs_are_the_references():
    for dim in (32, 128):
        half = dim // 2
        t = torch.tensor([0.0, 1.0, 999.0])
        assert torch.equal(O.sinusoidal_embedding(t, dim)[:, :half], (t[:, None] * sinusoid_freqs(dim)[None]).sin())


@pytest.mark.parametrize("cfg,times", [(CFG2, torch.arange(1000).float()), (CFG1, torch.linspace(0, 999, 257)),
                                       (dict(CFG2, groups=4), loop_times("ve"))])
def test_mirror_agrees_with_oracle_within_bound(cfg, times):
    sd, cols, y, b = _ref(cfg, times)
    temb = O.time_mlp_fwd(sd, times.float(), cfg["dim"])
    ref = torch.full_like(y, float("nan"), dtype=torch.float32)
    for p, c in cols.items():
        w = sd[p + ".mlp.1.weight"]
        ref[:, c:c + w.shape[0]] = F.linear(F.silu(temb), w, sd[p + ".mlp.1.bias"])
    nv, ratio = T.check_bound(ref, y, b)
    print(f"oracle fp32 vs mirror: max err / bound = {ratio:.3f}, max bound {float(b.max()):.2e}")
    assert nv == 0


def test_film_mirror_agrees_with_oracle_within_bound():
    with host_plan(WG) as h:
        _, sum_c, _, cols = time_layout(h)
        ch = (C.c_int32 * 16)()
        n = L.lib().dmn_plan_film_layout(h, ch, 16)
    channels = [ch[i] for i in range(n)]
    freq, is_cos = T.film_columns(channels)
    assert torch.equal(freq, film_freqs(channels)) and freq.numel() == sum_c
    levels = torch.cat([torch.tensor([0.0, 1e-6, 1e-3, 0.999, 1.0]), torch.rand(200, generator=torch.Generator().manual_seed(0))])
    v, b = T.film_table_ref(levels, freq, is_cos)
    for j, c in enumerate(channels):
        col = cols[f"films.{j}"]
        ref = O.film_positional_encoding(levels[:, None, None, None], c).reshape(levels.numel(), c)
        nv, ratio = T.check_bound(ref, v[:, col:col + c], b[:, col:col + c])
        assert nv == 0, (j, ratio)


def test_abi_columns_tile_the_table():
    for cfg in (CFG2, CFG1, dict(CFG2, learned_variance=True), dict(CFG2, groups=4), WG):
        with host_plan(cfg) as h:
            _, sum_c, rows, cols = time_layout(h)
            lib = L.lib()
            for i in range(lib.dmn_plan_num_params(h)):
                name = lib.dmn_plan_param_name(h, i).decode()
                c = lib.dmn_plan_param_time_col(h, i)
                if ".mlp.1." in name:
                    assert c == cols[name.rsplit(".mlp.1.", 1)[0]]
                else:
                    assert c == -1, name
            assert lib.dmn_plan_param_time_col(h, -1) == -1 and lib.dmn_plan_film_col(h, 99) == -1
        shapes = O.unet_param_shapes(cfg)
        widths = {p: (shapes[p + ".mlp.1.weight"][0] if not p.startswith("films.") else
                      shapes[p + ".scale_conv.weight"][0]) for p in cols}
        spans = sorted((c, c + widths[p]) for p, c in cols.items())
        assert spans[0][0] == 0 and spans[-1][1] == sum_c and all(a[1] == b[0] for a, b in zip(spans, spans[1:])), spans
        assert rows == 1000


def test_plan_without_time_table_has_no_view_and_rows_are_capped():
    lib = L.lib()
    with host_plan(dict(CFG1)) as h:
        assert lib.dmn_time_table(h, C.c_void_p(16), 0, 65536, None) == -1
        assert b"65535" in lib.dmn_last_error()
    c = L.UnetCfg()
    c.dim, c.n_mults, c.dim_mults[0], c.channels, c.out_dim, c.groups = 32, 1, 1, 1, 1, 8
    c.image_size, c.max_batch, c.act_dtype, c.conv_engine, c.max_time_rows = 16, 1, L.ACT_F32, L.CONV_SIMT, 1
    h = C.c_void_p()
    L.check(lib.dmn_plan_create(C.byref(c), C.byref(h)))
    try:
        assert lib.dmn_plan_time_table_info(h, None, None, None) == -1
    finally:
        lib.dmn_plan_destroy(h)


# ---- discrimination -----------------------------------------------------------------------------------------------------------------
def _separation(y, b, other_y, other_b):
    """Per row: max over columns of |y - other| / (bound + other bound) -- above 1, a kernel within its bound of `other` cannot be
    within its bound of y."""
    return ((y - other_y).abs() / (b + other_b)).amax(1)


@pytest.mark.parametrize("cfg,kind", [(CFG2, "ddpm1000"), (dict(CFG2, learned_variance=True), "cosine250"),
                                      (dict(CFG2, learned_variance=True), "ddim50"), (dict(CFG2, groups=4), "vp"),
                                      (dict(CFG2, groups=4), "ve"), (CFG1, "ddpm1000")])
def test_neighbouring_rows_and_shifted_slices_fall_outside_the_bound(cfg, kind):
    times = loop_times(kind)
    sd, cols, y, b = _ref(cfg, times)
    # a loop reading row s - 1 or s + 1 of the table instead of row s
    rows = torch.minimum(_separation(y[1:], b[1:], y[:-1], b[:-1]), _separation(y[:-1], b[:-1], y[1:], b[1:]))
    if kind == "ve":
        # adjacent VE labels sigma(t) differ by 0.85 % (0.42 at sigma = 50, 1e-4 at sigma = 0.01): from sigma ~ 37 down the rows are
        # closer than the bound, so the element-wise pin cannot tell them apart and the PC loop's row binding is pinned by the
        # bit-exact replay of tests/test_gpu_time_table.py instead.  The first rows still separate.
        assert float(rows[:30].min()) > 1 and float(rows[-1]) < 1
        worst = float("inf")
    else:
        worst = float(rows.min())
    # a block reading its column slice shifted by one column (into its neighbour's columns at the ends of the table)
    sum_c = y.shape[1]
    for p, c in cols.items():
        n = sd[p + ".mlp.1.weight"].shape[0]
        for d in (-1, 1):
            if 0 <= c + d and c + d + n <= sum_c:
                sep = _separation(y[:, c:c + n], b[:, c:c + n], y[:, c + d:c + d + n], b[:, c + d:c + d + n])
                worst = min(worst, float(sep.min()))
    print(f"{kind}: {times.numel()} rows, smallest separation / (sum of bounds) = {worst:.1f}, max bound {float(b.max()):.2e}")
    assert worst > 1


def test_film_neighbouring_levels_fall_outside_the_bound():
    with host_plan(WG) as h:
        ch = (C.c_int32 * 16)()
        n = L.lib().dmn_plan_film_layout(h, ch, 16)
    freq, is_cos = T.film_columns([ch[i] for i in range(n)])
    levels = M.WaveGradDiffusion(1000, "linear")._loop_tables(torch.arange(999, -1, -1), "cpu")[1]
    v, b = T.film_table_ref(levels, freq, is_cos)
    sep = min(float(_separation(v[1:], b[1:], v[:-1], b[:-1]).min()), float(_separation(v, b, v.roll(1, 1), b.roll(1, 1)).min()))
    print(f"FiLM: smallest separation / (sum of bounds) = {sep:.1f}")
    assert sep > 1

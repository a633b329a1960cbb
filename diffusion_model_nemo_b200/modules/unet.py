"""Drop-in for the reference `diffusion_model_nemo.modules.Unet` (reference modules/unet.py:13-168).

Same constructor keywords, same `forward(x, time, classes=None)`, same parameter names and shapes (so a
reference `state_dict` / `.nemo` restore loads key-for-key), but the arithmetic runs in libdmn_b200.so:
the torch sub-modules below only HOLD parameters (and give them torch's default initialisation in the
reference's construction order); their `forward` is never called.
"""
from typing import List, Optional

import torch
import torch.nn as nn

from .. import _lib as L
from ..engine import UnetPlan

_DTYPES = {"bf16": L.ACT_BF16, "bfloat16": L.ACT_BF16, "fp32": L.ACT_F32, "float32": L.ACT_F32}
_ENGINES = {"tcgen05": L.CONV_TCGEN05, "simt": L.CONV_SIMT}


class _Holder(nn.Module):
    """Parameter container; never evaluated."""

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("parameter holder: the native engine evaluates this layer")


def _block(ci, co, groups):
    # reference parts/convnext.py:8-13  (proj conv3x3, GroupNorm)
    m = _Holder()
    m.proj = nn.Conv2d(ci, co, kernel_size=3, padding=1)
    m.norm = nn.GroupNorm(groups, co)
    return m


def _resnet_block(ci, co, time_dim, groups):
    # reference parts/convnext.py:63-76
    m = _Holder()
    if time_dim is not None:
        m.mlp = nn.Sequential(nn.SiLU(), nn.Linear(time_dim, co))
    m.block1 = _block(ci, co, groups)
    m.block2 = _block(co, co, groups)
    if ci != co:
        m.res_conv = nn.Conv2d(ci, co, kernel_size=1)
    return m


def _attention(dim, linear, heads=4, dim_head=32):
    # reference parts/mha.py:8-14,33-42 wrapped as Residual(PreNorm(dim, fn)) (utils.py:68-93)
    fn = _Holder()
    hidden = heads * dim_head
    fn.to_qkv = nn.Conv2d(dim, hidden * 3, kernel_size=1, bias=False)
    if linear:
        fn.to_out = nn.Sequential(nn.Conv2d(hidden, dim, 1), nn.GroupNorm(1, dim))
    else:
        fn.to_out = nn.Conv2d(hidden, dim, kernel_size=1)
    pre = _Holder()
    pre.fn = fn
    pre.norm = nn.GroupNorm(1, dim)
    res = _Holder()
    res.fn = pre
    return res


class Unet(nn.Module):
    def __init__(
        self,
        input_dim: None,
        dim: int,
        out_dim: Optional[int] = None,
        dim_mults: Optional[List[int]] = None,
        channels: int = 3,
        with_time_emb: bool = True,
        resnet_block_groups: int = 8,
        use_convnext: bool = True,
        convnext_mult: int = 2,
        resnet_block_order: str = "bn_act_conv",
        dropout: Optional[float] = None,
        learned_variance: bool = False,
        num_classes: Optional[int] = None,
        compute_dtype: str = "bf16",
        conv_engine: str = "tcgen05",
    ):
        super().__init__()
        if use_convnext:
            raise NotImplementedError(
                "use_convnext=True (ConvNextBlock) is outside the sampling hot path built here; every shipped config "
                "sets use_convnext: False"
            )
        if resnet_block_order not in ("conv_bn_act", "bn_act_conv"):
            raise ValueError("Valid ordering for block are : ['conv_bn_act', 'bn_act_conv']")
        if dim_mults is None:
            dim_mults = (1, 2, 4, 8)
        self.channels, self.learned_variance, self.dim = channels, learned_variance, dim
        self.resnet_block_order, self.num_classes = resnet_block_order, num_classes
        self.groups = resnet_block_groups
        self.dim_mults = tuple(int(m) for m in dim_mults)
        self.compute_dtype, self.conv_engine = compute_dtype, conv_engine
        if compute_dtype not in _DTYPES or conv_engine not in _ENGINES:
            raise ValueError("compute_dtype in {bf16, fp32}; conv_engine in {tcgen05, simt}")

        # ---- parameter tree: same names, shapes and construction order as the reference ----
        self.init_conv = nn.Conv2d(channels, dim, kernel_size=7, padding=3)
        dims = [dim, *[dim * m for m in self.dim_mults]]
        in_out = list(zip(dims[:-1], dims[1:]))
        self.dim_list, self.in_out_list = dims, in_out
        self.with_time_emb = bool(with_time_emb)
        if with_time_emb:
            time_dim = dim * 4
            self.time_mlp = nn.Sequential(_Holder(), nn.Linear(dim, time_dim), nn.GELU(), nn.Linear(time_dim, time_dim))
        else:                       # reference unet.py:67-69
            time_dim = None
            self.time_mlp = None
        g = resnet_block_groups
        self.downs, self.ups = nn.ModuleList([]), nn.ModuleList([])
        n = len(in_out)
        for i, (ci, co) in enumerate(in_out):
            last = i >= n - 1
            self.downs.append(nn.ModuleList([
                _resnet_block(ci, co, time_dim, g), _resnet_block(co, co, time_dim, g), _attention(co, True),
                nn.Conv2d(co, co, kernel_size=4, stride=2, padding=1) if not last else nn.Identity(),
            ]))
        mid = dims[-1]
        self.mid_block1 = _resnet_block(mid, mid, time_dim, g)
        self.mid_attn = _attention(mid, False)
        self.mid_block2 = _resnet_block(mid, mid, time_dim, g)
        for i, (ci, co) in enumerate(reversed(in_out[1:])):
            self.ups.append(nn.ModuleList([
                _resnet_block(co * 2, ci, time_dim, g), _resnet_block(ci, ci, time_dim, g), _attention(ci, True),
                nn.ConvTranspose2d(ci, ci, kernel_size=4, stride=2, padding=1),
            ]))
        default_out = channels * (2 if learned_variance else 1)
        self.out_dim = out_dim if out_dim is not None else default_out
        if resnet_block_order == "bn_act_conv":      # reference unet.py:112-116
            tail = [nn.GroupNorm(g, dim), nn.SiLU(), nn.Conv2d(dim, self.out_dim, kernel_size=1)]
        else:                                          # 'conv_bn_act': the ResnetBlock is followed by the bare 1x1
            tail = [nn.Conv2d(dim, self.out_dim, kernel_size=1)]
        self.final_conv = nn.Sequential(_resnet_block(dim, dim, None, g), *tail)
        if num_classes is not None:
            self.class_embed = nn.Embedding(num_classes + 1, embedding_dim=dim, padding_idx=num_classes)
        self._film = False
        self.requires_grad_(False)
        self._plans = {}

    # ---- engine management -------------------------------------------------------------------------
    def set_precision(self, compute_dtype: str, conv_engine: Optional[str] = None):
        """'fp32' (parity mode, CUDA-core convs) or 'bf16' (tensor-core convs)."""
        if compute_dtype not in _DTYPES:
            raise ValueError(compute_dtype)
        self.compute_dtype = compute_dtype
        if conv_engine is not None:
            self.conv_engine = conv_engine
        if _DTYPES[self.compute_dtype] == L.ACT_F32:
            self.conv_engine = "simt"
        return self

    def _params_version(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def plan(self, image_size: int, batch: int, device, time_rows: int = 0) -> UnetPlan:
        act = _DTYPES[self.compute_dtype]
        eng = L.CONV_SIMT if act == L.ACT_F32 else _ENGINES[self.conv_engine]
        key = (int(image_size), act, eng, str(torch.device(device)))
        p = self._plans.get(key)
        if p is None or p.max_batch < batch or p.max_time_rows < max(time_rows, batch):
            mb = batch if p is None else max(batch, p.max_batch)
            rows = max(time_rows, batch, 0 if p is None else p.max_time_rows)
            p = UnetPlan(dim=self.dim, dim_mults=self.dim_mults, channels=self.channels, out_dim=self.out_dim,
                         groups=self.groups, num_classes=self.num_classes, image_size=image_size, max_batch=mb,
                         act_dtype=act, conv_engine=eng, max_time_rows=rows, device=device,
                         with_time_emb=self.with_time_emb, film=self._film,
                         plain_tail=self.resnet_block_order == "conv_bn_act")
            self._plans[key] = p
        ver = self._params_version()
        if p._loaded_version != ver:
            p.load_state_dict(self.state_dict(), version=ver)
        return p

    # ---- reference API -------------------------------------------------------------------------------
    def forward(self, x, time, classes=None):
        """eps = Unet.forward(x, time, classes) (reference modules/unet.py:131-168); x fp32 NCHW on a CUDA device."""
        if x.device.type != "cuda":
            raise L.DmnError("diffusion_model_nemo_b200.Unet runs on CUDA only: there is no CPU fallback")
        assert x.dim() == 4 and x.shape[1] == self.channels and x.shape[2] == x.shape[3], f"bad input shape {tuple(x.shape)}"
        time = time.reshape(-1)
        assert time.shape[0] == x.shape[0], "time must have one entry per sample"
        p = self.plan(x.shape[-1], x.shape[0], x.device)
        return p.forward(x.float().contiguous(), time, classes)

    def jvp(self, x, time, v, classes=None):
        """Forward-mode Jacobian-vector product: (forward(x, time, classes), d forward / dx . v) in one native pass.

        fp32 only (compute_dtype='fp32'); the output equals forward() bit for bit.  time and classes enter through embeddings
        that do not depend on x, so their tangents are zero."""
        if _DTYPES[self.compute_dtype] != L.ACT_F32:
            raise ValueError("Unet.jvp runs in fp32 only: set compute_dtype='fp32' (set_precision('fp32'))")
        if x.device.type != "cuda":
            raise L.DmnError("diffusion_model_nemo_b200.Unet runs on CUDA only: there is no CPU fallback")
        assert x.dim() == 4 and x.shape[1] == self.channels and x.shape[2] == x.shape[3], f"bad input shape {tuple(x.shape)}"
        if tuple(v.shape) != tuple(x.shape):
            raise ValueError(f"tangent direction v has shape {tuple(v.shape)}; expected {tuple(x.shape)}")
        time = time.reshape(-1)
        assert time.shape[0] == x.shape[0], "time must have one entry per sample"
        p = self.plan(x.shape[-1], x.shape[0], x.device)
        return p.jvp(x.float().contiguous(), time, v.to(x.device, torch.float32).contiguous(), classes)


def _film(c):
    # reference parts/film.py:29-54 (signal conv3x3 + LeakyReLU, scale / shift conv3x3)
    m = _Holder()
    m.signal_conv = nn.Sequential(nn.Conv2d(c, c, kernel_size=3, stride=1, padding=1), nn.LeakyReLU(0.2))
    m.positional_encoding = _Holder()
    m.scale_conv = nn.Conv2d(c, c, kernel_size=3, stride=1, padding=1)
    m.shift_conv = nn.Conv2d(c, c, kernel_size=3, stride=1, padding=1)
    return m


class WaveGradUNet(Unet):
    """Drop-in for the reference `WaveGradUNet` (modules/unet.py:171-266): the U-Net without time embedding whose up path is
    modulated by FeatureWiseLinearModulation statistics (parts/film.py) computed on the way down from a CONTINUOUS noise level.
    `forward(x, noise_level, classes=None)`, noise_level float [B,1,1,1] (or [B]).  Same parameter names / shapes as the
    reference, including the three FiLM layers the reference constructs but never evaluates and the bottleneck FiLM whose
    output it discards (unet.py:204-210,247): they are held for state_dict compatibility and skipped by the engine."""

    def __init__(
        self,
        input_dim: None,
        dim: int,
        out_dim: Optional[int] = None,
        dim_mults: Optional[List[int]] = None,
        channels: int = 3,
        with_time_emb: bool = None,  # ignored, as in the reference
        resnet_block_groups: int = 8,
        use_convnext: bool = True,
        convnext_mult: int = 2,
        resnet_block_order: str = "bn_act_conv",
        dropout: Optional[float] = None,
        learned_variance: bool = False,
        num_classes: Optional[int] = None,
        compute_dtype: str = "bf16",
        conv_engine: str = "tcgen05",
    ):
        super().__init__(input_dim=input_dim, dim=dim, out_dim=out_dim, dim_mults=dim_mults, channels=channels,
                         with_time_emb=False, resnet_block_groups=resnet_block_groups, use_convnext=use_convnext,
                         convnext_mult=convnext_mult, resnet_block_order=resnet_block_order, dropout=dropout,
                         learned_variance=learned_variance, num_classes=num_classes, compute_dtype=compute_dtype,
                         conv_engine=conv_engine)
        films = [_film(dim)]
        films.extend(_film(co) for (_, co) in self.in_out_list)
        films.extend(_film(co) for (_, co) in reversed(self.in_out_list[1:]))
        self.films = nn.ModuleList(films)
        self._film = True
        self.requires_grad_(False)

    def forward(self, x, noise_level, classes=None):
        """eps = WaveGradUNet.forward(x, noise_level, classes) (reference modules/unet.py:212-266)."""
        if x.device.type != "cuda":
            raise L.DmnError("diffusion_model_nemo_b200.WaveGradUNet runs on CUDA only: there is no CPU fallback")
        assert x.dim() == 4 and x.shape[1] == self.channels and x.shape[2] == x.shape[3], f"bad input shape {tuple(x.shape)}"
        level = noise_level.reshape(-1)
        assert level.shape[0] == x.shape[0], "noise_level must have one entry per sample"
        p = self.plan(x.shape[-1], x.shape[0], x.device)
        return p.forward(x.float().contiguous(), level, classes)

    def jvp(self, x, noise_level, v, classes=None):
        raise NotImplementedError("WaveGradUNet has no tangent program: the JVP is built for Unet only")

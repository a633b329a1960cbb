"""Host-side owner of one native U-Net plan (libdmn_b200.so): device buffers, parameter upload, forward, loops.

PyTorch is plumbing here: it allocates the device buffers the C ABI asks for and provides the stream.
"""
import ctypes as C
import math
from typing import Dict, Optional

import torch

from . import _lib as L


def film_freqs(channels) -> torch.Tensor:
    """Per-column frequencies of the FiLM positional encodings: for every FiLM layer (C channels) its
    [exponents | exponents] with exponents = 1e-4 ** (arange(C/2) / (C/2)), built with the reference's own torch CPU ops
    (reference parts/film.py:19-21)."""
    cols = []
    for c in channels:
        half = c // 2
        e = torch.arange(half, dtype=torch.float32) / float(half)
        e = 1e-4 ** e
        cols += [e, e]
    return torch.cat(cols).float().contiguous()


def sinusoid_freqs(dim: int) -> torch.Tensor:
    """Frequencies of SinusoidalPositionEmbeddings, built with the reference's own torch CPU ops
    (reference parts/positional_encoding.py:13-15) so the device table starts from bit-identical values."""
    half = dim // 2
    e = math.log(10000) / (half - 1)
    return torch.exp(torch.arange(half) * -e).float().contiguous()


class UnetPlan:
    """One (config, image_size, max_batch, dtype, engine) instance of the native U-Net."""

    def __init__(self, *, dim, dim_mults, channels, out_dim, groups, num_classes, image_size, max_batch,
                 act_dtype, conv_engine, max_time_rows, device, with_time_emb=True, film=False, plain_tail=False):
        self.lib = L.lib()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise L.DmnError("the native U-Net runs on CUDA devices only (no CPU fallback)")
        cfg = L.UnetCfg()
        cfg.dim = dim
        cfg.n_mults = len(dim_mults)
        for i, m in enumerate(dim_mults):
            cfg.dim_mults[i] = int(m)
        cfg.channels, cfg.out_dim, cfg.groups = channels, out_dim, groups
        cfg.with_time_emb = 1 if with_time_emb else 0
        cfg.film = 1 if film else 0
        cfg.plain_tail = 1 if plain_tail else 0
        cfg.num_classes = -1 if num_classes is None else int(num_classes)
        cfg.image_size, cfg.max_batch = image_size, max_batch
        cfg.act_dtype, cfg.conv_engine = act_dtype, conv_engine
        cfg.max_time_rows = max(max_time_rows, max_batch)
        self.cfg = cfg
        h = C.c_void_p()
        L.check(self.lib.dmn_plan_create(C.byref(cfg), C.byref(h)), "dmn_plan_create")
        self.h = h
        self.max_batch, self.max_time_rows = max_batch, cfg.max_time_rows
        self.image_size, self.channels, self.out_dim, self.dim = image_size, channels, out_dim, dim
        with torch.cuda.device(self.device):
            self.weights = torch.empty(self.lib.dmn_plan_weights_bytes(h) + 256, dtype=torch.uint8, device=self.device)
            self.workspace = torch.empty(self.lib.dmn_plan_workspace_bytes(h) + 256, dtype=torch.uint8, device=self.device)
        L.check(self.lib.dmn_plan_bind(h, self._aligned(self.weights), self.weights.numel() - 256,
                                       self._aligned(self.workspace), self.workspace.numel() - 256), "dmn_plan_bind")
        self.param_names = [self.lib.dmn_plan_param_name(h, i).decode() for i in range(self.lib.dmn_plan_num_params(h))]
        self._loaded_version = None
        self._keep = []        # tensors a cached CUDA graph points at
        self.time_rows_key = None

    @staticmethod
    def _aligned(t):
        p = t.data_ptr()
        return C.c_void_p((p + 255) // 256 * 256)

    def param_shapes(self) -> Dict[str, tuple]:
        out = {}
        for i, n in enumerate(self.param_names):
            shp = (C.c_int64 * 4)()
            nd = self.lib.dmn_plan_param_shape(self.h, i, C.byref(shp))
            out[n] = tuple(shp[k] for k in range(nd))
        return out

    def load_state_dict(self, sd: Dict[str, torch.Tensor], version=None):
        st = L.stream_ptr(self.device)
        with torch.cuda.device(self.device):
            for name in self.param_names:
                if name not in sd:
                    raise KeyError(f"missing parameter {name}")
                t = sd[name].detach().to("cpu", torch.float32).contiguous()
                L.check(self.lib.dmn_plan_load_param(self.h, name.encode(), L.ptr(t), t.numel(), st), f"load {name}")
            if self.cfg.film:
                ch = (C.c_int32 * 16)()
                n = self.lib.dmn_plan_film_layout(self.h, ch, 16)
                f = film_freqs([ch[i] for i in range(n)])
            elif self.cfg.with_time_emb:
                f = sinusoid_freqs(self.dim)
            else:
                f = None
            if f is not None:
                L.check(self.lib.dmn_plan_load_freqs(self.h, L.ptr(f), f.numel(), st), "load freqs")
        self._loaded_version = version
        self.time_rows_key = None

    def time_table(self, times: torch.Tensor, row0: int = 0):
        """times: fp32 device tensor [rows] -> table rows [row0, row0+rows)."""
        times = times.to(self.device, torch.float32).contiguous()
        with torch.cuda.device(self.device):
            L.check(self.lib.dmn_time_table(self.h, L.ptr(times), row0, times.numel(), L.stream_ptr(self.device)), "dmn_time_table")
        self.time_rows_key = None

    def forward(self, x: torch.Tensor, time: torch.Tensor, classes: Optional[torch.Tensor] = None) -> torch.Tensor:
        b = x.shape[0]
        out = torch.empty((b, self.out_dim, self.image_size, self.image_size), dtype=torch.float32, device=self.device)
        self.time_table(time.reshape(-1).float(), 0)
        if classes is not None:
            classes = classes.to(self.device, torch.int64).contiguous()
        with torch.cuda.device(self.device):
            L.check(self.lib.dmn_unet_forward(self.h, L.ptr(x), None, L.ptr(classes), L.ptr(out), b, L.stream_ptr(self.device)),
                    "dmn_unet_forward")
        return out

    def jvp(self, x: torch.Tensor, time: torch.Tensor, v: torch.Tensor, classes: Optional[torch.Tensor] = None):
        """(u(x, time), du/dx . v) in one pass of the forward program with its tangent program (fp32 SIMT plans only)."""
        b = x.shape[0]
        shape = (b, self.out_dim, self.image_size, self.image_size)
        out = torch.empty(shape, dtype=torch.float32, device=self.device)
        tangent = torch.empty(shape, dtype=torch.float32, device=self.device)
        self.time_table(time.reshape(-1).float(), 0)
        if classes is not None:
            classes = classes.to(self.device, torch.int64).contiguous()
        work = self.jvp_work(b)
        with torch.cuda.device(self.device):
            L.check(self.lib.dmn_unet_jvp(self.h, L.ptr(x), L.ptr(v), None, L.ptr(classes), L.ptr(out), L.ptr(tangent),
                                          self._aligned(work), work.numel() - 256, b, L.stream_ptr(self.device)), "dmn_unet_jvp")
        return out, tangent

    def jvp_work(self, batch: int) -> torch.Tensor:
        """Device buffer of dmn_unet_jvp for `batch` samples (kept with the plan, grown on demand; 256 bytes of alignment slack)."""
        nbytes = int(self.lib.dmn_unet_jvp_work_bytes(self.h, batch)) + 256
        w = getattr(self, "_jvp_work", None)
        if w is None or w.numel() < nbytes:
            w = self._jvp_work = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        return w

    def op_table(self):
        """[(name, kind, engine, flops_per_sample, bytes_per_sample)] of the forward program."""
        out = []
        for i in range(self.lib.dmn_plan_num_ops(self.h)):
            name = C.create_string_buffer(128)
            kind, eng, fl, by = C.c_int32(), C.c_int32(), C.c_double(), C.c_double()
            L.check(self.lib.dmn_plan_op_info(self.h, i, name, 128, C.byref(kind), C.byref(eng), C.byref(fl), C.byref(by)))
            out.append((name.value.decode(), kind.value, eng.value, fl.value, by.value))
        return out

    def profile_forward(self, x: torch.Tensor, row_dev: Optional[torch.Tensor] = None, in_graph: bool = False):
        """Per-launch milliseconds of one forward (CUDA events around every launch); time table must be filled.
        in_graph=True measures inside one CUDA graph (event-record nodes): back-to-back kernels as in the sampling loop."""
        n = self.lib.dmn_plan_num_ops(self.h)
        ms = (C.c_float * n)()
        out = torch.empty((x.shape[0], self.out_dim, self.image_size, self.image_size), dtype=torch.float32, device=self.device)
        fn = self.lib.dmn_plan_profile_forward_graph if in_graph else self.lib.dmn_plan_profile_forward
        with torch.cuda.device(self.device):
            L.check(fn(self.h, L.ptr(x), L.ptr(row_dev), None, L.ptr(out), x.shape[0], L.stream_ptr(self.device), ms, n),
                    "dmn_plan_profile_forward")
        return list(ms)

    def launches_per_forward(self) -> int:
        return self.lib.dmn_plan_launches_per_forward(self.h)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.dmn_plan_destroy(self.h)
                self.h = None
        except Exception:
            pass

"""ctypes callers of the layer-level C ABI used by the GPU parity tests."""
import ctypes as C

import torch

from diffusion_model_nemo_b200 import _lib as L


def conv_forward(x, w, bias=None, *, mode=0, ksize=3, gn=None, silu=False, temb=None, out_groups=0, act=L.ACT_F32,
                 engine=L.CONV_SIMT, x2=None):
    """x fp32 NCHW cuda; w torch-layout weights; gn = (groups, gamma, beta) prologue; x2: second source of a channel concatenation
    cat(x, x2) (dmn_conv_forward_cat; w is then the concat weight).  Returns (y NCHW fp32, stats|None)."""
    lib = L.lib()
    dev = x.device
    b, cin, h, wd = x.shape
    cin2 = 0 if x2 is None else x2.shape[1]
    cin += cin2
    cout = w.shape[1] if mode == 2 else w.shape[0]
    ho = h // 2 if mode == 1 else (h * 2 if mode == 2 else h)
    a = L.ConvArgs()
    a.mode, a.ksize, a.batch, a.cin, a.cout, a.hin, a.win = mode, ksize, b, cin, cout, h, wd
    a.gn_groups = gn[0] if gn else 0
    a.silu = int(silu)
    a.out_groups = out_groups
    a.act, a.engine = act, engine
    keep = [x.float().contiguous(), w.float().contiguous()]
    a.x, a.w = keep[0].data_ptr(), keep[1].data_ptr()
    if bias is not None:
        keep.append(bias.float().contiguous())
        a.bias = keep[-1].data_ptr()
    if gn:
        keep += [gn[1].float().contiguous(), gn[2].float().contiguous()]
        a.gn_gamma, a.gn_beta = keep[-2].data_ptr(), keep[-1].data_ptr()
    if temb is not None:
        keep.append(temb.float().contiguous())
        a.temb = keep[-1].data_ptr()
    assert h == wd
    y = torch.empty(b, cout, ho, ho, device=dev, dtype=torch.float32)
    a.y = y.data_ptr()
    stats = None
    if out_groups:
        stats = torch.empty(b, out_groups, 2, device=dev, dtype=torch.float32)
        a.out_stats = stats.data_ptr()
    scratch = torch.empty(lib.dmn_conv_scratch_bytes(C.byref(a)) + 256, dtype=torch.uint8, device=dev)
    a.scratch_dev = (scratch.data_ptr() + 255) // 256 * 256
    a.scratch_bytes = scratch.numel() - 256
    with torch.cuda.device(dev):
        if x2 is None:
            L.check(lib.dmn_conv_forward(C.byref(a), L.stream_ptr(dev)), "dmn_conv_forward")
        else:
            keep.append(x2.float().contiguous())
            L.check(lib.dmn_conv_forward_cat(C.byref(a), L.ptr(keep[-1]), cin2, L.stream_ptr(dev)), "dmn_conv_forward_cat")
    torch.cuda.synchronize(dev)
    return y, stats


LOG_INTS = 64


def conv_log(cap=4096):
    """Records of the tcgen05 conv launches since the previous call (dmn_debug_conv_log, a debug symbol outside the header; the
    first call starts the recording).  Each: dict of the launch parameters, the kernel's name and its tiling regime."""
    lib = L.lib()
    fn = lib.dmn_debug_conv_log
    fn.restype, fn.argtypes = C.c_int, [C.c_void_p, C.c_int]
    buf = (C.c_int32 * (LOG_INTS * cap))()
    n = fn(buf, cap)
    assert n <= cap, "launch log overflow"
    keys = ("fn_lo", "fn_hi", "geo", "ksize", "C1", "C2", "Cout", "H", "B", "pro", "pgroups", "ogroups", "swap", "atma", "mt",
            "n_big_tiles", "total_tiles", "grid", "threads", "n_tiles_n", "big_rows", "total_flat", "n_pass")
    out = []
    for i in range(n):
        r = buf[i * LOG_INTS:(i + 1) * LOG_INTS]
        d = dict(zip(keys, r))
        raw = b"".join(int(v & 0xffffffff).to_bytes(4, "little") for v in r[24:])
        d["name"] = raw.split(b"\0")[0].decode() or f"fn@{(d['fn_hi'] & 0xffffffff) << 32 | (d['fn_lo'] & 0xffffffff):x}"
        d["mixed"] = 0 < d["n_big_tiles"] < d["total_tiles"]
        d["multi"] = d["total_tiles"] > d["grid"]
        out.append(d)
    return out


def attention_core(qkv, linear, act=L.ACT_F32, heads=4, dh=32):
    lib = L.lib()
    dev = qkv.device
    b, c3, h, w = qkv.shape
    n = h * w
    out = torch.empty(b, heads * dh, h, w, device=dev, dtype=torch.float32)
    scratch = torch.empty(b * n * 4 * heads * dh * 4 + 1024, dtype=torch.uint8, device=dev)
    sp = (scratch.data_ptr() + 255) // 256 * 256
    fn = lib.dmn_linear_attention_core if linear else lib.dmn_attention_core
    q = qkv.float().contiguous()
    with torch.cuda.device(dev):
        L.check(fn(L.ptr(q), L.ptr(out), b, heads, dh, n, act, C.c_void_p(sp), scratch.numel() - 256, L.stream_ptr(dev)), "attention core")
    torch.cuda.synchronize(dev)
    return out


def linear_attention_block(x, sd, prefix, softmax=False):
    """Residual(PreNorm(LinearAttention)) -- or, with softmax=True, Residual(PreNorm(Attention)) -- through the fused tcgen05 kernel.
    x fp32 NCHW cuda; sd holds the reference parameter names under `prefix` (fn.norm.*, fn.fn.to_qkv.weight, fn.fn.to_out.0.* and
    fn.fn.to_out.1.* for the linear form, fn.fn.to_out.* for the softmax form)."""
    lib = L.lib()
    dev = x.device
    b, c, h, w = x.shape
    a = L.AttnBlockArgs()
    a.batch, a.dim, a.n_tokens, a.softmax = b, c, h * w, int(softmax)
    names = [".fn.norm.weight", ".fn.norm.bias", ".fn.fn.to_qkv.weight"]
    names += [".fn.fn.to_out.weight", ".fn.fn.to_out.bias"] if softmax else [".fn.fn.to_out.0.weight", ".fn.fn.to_out.0.bias",
                                                                              ".fn.fn.to_out.1.weight", ".fn.fn.to_out.1.bias"]
    keep = {k: sd[prefix + k].float().contiguous().to(dev) for k in names}
    xc = x.float().contiguous()
    y = torch.empty_like(xc)
    a.x, a.y = xc.data_ptr(), y.data_ptr()
    a.norm_w, a.norm_b = keep[".fn.norm.weight"].data_ptr(), keep[".fn.norm.bias"].data_ptr()
    a.w_qkv = keep[".fn.fn.to_qkv.weight"].data_ptr()
    if softmax:
        a.w_out, a.b_out = keep[".fn.fn.to_out.weight"].data_ptr(), keep[".fn.fn.to_out.bias"].data_ptr()
    else:
        a.w_out, a.b_out = keep[".fn.fn.to_out.0.weight"].data_ptr(), keep[".fn.fn.to_out.0.bias"].data_ptr()
        a.out_norm_w, a.out_norm_b = keep[".fn.fn.to_out.1.weight"].data_ptr(), keep[".fn.fn.to_out.1.bias"].data_ptr()
    scratch = torch.empty(lib.dmn_linear_attention_block_scratch_bytes(C.byref(a)) + 256, dtype=torch.uint8, device=dev)
    a.scratch_dev = (scratch.data_ptr() + 255) // 256 * 256
    a.scratch_bytes = scratch.numel() - 256
    with torch.cuda.device(dev):
        L.check(lib.dmn_linear_attention_block(C.byref(a), L.stream_ptr(dev)), "dmn_linear_attention_block")
    torch.cuda.synchronize(dev)
    return y

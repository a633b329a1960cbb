"""128x128 sampling: DDPM steps of the two 128x128 U-Nets (graph replay) and the bf16 softmax-attention core above 64 tokens.

Workloads (bf16 activations, tcgen05 convolutions, seeded random weights oracle.random_state_dict(seed=0), 3x128x128, B = --batch):
  A: Unet dim 128, dim_mults (1, 2, 2, 2)       bottleneck 16x16 = 256 tokens, C = 256
  B: Unet dim 64,  dim_mults (1, 2, 4, 8)       the reference constructor's defaults; bottleneck 256 tokens, C = 512
For each: K steps of the 1000-step linear DDPM schedule through the native loop (one CUDA graph replay per step, in-kernel Philox
noise), CUDA events around the K steps ending in a device synchronise, --repeats times: median ms per step, spread (max / min - 1),
samples/s for 1000 steps and the U-Net FLOP rate (oracle.unet_flops_per_sample).  Then the per-launch table of one forward (device
time stamps between the launches of one CUDA graph of the forward program) with the attention core's share of the step.
Last, attn_flash_kernel alone through dmn_attention_core (bf16) at N = 256, 1024 and 4096 tokens, B = --batch: CUDA events around
--core-iters calls (each includes the two layout conversions of the C ABI), and the kernel's share from torch.profiler in a separate
pass; FLOP/s from 4 N^2 * 32 * 4 heads per image (q k^T and P v).

    python tools/bench_hires.py [--batch 64] [--steps 20] [--repeats 5] [--out profiles/r08_bench_hires.json]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import diffusion_model_nemo_b200.modules as M  # noqa: E402
from diffusion_model_nemo_b200 import _lib as L  # noqa: E402
from diffusion_model_nemo_b200.modules import _runtime as R  # noqa: E402
from oracle import ref_port as O  # noqa: E402

S = 128
CFGS = {"A": dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8),
        "B": dict(dim=64, dim_mults=[1, 2, 4, 8], channels=3, groups=8)}
KIND = {0: "memset", 1: "init_conv", 2: "conv", 3: "gn_finalize", 4: "linattn_core", 5: "attn_core (attn_flash_kernel)",
        6: "final_proj", 7: "film_modulate", 8: "class_embed_add", 9: "attn_fused_tcgen05"}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return name, q


def bench_unet(name, batch, steps, repeats, dev):
    cfg = CFGS[name]
    u = M.Unet(None, dim=cfg["dim"], dim_mults=cfg["dim_mults"], channels=3, use_convnext=False, resnet_block_groups=8,
               compute_dtype="bf16", conv_engine="tcgen05")
    u.load_state_dict(O.random_state_dict(cfg, seed=0))
    u.to(dev)
    s = M.GaussianDiffusion(1000, "linear")
    coef, times = s._loop_tables(s._visit_order(), dev)
    shape = [batch, 3, S, S]
    plan = u.plan(S, batch, dev, time_rows=int(times.shape[0]))

    def run(res=None):
        return R.run_native_loop(u, kind=L.LOOP_DDPM, shape=shape, device=dev, times=times, coef=coef, seed=1234, use_graph=True,
                                 x_init=None if res is None else res.final, n_steps=steps)

    res = run()                      # uploads weights, captures the graph
    res = run(res)
    ms = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        res = run(res)
        e1.record()
        torch.cuda.synchronize(dev)
        ms.append(e0.elapsed_time(e1) / steps)
    assert torch.isfinite(res.final).all()
    med = statistics.median(ms)
    flops = O.unet_flops_per_sample(cfg, S)
    # per-launch table of one forward inside a CUDA graph
    ops = plan.op_table()
    row = torch.zeros(1, dtype=torch.int32, device=dev)
    x = res.final.clone()
    plan.profile_forward(x, row, in_graph=True)
    acc = [0.0] * len(ops)
    for _ in range(3):
        for i, v in enumerate(plan.profile_forward(x, row, in_graph=True)):
            acc[i] += v / 3
    table, groups = [], {}
    for (oname, kind, eng, fl, by), t in zip(ops, acc):
        key = KIND.get(kind, "other") + ("" if kind != 2 else (" tcgen05" if eng else " simt"))
        table.append({"op": oname, "kind": key, "engine": "tcgen05" if eng else "simt", "ms": round(t, 5),
                      "gflop": round(fl * batch / 1e9, 3)})
        g = groups.setdefault(key, {"ms": 0.0, "launches": 0})
        g["ms"] += t
        g["launches"] += 1
    fwd_ms = sum(acc)
    core_ms = sum(t for (_, kind, _, _, _), t in zip(ops, acc) if kind == 5)
    return {
        "config": name, "cfg": cfg, "batch": batch, "steps_timed": steps, "repeats": repeats,
        "ms_per_step_all": [round(v, 4) for v in ms], "ms_per_step_median": round(med, 4),
        "spread": round(max(ms) / min(ms) - 1, 4),
        "samples_per_s_1000_steps": round(batch / (1000 * med / 1e3), 3),
        "unet_gflop_per_sample": round(flops / 1e9, 3), "unet_tflops": round(flops * batch / (med / 1e3) / 1e12, 1),
        "forward_profile_ms": round(fwd_ms, 4), "attn_core_ms": round(core_ms, 4),
        "attn_core_share_of_forward": round(core_ms / fwd_ms, 4),
        "groups": {k: {"ms": round(v["ms"], 4), "launches": v["launches"]} for k, v in sorted(groups.items(), key=lambda kv: -kv[1]["ms"])},
        "per_launch": table,
    }


def bench_core(n, batch, iters, dev):
    lib = L.lib()
    side = int(round(n ** 0.5))
    assert side * side == n
    qkv = torch.randn(batch, 384, side, side, device=dev, generator=torch.Generator(device=dev).manual_seed(n))
    out = torch.empty(batch, 128, side, side, device=dev)
    scratch = torch.empty(batch * n * 512 * 4 + 1024, dtype=torch.uint8, device=dev)
    sp = C.c_void_p((scratch.data_ptr() + 255) // 256 * 256)

    def call():
        L.check(lib.dmn_attention_core(L.ptr(qkv), L.ptr(out), batch, 4, 32, n, L.ACT_BF16, sp, scratch.numel() - 256,
                                       L.stream_ptr(dev)), "dmn_attention_core")

    for _ in range(3):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for _ in range(iters):
        call()
    e1.record()
    torch.cuda.synchronize(dev)
    call_ms = e0.elapsed_time(e1) / iters
    # kernel time alone: torch.profiler (CUDA activities) in its own pass
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            call()
        torch.cuda.synchronize(dev)
    kus = [e.device_time_total for e in prof.key_averages() if "attn_flash_kernel" in e.key]
    kern_ms = kus[0] / iters / 1e3 if kus else None
    flop = 4.0 * n * n * 32 * 4 * batch
    r = {"n_tokens": n, "batch": batch, "iters": iters, "call_ms_incl_layout_conversions": round(call_ms, 4),
         "kernel_ms": None if kern_ms is None else round(kern_ms, 4), "gflop": round(flop / 1e9, 3)}
    if kern_ms:
        r["kernel_tflops"] = round(flop / (kern_ms / 1e3) / 1e12, 2)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--core-iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_hires: no CUDA device (timings are only meaningful on the GPU)")
    dev = torch.device("cuda:0")
    name, power = card()
    res = {"card": name, "power_limit_and_max_sm_clock": power, "image": [3, S, S], "dtype": "bf16", "conv_engine": "tcgen05",
           "sampler": "GaussianDiffusion(1000, linear), native DDPM loop, graph replay, in-kernel Philox",
           "unets": [bench_unet(k, args.batch, args.steps, args.repeats, dev) for k in ("A", "B")],
           "attn_core": [bench_core(n, args.batch, args.core_iters, dev) for n in (256, 1024, 4096)]}
    line = json.dumps(res)
    print(f"{name} [{power}]")
    for u in res["unets"]:
        print(f"{u['config']}: {u['ms_per_step_median']} ms/step (spread {u['spread']}), {u['samples_per_s_1000_steps']} samples/s "
              f"at 1000 steps, {u['unet_tflops']} TFLOP/s; attention core {u['attn_core_ms']} ms = "
              f"{100 * u['attn_core_share_of_forward']:.2f} % of the forward")
    for c in res["attn_core"]:
        print(f"core N={c['n_tokens']} B={c['batch']}: kernel {c['kernel_ms']} ms, {c.get('kernel_tflops')} TFLOP/s "
              f"(call incl. conversions {c['call_ms_incl_layout_conversions']} ms)")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()

"""RePaint inpainting (GaussianDiffusion.inpaint, one CUDA graph replay per event) against plain DDPM sampling.

Workload: the benchmark shape (B=256, 3x32x32, Unet dim 128 mults 1-2-2-2, bf16 activations / tcgen05 convolutions, seeded random
weights oracle.random_state_dict(seed=0)), linear schedule, graph mode, in-kernel noise from a fixed seed, a random known image with
its left half kept.  Timed alternately in one process, CUDA events around whole calls that end in a device synchronise and the copy
of the final images to the host:
  - sample() and inpaint() with jump_length = jump_n_sample = 1 at T = --steps (the same events and update rows);
  - RePaint's setting T = 250, jump_length = jump_n_sample = 10 (2410 events) against sample() at T = 250.
Reported: median ms per step / event, the overhead of an inpainting event over a plain step, kernel launches per step / event.

    python tools/bench_inpaint.py [--batch 256] [--repeats 5] [--steps 100] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import diffusion_model_nemo_b200.modules as M  # noqa: E402
from oracle import ref_port as O  # noqa: E402

CFG2 = dict(dim=128, dim_mults=[1, 2, 2, 2], channels=3, groups=8)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return name, q


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_inpaint needs a CUDA device")
    dev = torch.device("cuda:0")
    B = args.batch
    shape = [B, 3, 32, 32]
    unet = M.Unet(None, dim=CFG2["dim"], dim_mults=CFG2["dim_mults"], channels=3, use_convnext=False, resnet_block_groups=8,
                  compute_dtype="bf16", conv_engine="tcgen05")
    unet.load_state_dict(O.random_state_dict(CFG2, seed=0))
    unet.to(dev)
    known = torch.rand(shape, generator=torch.Generator().manual_seed(1)) * 2 - 1
    mask = torch.zeros(1, 1, 32, 32)
    mask[..., :16] = 1.0

    def launches():
        return unet.plan(32, B, dev).last_loop_launches

    rows = []
    for T, j, r in ((args.steps, 1, 1), (250, 10, 10)):
        s = M.GaussianDiffusion(T, "linear")
        s.seed = 0
        n_ev = len(s._inpaint_tables(j, r, dev)[3])
        run_sample = lambda: s.sample(unet, shape, device=dev)                                                # noqa: E731
        run_inpaint = lambda: s.inpaint(unet, known, mask, device=dev, jump_length=j, jump_n_sample=r)       # noqa: E731
        run_sample()                   # warm-up: graph capture and instantiation of both loops
        sample_launches = launches() / T
        run_inpaint()
        inpaint_launches = launches() / n_ev
        s_ms, i_ms = [], []
        for _ in range(args.repeats):
            t, out = timed(run_inpaint)
            i_ms.append(t)
            assert torch.isfinite(out[-1]).all()
            t, _ = timed(run_sample)
            s_ms.append(t)
        sm, im = statistics.median(s_ms) / T, statistics.median(i_ms) / n_ev
        rows.append({
            "T": T, "jump_length": j, "jump_n_sample": r, "events": n_ev,
            "sample_ms_per_call": [round(v, 3) for v in s_ms], "sample_ms_per_step": round(sm, 4),
            "sample_launches_per_step": sample_launches,
            "inpaint_ms_per_call": [round(v, 3) for v in i_ms], "inpaint_ms_per_event": round(im, 4),
            "inpaint_launches_per_event": inpaint_launches,
            "event_overhead_us": round((im - sm) * 1e3, 2), "event_overhead_rel": round(im / sm - 1.0, 4),
        })
        x = rows[-1]
        print(f"T={T} j={j} r={r} ({n_ev} events): sample {sm:.4f} ms/step ({sample_launches:g} launches), inpaint {im:.4f} ms/event "
              f"({inpaint_launches:g} launches); overhead {x['event_overhead_us']:+.2f} us = {100 * x['event_overhead_rel']:+.2f} %",
              flush=True)
    name, power = card()
    res = {
        "card": name, "power_limit_and_max_sm_clock": power, "batch": B, "shape": shape, "dtype": "bf16", "conv_engine": "tcgen05",
        "weights": "seeded random init (oracle.random_state_dict(seed=0))", "schedule": "linear", "graph": True,
        "mask": "left half kept", "repeats": args.repeats,
        "timing": "median of CUDA-event times of whole calls (device sync + D2H of the images)", "rows": rows,
    }
    line = json.dumps(res)
    print(line)
    print(f"{name} [{power}]")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

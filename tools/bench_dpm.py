"""DPM-Solver++ multistep sampler (DPMSolverDiffusion, one CUDA graph step per solver step) against DDIM at the same step count.

Workload: the benchmark shape (B=256, 3x32x32, Unet dim 128 mults 1-2-2-2, bf16 activations / tcgen05 convolutions, seeded random
weights oracle.random_state_dict(seed=0)), linear schedule T=1000, graph mode, x_T drawn in-kernel from a fixed seed.  For every
K in --steps and order in --orders, DPM-Solver++ and DDIM (eta = 0, ddim_timesteps = K: the same grid and U-Net time labels) are
timed alternately in the same process: CUDA events around whole sample() calls, each ending in a device synchronise and the copy of
the final images to the host.  Reported per step: the median call time over K, samples/s and kernel launches per step.

    python tools/bench_dpm.py [--batch 256] [--repeats 7] [--steps 10 20 50] [--orders 2 3] [--out FILE]
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
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--steps", type=int, nargs="+", default=[10, 20, 50])
    ap.add_argument("--orders", type=int, nargs="+", default=[2, 3])
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_dpm needs a CUDA device")
    dev = torch.device("cuda:0")
    B = args.batch
    shape = [B, 3, 32, 32]
    unet = M.Unet(None, dim=CFG2["dim"], dim_mults=CFG2["dim_mults"], channels=3, use_convnext=False, resnet_block_groups=8,
                  compute_dtype="bf16", conv_engine="tcgen05")
    unet.load_state_dict(O.random_state_dict(CFG2, seed=0))
    unet.to(dev)

    def launches_per_step(k):
        return unet.plan(32, B, dev).last_loop_launches / k

    rows = []
    for k in args.steps:
        ddim = M.GeneralizedGaussianDiffusion(1000, "linear", eta=0.0, ddim_timesteps=k)
        ddim.seed = 0
        n_steps = len(ddim.timestep_pairs())
        for order in args.orders:
            dpm = M.DPMSolverDiffusion(1000, "linear", steps=k, order=order)
            dpm.seed = 0
            run_dpm = lambda: dpm.sample(unet, shape, device=dev)      # noqa: E731
            run_ddim = lambda: ddim.sample(unet, shape, device=dev)    # noqa: E731
            run_dpm()                  # warm-up: graph capture and instantiation of both loops
            dpm_launches = launches_per_step(n_steps)
            run_ddim()
            ddim_launches = launches_per_step(n_steps)
            dpm_ms, ddim_ms = [], []
            for _ in range(args.repeats):
                t, out = timed(run_dpm)
                dpm_ms.append(t)
                assert torch.isfinite(out[-1]).all()
                t, _ = timed(run_ddim)
                ddim_ms.append(t)
            dm, gm = statistics.median(dpm_ms), statistics.median(ddim_ms)
            rows.append({
                "steps": n_steps, "order": order,
                "dpm_ms_per_call": [round(v, 3) for v in dpm_ms], "dpm_ms_per_step": round(dm / n_steps, 4),
                "dpm_samples_per_s": round(B / dm * 1e3, 1), "dpm_launches_per_step": dpm_launches,
                "ddim_ms_per_call": [round(v, 3) for v in ddim_ms], "ddim_ms_per_step": round(gm / n_steps, 4),
                "ddim_samples_per_s": round(B / gm * 1e3, 1), "ddim_launches_per_step": ddim_launches,
                "dpm_over_ddim": round(dm / gm - 1.0, 4),
            })
            r = rows[-1]
            print(f"K={n_steps} order {order}: DPM-Solver++ {r['dpm_ms_per_step']:.4f} ms/step ({r['dpm_samples_per_s']} samples/s, "
                  f"{dpm_launches:g} launches/step); DDIM {r['ddim_ms_per_step']:.4f} ms/step ({r['ddim_samples_per_s']} samples/s, "
                  f"{ddim_launches:g} launches/step); difference {100 * r['dpm_over_ddim']:+.2f} %", flush=True)
    name, power = card()
    res = {
        "card": name, "power_limit_and_max_sm_clock": power, "batch": B, "shape": shape, "dtype": "bf16", "conv_engine": "tcgen05",
        "weights": "seeded random init (oracle.random_state_dict(seed=0))", "schedule": "linear, T=1000", "graph": True,
        "repeats": args.repeats, "timing": "median of CUDA-event times of whole sample() calls (device sync + D2H of the images)",
        "rows": rows,
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

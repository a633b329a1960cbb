"""Probability-flow ODE sampler (device-side RK45, one CUDA graph per solve) against the PC loop, per model evaluation.

Workload: the benchmark shape (B=256, 3x32x32, Unet dim 128 mults 1-2-2-2, bf16 activations / tcgen05 convolutions, seeded random
weights oracle.random_state_dict(seed=0)), VP-SDE, ProbabilityFlowSampler with score_sde's default tolerances (1e-5).  The PC
reference point is the native PC loop with the reverse-diffusion predictor and no corrector, N steps = one U-Net evaluation and one
fused update kernel per step.  Both are timed in the same process, alternating, with CUDA events around whole sample() calls whose
x_T is already on the device; each call ends in a device synchronise.

    python tools/bench_ode.py [--batch 256] [--repeats 5] [--pc-steps 100] [--out FILE]
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
    ap.add_argument("--pc-steps", type=int, default=100)
    ap.add_argument("--rtol", type=float, default=1e-5)
    ap.add_argument("--atol", type=float, default=1e-5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_ode needs a CUDA device")
    dev = torch.device("cuda:0")
    B = args.batch
    shape = [B, 3, 32, 32]
    unet = M.Unet(None, dim=CFG2["dim"], dim_mults=CFG2["dim_mults"], channels=3, use_convnext=False, resnet_block_groups=8,
                  compute_dtype="bf16", conv_engine="tcgen05")
    unet.load_state_dict(O.random_state_dict(CFG2, seed=0))
    unet.to(dev)
    z = torch.randn([1] + shape, generator=torch.Generator().manual_seed(0)).to(dev)
    ode = M.ProbabilityFlowSampler(rtol=args.rtol, atol=args.atol)
    ode.update_sde(M.VPSDE())
    pc = M.PredictorCorrectorSampler("reverse_diffusion", "none", snr=0.16, n_steps=1, denoise=False)
    pc.update_sde(M.VPSDE(N=args.pc_steps))
    pc.seed = 0
    run_ode = lambda: ode.sample(unet, shape, device=dev, noise=z)        # noqa: E731
    run_pc = lambda: pc.sample(unet, shape, device=dev)                   # noqa: E731
    run_ode()                      # warm-up: plan, graph capture and instantiation of both paths
    run_pc()
    ode_ms, pc_ms, stats = [], [], None
    for _ in range(args.repeats):
        t, _ = timed(run_ode)
        ode_ms.append(t)
        stats = dict(ode.last_stats)
        t, _ = timed(run_pc)
        pc_ms.append(t)
    name, power = card()
    nfev = stats["nfev"]
    ode_per = statistics.median(ode_ms) / nfev
    pc_per = statistics.median(pc_ms) / args.pc_steps
    res = {
        "card": name, "power_limit_and_max_sm_clock": power, "batch": B, "shape": shape, "dtype": "bf16", "conv_engine": "tcgen05",
        "weights": "seeded random init (oracle.random_state_dict(seed=0))", "sde": "VPSDE(0.1, 20, 1000)",
        "rtol": args.rtol, "atol": args.atol, "nfev": nfev, "n_accepted": stats["n_accepted"], "n_rejected": stats["n_rejected"],
        "ode_ms_per_solve": [round(v, 3) for v in ode_ms], "ode_ms_per_solve_median": round(statistics.median(ode_ms), 3),
        "ode_ms_per_eval": round(ode_per, 4), "ode_samples_per_s": round(B / statistics.median(ode_ms) * 1e3, 1),
        "pc_steps": args.pc_steps, "pc_ms_per_loop": [round(v, 3) for v in pc_ms], "pc_ms_per_eval": round(pc_per, 4),
        "solver_overhead": round(ode_per / pc_per - 1.0, 4),
        "note": "evaluation counts from random-init weights say nothing about the step counts of a trained model",
    }
    line = json.dumps(res)
    print(line)
    print(f"{name} [{power}]: ODE nfev {nfev} ({stats['n_accepted']} accepted, {stats['n_rejected']} rejected), "
          f"{res['ode_ms_per_solve_median']} ms/solve, {ode_per:.4f} ms/eval; PC {pc_per:.4f} ms/eval; "
          f"solver overhead {100 * res['solver_overhead']:+.2f} %")
    print("note: evaluation counts from random-init weights say nothing about the step counts of a trained model")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

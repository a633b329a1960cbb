"""Few-step score-SDE sampling (DPMSolverSampler: DPM-Solver++ and SDE-DPM-Solver++, one CUDA graph replay per step) against the
PC loop, per step.

Workload: the U-Net of tools/bench_ode.py (B=256, 3x32x32, Unet dim 128 mults 1-2-2-2, bf16 activations / tcgen05 convolutions,
seeded random weights oracle.random_state_dict(seed=0)), VP-SDE(0.1, 20) and VE-SDE(0.01, 50), logSNR grid, order 2, graph mode,
every draw in-kernel from a fixed seed.  For each SDE, step count in --steps and algorithm, the sampler and the native PC loop
(reverse-diffusion predictor, no corrector, --pc-steps steps: one U-Net evaluation and one fused update per step) are timed
alternately in the same process: CUDA events around whole sample() calls, each ending in a device synchronise and the copy of the
final images to the host.  Reported: every call time, the median per step, the spread (max / min - 1) over the repeats and
samples/s.

    python tools/bench_score_dpm.py [--batch 256] [--repeats 7] [--steps 10 20] [--pc-steps 100] [--out FILE]
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
    ap.add_argument("--steps", type=int, nargs="+", default=[10, 20])
    ap.add_argument("--pc-steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_score_dpm needs a CUDA device")
    dev = torch.device("cuda:0")
    B = args.batch
    shape = [B, 3, 32, 32]
    unet = M.Unet(None, dim=CFG2["dim"], dim_mults=CFG2["dim_mults"], channels=3, use_convnext=False, resnet_block_groups=8,
                  compute_dtype="bf16", conv_engine="tcgen05")
    unet.load_state_dict(O.random_state_dict(CFG2, seed=0))
    unet.to(dev)

    def spread(v):
        return round(max(v) / min(v) - 1.0, 4)

    rows = []
    for sde_name, make_sde in (("VP", lambda n: M.VPSDE(0.1, 20, n)), ("VE", lambda n: M.VESDE(0.01, 50, n))):
        pc = M.PredictorCorrectorSampler("reverse_diffusion", "none", snr=0.16, n_steps=1, denoise=False)
        pc.update_sde(make_sde(args.pc_steps))
        pc.seed = 0
        for k in args.steps:
            for algorithm in ("dpmsolver++", "sde-dpmsolver++"):
                dpm = M.DPMSolverSampler(steps=k, order=2, algorithm_type=algorithm)
                dpm.update_sde(make_sde(1000))
                dpm.seed = 0
                run_dpm = lambda: dpm.sample(unet, shape, device=dev)      # noqa: E731
                run_pc = lambda: pc.sample(unet, shape, device=dev)        # noqa: E731
                run_dpm()                  # warm-up: plan, graph capture and instantiation of both loops
                run_pc()
                dpm_ms, pc_ms = [], []
                for _ in range(args.repeats):
                    t, out = timed(run_dpm)
                    dpm_ms.append(t)
                    assert torch.isfinite(out[-1]).all()
                    t, _ = timed(run_pc)
                    pc_ms.append(t)
                dm, pm = statistics.median(dpm_ms), statistics.median(pc_ms)
                rows.append({
                    "sde": sde_name, "steps": k, "algorithm": algorithm, "order": 2,
                    "dpm_ms_per_call": [round(v, 3) for v in dpm_ms], "dpm_ms_per_step": round(dm / k, 4),
                    "dpm_spread": spread(dpm_ms), "dpm_samples_per_s": round(B / dm * 1e3, 1),
                    "pc_steps": args.pc_steps, "pc_ms_per_call": [round(v, 3) for v in pc_ms],
                    "pc_ms_per_step": round(pm / args.pc_steps, 4), "pc_spread": spread(pc_ms),
                    "dpm_step_over_pc_step": round((dm / k) / (pm / args.pc_steps) - 1.0, 4),
                })
                r = rows[-1]
                print(f"{sde_name} {algorithm} K={k}: {r['dpm_ms_per_step']:.4f} ms/step (spread {100 * r['dpm_spread']:.2f} %), "
                      f"{r['dpm_samples_per_s']} samples/s; PC {r['pc_ms_per_step']:.4f} ms/step (spread {100 * r['pc_spread']:.2f} %); "
                      f"difference per step {100 * r['dpm_step_over_pc_step']:+.2f} %", flush=True)
    name, power = card()
    res = {
        "card": name, "power_limit_and_max_sm_clock": power, "batch": B, "shape": shape, "dtype": "bf16", "conv_engine": "tcgen05",
        "weights": "seeded random init (oracle.random_state_dict(seed=0))", "skip_type": "logSNR", "graph": True,
        "repeats": args.repeats, "timing": "CUDA-event times of whole sample() calls (device sync + D2H of the images); median per step",
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

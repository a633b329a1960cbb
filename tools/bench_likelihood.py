"""Probability-flow ODE likelihood (LikelihoodEstimate, one CUDA graph per solve) at the benchmark U-Net shape.

Workload: 3x32x32, Unet dim 128 mults 1-2-2-2 (cfg2), seeded random weights oracle.random_state_dict(seed=0), fp32 activations on the
SIMT engine (the only precision the JVP is built for), VP-SDE, score_sde's default tolerances (1e-5), Rademacher noise, data
uniform in [-1, 1].  For each batch size it records, in one process:
  * one U-Net forward and one JVP pass (dmn_unet_forward / dmn_unet_jvp), warm, CUDA events around `--passes` back-to-back calls;
  * one full likelihood solve after a warm-up solve (graph captured), CUDA events around likelihood(), which ends in a synchronise;
  * the card name and power limit.

    python tools/bench_likelihood.py [--batches 64 256] [--passes 5] [--out profiles/r06_bench_likelihood.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import diffusion_model_nemo_b200.modules as M  # noqa: E402
from oracle import ref_port as O  # noqa: E402
from tools.bench_ode import CFG2, card, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[64, 256])
    ap.add_argument("--passes", type=int, default=5)
    ap.add_argument("--rtol", type=float, default=1e-5)
    ap.add_argument("--atol", type=float, default=1e-5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_likelihood needs a CUDA device")
    dev = torch.device("cuda:0")
    unet = M.Unet(None, dim=CFG2["dim"], dim_mults=CFG2["dim_mults"], channels=3, use_convnext=False, resnet_block_groups=8,
                  compute_dtype="fp32", conv_engine="simt")
    unet.load_state_dict(O.random_state_dict(CFG2, seed=0))
    unet.to(dev)
    rows = []
    for B in args.batches:
        g = torch.Generator().manual_seed(0)
        x = (torch.rand(B, 3, 32, 32, generator=g) * 2 - 1).to(dev)
        v = torch.randn(B, 3, 32, 32, generator=g).to(dev)
        t = torch.full((B,), 500.0, device=dev)
        unet(x, t)
        unet.jvp(x, t, v)
        fwd_ms, _ = timed(lambda: [unet(x, t) for _ in range(args.passes)])
        jvp_ms, _ = timed(lambda: [unet.jvp(x, t, v) for _ in range(args.passes)])
        le = M.LikelihoodEstimate(rtol=args.rtol, atol=args.atol)
        le.update_sde(M.VPSDE())
        le.seed = 0
        le.likelihood(unet, x)                   # warm-up: graph capture and instantiation
        solve_ms, (bpd, _, nfe) = timed(lambda: le.likelihood(unet, x))
        row = {"batch": B, "forward_ms": fwd_ms / args.passes, "jvp_ms": jvp_ms / args.passes,
               "jvp_over_forward": jvp_ms / fwd_ms, "solve_nfe": nfe, "solve_s": solve_ms / 1e3,
               "solve_stats": le.last_stats, "bpd_mean": float(bpd.mean())}
        rows.append(row)
        print(json.dumps(row))
    name, q = card()
    out = {"workload": "cfg2 U-Net 3x32x32, random init seed 0, fp32 SIMT, VP-SDE, LikelihoodEstimate rtol=atol=%g, Rademacher" % args.rtol,
           "timing": "CUDA events; forward / JVP: mean of %d back-to-back warm calls (time table build included, as in Unet.forward); "
                     "solve: one warm likelihood() call (graph already captured)" % args.passes,
           "card": name, "power_limit_and_max_sm_clock": q, "rows": rows}
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

"""Cost of the opacity / scale regularisers in the fused Adam step (gut_optim.cu).

Times optimizers.FusedGaussianAdam.step at N Gaussians (default 300k, the C2 workload's N) in three variants, interleaved iteration by
iteration so that all three see the same machine state:
  off       gutb200_gaussian_adam_step (the plain step, as bench.py's optimizer_step times it)
  reg       gutb200_gaussian_adam_step_reg, lambda_opacity = lambda_scale = 0.01, no loss report
  reg_loss  the same plus the two loss values (block reductions + one atomic per block, and the zeroing of the two floats)
CUDA events around each step; a 256 MiB fill between timed steps overwrites L2 (126 MB), so parameters, moments and gradients come
from HBM.  Prints one JSON line (and writes it to --out if given), with the GPU's name and power limit beside the times.

    python scripts/adam_reg_cost.py [--n 300000] [--iters 200] [--out FILE]"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "3dgrut_b200")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

import optimizers  # noqa: E402

BYTES_PER_GAUSSIAN = 1660  # 59 floats x (param r/w + two moments r/w) + 240 B gradients + 4 B visibility (bench.py's optimizer_step)


def gpu_info(index: int) -> dict:
    info = {"name": torch.cuda.get_device_name(index)}
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30, check=True).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except (OSError, subprocess.SubprocessError, ValueError, IndexError) as e:
        info["power_limit_w"] = f"unavailable ({e!r})"
    return info


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--n", type=int, default=300_000)
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("adam_reg_cost.py needs a CUDA device: there is nothing to measure without one")
    dev = torch.device("cuda", 0)
    n = args.n
    g = torch.Generator(device=dev).manual_seed(5)
    widths = dict(zip(optimizers.GROUPS, optimizers.WIDTHS))
    leaves = {k: torch.randn((n, w), device=dev, generator=g) for k, w in widths.items()}
    lrs = dict(positions=1.6e-4, density=0.05, rotation=1e-3, scale=5e-3, features_albedo=2.5e-3, features_specular=1.25e-4)
    opt = optimizers.FusedGaussianAdam(leaves, lrs, eps=1e-15)
    dp = torch.randn((n, 12), device=dev, generator=g)
    ds = torch.randn((n, 48), device=dev, generator=g)
    reg_loss = torch.zeros(2, device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    variants = {
        "off": lambda: opt.step(dp, ds),
        "reg": lambda: opt.step(dp, ds, lambda_opacity=0.01, lambda_scale=0.01),
        "reg_loss": lambda: opt.step(dp, ds, lambda_opacity=0.01, lambda_scale=0.01, reg_loss=reg_loss),
    }
    for _ in range(args.warmup):
        for run in variants.values():
            run()
    torch.cuda.synchronize(dev)
    ms = {k: [] for k in variants}
    for i in range(args.iters):
        order = list(variants) if i % 2 == 0 else list(reversed(variants))
        for k in order:
            flush.fill_(float(i))
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            variants[k]()
            b.record()
            torch.cuda.synchronize(dev)
            ms[k].append(a.elapsed_time(b))
    stats = {}
    for k, v in ms.items():
        arr = np.asarray(v)
        med = float(np.median(arr))
        stats[k] = {"median_ms": med, "p10_ms": float(np.percentile(arr, 10)), "p90_ms": float(np.percentile(arr, 90)),
                    "algorithmic_gbs": BYTES_PER_GAUSSIAN * n / (med * 1e-3) / 1e9}
    line = {
        "what": "FusedGaussianAdam.step with and without the opacity / scale regularisers",
        "n": n, "iters": args.iters, "timing": "CUDA events per step, variants interleaved, L2 overwritten (256 MiB fill) before every step",
        "gpu": gpu_info(0), "variants": stats,
        "reg_over_off": stats["reg"]["median_ms"] / stats["off"]["median_ms"],
        "reg_loss_over_off": stats["reg_loss"]["median_ms"] / stats["off"]["median_ms"],
        "loss_values": [float(x) for x in reg_loss.cpu()],
    }
    text = json.dumps(line)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()

"""One PixelDiscriminator forward + backward (weight and feature gradients) at the adversarial shape (4 x 2048 x 64 x 128, ndf 256,
C = 19): K6 bf16, K6 TF32 (PixelDiscriminator.tf32), cuDNN with allow_tf32 and cuDNN strict fp32, alternated in one process.

    python profiles/time_disc_tf32.py [--iters 20] [--repeats 7] [--out results.json]

CUDA events around `iters` steps after warm-up; each arm's per-step time is the median over `repeats` windows, with the min / max of
those windows as its spread.  The TF32 arm's rate is credited with 3 x 10.1 MFLOP per pixel (forward, data and weight gradient of
the three layers) against the 1,125 TFLOP/s dense TF32 data-sheet figure.  Prints one JSON line (also written to --out if given).
The working set (x: 268 MB fp32) exceeds the 126 MB L2."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rnd_semantic_segmentation_b200 as b200  # noqa: E402
from oracle import torch_oracle as to  # noqa: E402

N, CIN, NDF, C, H, W = 4, 2048, 256, 19, 64, 128
FLOP = 3 * 10.1e6 * N * H * W


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # pragma: no cover - depends on the host
        q = f"unavailable ({e})"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--out", default=None, help="write the JSON result line here")
    args = ap.parse_args()
    torch.manual_seed(0)
    name, power = card()
    print(f"card: {name}, power limit / max SM clock: {power}")
    ref = to.PixelDiscriminatorOracle(CIN, NDF, num_classes=C).cuda()
    ours = b200.PixelDiscriminator(CIN, NDF, num_classes=C).cuda()
    ours.load_state_dict(ref.state_dict())
    ours_tf32 = b200.PixelDiscriminator(CIN, NDF, num_classes=C).cuda()
    ours_tf32.load_state_dict(ref.state_dict())
    ours_tf32.tf32 = True
    x = torch.relu(torch.randn(N, CIN, H, W, device="cuda")).requires_grad_(True)
    go = torch.randn(N, 2 * C, H, W, device="cuda") * 1e-3

    def step(module, allow_tf32=None):
        def run():
            if allow_tf32 is not None:
                torch.backends.cudnn.allow_tf32 = allow_tf32
            x.grad = None
            for p in module.parameters():
                p.grad = None
            module(x).backward(go)
        return run

    arms = {"k6_bf16": step(ours), "k6_tf32": step(ours_tf32), "cudnn_tf32": step(ref, True), "cudnn_fp32": step(ref, False)}
    for run in arms.values():                     # warm-up: modules, cuDNN algorithm choice, graph capture of the one-call entries
        for _ in range(5):
            run()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(args.repeats):
        for k, run in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                run()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) / args.iters)
    torch.backends.cudnn.allow_tf32 = True
    res = {"card": name, "power_limit_max_sm_clock": power, "shape": [N, CIN, H, W], "ndf": NDF, "C": C, "iters": args.iters,
           "repeats": args.repeats}
    for k, v in times.items():
        med = statistics.median(v)
        res[k] = {"median_ms": round(med, 4), "min_ms": round(min(v), 4), "max_ms": round(max(v), 4),
                  "tflops": round(FLOP / (med * 1e-3) / 1e12, 1)}
        print(f"{k:11s} {med:.3f} ms  [{min(v):.3f}, {max(v):.3f}]  {res[k]['tflops']} TFLOP/s")
    res["k6_tf32_share_of_1125_tflops"] = round(res["k6_tf32"]["tflops"] / 1125.0, 3)
    res["k6_tf32_faster_than_cudnn_tf32"] = res["k6_tf32"]["median_ms"] < res["cudnn_tf32"]["median_ms"]
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

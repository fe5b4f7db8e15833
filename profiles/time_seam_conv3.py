"""Fused backbone tail with conv3 (ops.seam_conv3_tail) against cuDNN conv3 + the tail, forward and backward separately.

    python profiles/time_seam_conv3.py [--out profiles/seam_conv3_b200.json]

At the bench shape (out2 8 x 512 x 64 x 128 -> features 8 x 2048 x 64 x 128) and the eval shape (1 x 512 x 128 x 256 -> 1 x 2048 x
128 x 256), three variants of the end of the last Bottleneck (resnet.py:106-113, bn3 folded to x * scale + bias), each producing the
bf16 channels_last features the head takes:
  - stock:       conv3 (cuDNN) + bn3 + add + relu in fp32, then .to(torch.bfloat16);
  - cudnn_tail:  conv3 (cuDNN) + ops.seam_tail (the fused fold tail);
  - conv3_fused: ops.seam_conv3_tail (feature pack + weight pack + one tcgen05 GEMM with the tail in its epilogue).
Forward: the three under no_grad.  Backward: one retained graph per variant, backward from the same bf16 dy to out2, identity and
conv3's weight.  Peak memory of one forward + backward above the inputs.  cuDNN runs under PyTorch's defaults (its TF32 flag is
recorded).  Times are CUDA events around many launches after warm-up, medians of alternating rounds; every working set is far larger
than the 126 MB L2.  Records the device name, power limit and max SM clock of the same run.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

import rnd_semantic_segmentation_b200 as b200
from time_seam_tail import alternate, device_info


def inputs(N, Cin, Cout, h, w, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    out2 = torch.relu(torch.randn(N, Cin, h, w, device="cuda", generator=g))
    identity = torch.relu(torch.randn(N, Cout, h, w, device="cuda", generator=g))
    W = torch.randn(Cout, Cin, 1, 1, device="cuda", generator=g) * (2.0 / Cin) ** 0.5
    scale = 0.5 + torch.rand(Cout, device="cuda", generator=g)
    bias = 0.1 * torch.randn(Cout, device="cuda", generator=g)
    return out2, identity, W, scale, bias


def variants(out2, identity, W, scale, bias):
    s, b = scale.view(1, -1, 1, 1), bias.view(1, -1, 1, 1)

    def stock():
        out = F.conv2d(out2, W) * s + b
        out += identity
        return torch.relu_(out).to(torch.bfloat16)

    return {"stock": stock,
            "cudnn_tail": lambda: b200.seam_tail(F.conv2d(out2, W), identity, scale, bias),
            "conv3_fused": lambda: b200.seam_conv3_tail(out2, identity, W, scale, bias)}


def measure(shape, res):
    N, Cin, Cout, h, w = shape
    key = "x".join(str(v) for v in shape)
    out2, identity, W, scale, bias = inputs(N, Cin, Cout, h, w, 1)
    fwd = variants(out2, identity, W, scale, bias)
    with torch.no_grad():
        ys = {k: f() for k, f in fwd.items()}
        t, spread = alternate(fwd, rounds=7, iters=20)
    for k in fwd:
        res[f"forward_{k}_{key}"] = {"us": round(t[k] * 1e3, 1), "us_min_max": [round(v * 1e3, 1) for v in spread[k]]}
        print(f"forward {k} {key}: {t[k] * 1e3:.1f} us", flush=True)
    d = (ys["conv3_fused"].float() - ys["stock"].float())
    res[f"forward_rel_l2_vs_stock_{key}"] = round((d.norm() / ys["stock"].float().norm()).item(), 6)
    del ys, d

    leaves = [t_.requires_grad_(True) for t_ in (out2, identity, W)]
    fwd = variants(out2, identity, W, scale, bias)
    dy = torch.randn(N, Cout, h, w, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    peaks = {}
    for k, f in fwd.items():
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        f().backward(dy)
        torch.cuda.synchronize()
        peaks[k] = torch.cuda.max_memory_allocated() - base
        for p in leaves:
            p.grad = None
    graphs = {k: f() for k, f in fwd.items()}

    def bwd(k):
        def run():
            for p in leaves:
                p.grad = None
            graphs[k].backward(dy, retain_graph=True)
        return run
    t, spread = alternate({k: bwd(k) for k in fwd}, rounds=7, iters=10)
    for k in fwd:
        res[f"backward_{k}_{key}"] = {"us": round(t[k] * 1e3, 1), "us_min_max": [round(v * 1e3, 1) for v in spread[k]],
                                      "peak_MB_above_inputs_fwd_bwd": round(peaks[k] / 1e6, 1)}
        print(f"backward {k} {key}: {t[k] * 1e3:.1f} us; peak above inputs (forward + backward) {peaks[k] / 1e6:.0f} MB", flush=True)
    del graphs, leaves, out2, identity, W, dy


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_seam_conv3.py measures on a CUDA device; none is available")
    torch.cuda.set_device(0)
    res = device_info()
    res["cudnn_allow_tf32"] = bool(torch.backends.cudnn.allow_tf32)
    print(res, flush=True)
    measure((8, 512, 2048, 64, 128), res)
    measure((1, 512, 2048, 128, 256), res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

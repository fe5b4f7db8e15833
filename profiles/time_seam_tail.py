"""Seam-format producer (ops.seam_tail): kernel times, and the step it changes, stock against fused.

    python profiles/time_seam_tail.py [--out profiles/seam_tail_b200.json]

At the bench shape (features 8 x 2048 x 64 x 128, C = 19 head, 512 x 1024 labels) and for one 1 x 2048 x 128 x 256 eval frame:
  - the tail kernels alone (forward, backward) with the achieved GB/s over their algorithmic bytes (fp32 c and identity read +
    bf16 y written; bf16 dy and y read + fp32 dc and didentity written) -- every pass moves > 1 GB, far more than the 126 MB L2;
  - stock tail (x * scale + bias, += identity, relu, fp32 NCHW) + forward_loss + backward to c / identity, against
    seam_tail + forward_loss on its bf16 channels_last output + the same backward, alternated, with the peak memory of each;
  - stock tail + head logits + segmentation_eval_step against the fused version, per frame.
Times are CUDA events around many launches after warm-up (medians of alternating rounds).  Prints the device name and power
limit of the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import rnd_semantic_segmentation_b200 as b200
from rnd_semantic_segmentation_b200 import _lib

RATES = [6, 12, 18, 24]
PEAK_TBS = 7.7                         # HBM3e data-sheet bandwidth of one B200


def device_info():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:                      # report, do not guess
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def time_ms(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def alternate(fns, rounds, iters):
    """{name: median ms} over `rounds` rounds that run every variant once per round, in turn."""
    got = {k: [] for k in fns}
    for k, f in fns.items():
        time_ms(f, 2)
    for _ in range(rounds):
        for k, f in fns.items():
            got[k].append(time_ms(f, iters, warm=1))
    return {k: statistics.median(v) for k, v in got.items()}, {k: (min(v), max(v)) for k, v in got.items()}


def tail_inputs(shape, seed, grad=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    c = torch.randn(shape, device="cuda", generator=g)
    identity = torch.relu(torch.randn(shape, device="cuda", generator=g))
    C = shape[1]
    scale = 0.5 + torch.rand(C, device="cuda", generator=g)
    bias = 0.1 * torch.randn(C, device="cuda", generator=g)
    if grad:
        c.requires_grad_(True)
        identity.requires_grad_(True)
    return c, identity, scale, bias


def stock_tail(c, identity, scale, bias):
    out = c * scale.view(1, -1, 1, 1) + bias.view(1, -1, 1, 1)       # FrozenBatchNorm2d (layers.py:17-23)
    out += identity                                                  # resnet.py:111-112
    return torch.relu_(out)


def kernels(shape, res):
    n = 1
    for s in shape:
        n *= s
    c, identity, scale, bias = tail_inputs(shape, 1)
    y = _lib.seam_tail_forward(c, identity, scale, bias)
    dy = torch.randn(shape, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    fwd_bytes, bwd_bytes = n * (4 + 4 + 2), n * (2 + 2 + 4 + 4)
    t, spread = alternate({"fwd": lambda: _lib.seam_tail_forward(c, identity, scale, bias),
                           "bwd": lambda: _lib.seam_tail_backward(dy, y, scale)}, rounds=5, iters=20)
    key = "x".join(str(s) for s in shape)
    for k, nbytes in (("fwd", fwd_bytes), ("bwd", bwd_bytes)):
        tbs = nbytes / (t[k] * 1e-3) / 1e12
        res[f"kernel_{k}_{key}"] = {"us": round(t[k] * 1e3, 1), "us_min_max": [round(v * 1e3, 1) for v in spread[k]],
                                    "MB": round(nbytes / 1e6, 1), "TB_s": round(tbs, 2), "of_7.7TB_s": round(tbs / PEAK_TBS, 3)}
        print(f"{k} {key}: {t[k] * 1e3:.1f} us  {nbytes / 1e6:.0f} MB  {tbs:.2f} TB/s = {tbs / PEAK_TBS:.3f} of {PEAK_TBS} TB/s",
              flush=True)
    del c, identity, y, dy


def train(res):
    shape = (8, 2048, 64, 128)
    c, identity, scale, bias = tail_inputs(shape, 2, grad=True)
    torch.manual_seed(3)
    head = b200.ASPP_Classifier_V2(2048, RATES, RATES, 19).cuda()
    labels = torch.randint(0, 19, (8, 512, 1024), device="cuda")

    def step(fused):
        c.grad = identity.grad = None
        for p in head.parameters():
            p.grad = None
        feat = b200.seam_tail(c, identity, scale, bias) if fused else stock_tail(c, identity, scale, bias)
        loss, _ = head.forward_loss(feat, labels)
        loss.backward()

    peaks = {}
    for name, fused in (("stock", False), ("fused", True)):
        step(fused)
        torch.cuda.synchronize()
        c.grad = identity.grad = None
        for p in head.parameters():
            p.grad = None
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        step(fused)
        torch.cuda.synchronize()
        peaks[name] = torch.cuda.max_memory_allocated() - base
    t, spread = alternate({"stock": lambda: step(False), "fused": lambda: step(True)}, rounds=5, iters=10)
    res["train_step_bench_shape"] = {k: {"ms": round(t[k], 4), "ms_min_max": [round(v, 4) for v in spread[k]],
                                         "peak_MB_above_inputs": round(peaks[k] / 1e6, 1)} for k in t}
    print(f"train step (tail + forward_loss + backward): stock {t['stock']:.3f} ms, fused {t['fused']:.3f} ms; peak above inputs "
          f"stock {peaks['stock'] / 1e6:.0f} MB, fused {peaks['fused'] / 1e6:.0f} MB", flush=True)
    del c, identity, head


def evaluate(res):
    shape = (1, 2048, 128, 256)
    c, identity, scale, bias = tail_inputs(shape, 4)
    torch.manual_seed(5)
    head = b200.ASPP_Classifier_V2(2048, RATES, RATES, 19).cuda().eval()
    labels = torch.randint(0, 19, (1, 1024, 2048), device="cuda")
    cm = torch.zeros(19, 19, dtype=torch.int64, device="cuda")

    def frame(fused):
        with torch.no_grad():
            feat = b200.seam_tail(c, identity, scale, bias) if fused else stock_tail(c, identity, scale, bias)
            b200.segmentation_eval_step(head.logits(feat), labels, cm=cm)

    t, spread = alternate({"stock": lambda: frame(False), "fused": lambda: frame(True)}, rounds=5, iters=20)
    res["eval_frame_1x2048x128x256"] = {k: {"ms": round(t[k], 4), "ms_min_max": [round(v, 4) for v in spread[k]],
                                            "img_s": round(1e3 / t[k], 1)} for k in t}
    print(f"eval frame (tail + head + argmax/confusion): stock {t['stock']:.3f} ms, fused {t['fused']:.3f} ms", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_seam_tail.py measures on a CUDA device; none is available")
    torch.cuda.set_device(0)
    res = device_info()
    print(res, flush=True)
    kernels((8, 2048, 64, 128), res)
    kernels((1, 2048, 128, 256), res)
    train(res)
    evaluate(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

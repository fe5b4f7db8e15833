"""Seam-format tail with batch statistics (ops.seam_tail_bn): kernel times, and the train step it changes, stock against fused.

    python profiles/time_seam_tail_bn.py [--out profiles/seam_tail_bn_b200.json]

At the bench shape (features 8 x 2048 x 64 x 128) and at cfg4's per-GPU 1 x 2048 x 64 x 128:
  - the five passes alone, with the achieved TB/s over their algorithmic bytes (n elements): statistics reads c (4n); the combine
    is [C]-sized (time only); the forward apply reads c and identity and writes bf16 y (10n); the backward reduce reads bf16 dy,
    bf16 y and c (8n); the backward apply reads the same and writes fp32 dc and didentity (16n) -- every pass but the combine
    moves more than 0.5 GB at the bench shape, far more than the 126 MB L2;
  - at the bench shape, a training-mode BatchNorm2d tail (F.batch_norm, += identity, relu, fp32 NCHW) + forward_loss + backward to
    c / identity / the norm's weight and bias, against seam_tail_bn + forward_loss on its bf16 channels_last output + the same
    backward, alternated, with the peak memory of each.
Times are CUDA events around many launches after warm-up (medians of alternating rounds).  Prints the device name and power
limit of the same run.
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
from rnd_semantic_segmentation_b200 import _lib
from time_seam_tail import PEAK_TBS, RATES, alternate, device_info


def bn_inputs(shape, seed, grad=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    C = shape[1]
    c = torch.randn(shape, device="cuda", generator=g)
    identity = torch.relu(torch.randn(shape, device="cuda", generator=g))
    weight = 0.5 + torch.rand(C, device="cuda", generator=g)
    bias = 0.1 * torch.randn(C, device="cuda", generator=g)
    if grad:
        for t in (c, identity, weight, bias):
            t.requires_grad_(True)
    return c, identity, weight, bias


def kernels(shape, res):
    n = 1
    for s in shape:
        n *= s
    C = shape[1]
    c, identity, weight, bias = bn_inputs(shape, 1)
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    record = _lib.bn_stats(c)
    mean, invstd, count = _lib.bn_combine_stats(record, 1e-5, 0.1, rm, rv)
    y = _lib.seam_tail_bn_forward(c, identity, mean, invstd, weight, bias)
    dy = torch.randn(shape, device="cuda").to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    sums, _, _ = _lib.seam_tail_bn_backward_reduce(dy, y, c, mean, invstd, True, True)
    fns = {"stats": lambda: _lib.bn_stats(c),
           "combine": lambda: _lib.bn_combine_stats(record, 1e-5, 0.1, rm, rv),
           "fwd_apply": lambda: _lib.seam_tail_bn_forward(c, identity, mean, invstd, weight, bias),
           "bwd_reduce": lambda: _lib.seam_tail_bn_backward_reduce(dy, y, c, mean, invstd, True, True),
           "bwd_apply": lambda: _lib.seam_tail_bn_backward(dy, y, c, mean, invstd, weight, sums, count)}
    nbytes = {"stats": 4 * n, "combine": None, "fwd_apply": 10 * n, "bwd_reduce": 8 * n, "bwd_apply": 16 * n}
    t, spread = alternate(fns, rounds=5, iters=20)
    key = "x".join(str(s) for s in shape)
    for k in fns:
        entry = {"us": round(t[k] * 1e3, 1), "us_min_max": [round(v * 1e3, 1) for v in spread[k]]}
        line = f"{k} {key}: {t[k] * 1e3:.1f} us"
        if nbytes[k]:
            tbs = nbytes[k] / (t[k] * 1e-3) / 1e12
            entry.update({"MB": round(nbytes[k] / 1e6, 1), "TB_s": round(tbs, 2), "of_7.7TB_s": round(tbs / PEAK_TBS, 3)})
            line += f"  {nbytes[k] / 1e6:.0f} MB  {tbs:.2f} TB/s = {tbs / PEAK_TBS:.3f} of {PEAK_TBS} TB/s"
        res[f"kernel_{k}_{key}"] = entry
        print(line, flush=True)
    del c, identity, y, dy


def train(res):
    shape = (8, 2048, 64, 128)
    C = shape[1]
    c, identity, weight, bias = bn_inputs(shape, 2, grad=True)
    rm, rv = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
    nbt = torch.zeros((), dtype=torch.int64, device="cuda")
    torch.manual_seed(3)
    head = b200.ASPP_Classifier_V2(2048, RATES, RATES, 19).cuda()
    labels = torch.randint(0, 19, (8, 512, 1024), device="cuda")
    leaves = [c, identity, weight, bias] + list(head.parameters())

    def step(fused):
        for p in leaves:
            p.grad = None
        if fused:
            feat = b200.seam_tail_bn(c, identity, weight, bias, rm, rv, nbt, 0.1, 1e-5)
        else:                                            # training-mode BatchNorm2d (resnet.py:106-113)
            feat = F.batch_norm(c, rm, rv, weight, bias, True, 0.1, 1e-5)
            feat += identity
            feat = torch.relu_(feat)
        loss, _ = head.forward_loss(feat, labels)
        loss.backward()

    peaks = {}
    for name, fused in (("stock", False), ("fused", True)):
        step(fused)
        torch.cuda.synchronize()
        for p in leaves:
            p.grad = None
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        step(fused)
        torch.cuda.synchronize()
        peaks[name] = torch.cuda.max_memory_allocated() - base
    t, spread = alternate({"stock": lambda: step(False), "fused": lambda: step(True)}, rounds=5, iters=10)
    res["train_step_bench_shape"] = {k: {"ms": round(t[k], 4), "ms_min_max": [round(v, 4) for v in spread[k]],
                                         "peak_MB_above_inputs": round(peaks[k] / 1e6, 1)} for k in t}
    print(f"train step (training-mode BN tail + forward_loss + backward): stock {t['stock']:.3f} ms, fused {t['fused']:.3f} ms; "
          f"peak above inputs stock {peaks['stock'] / 1e6:.0f} MB, fused {peaks['fused'] / 1e6:.0f} MB", flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="write the results as JSON here")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_seam_tail_bn.py measures on a CUDA device; none is available")
    torch.cuda.set_device(0)
    res = device_info()
    print(res, flush=True)
    kernels((8, 2048, 64, 128), res)
    kernels((1, 2048, 64, 128), res)
    train(res)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()

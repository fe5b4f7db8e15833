"""Memory-bound passes of the train step and the eval frame: kernel times and achieved bandwidth.

    python profiles/time_memory_passes.py [--out profiles/memory_passes_b200.json]
    B200SEG_LIB=/path/to/other/libb200seg.so python profiles/time_memory_passes.py --out /tmp/other.json    # A/B

Times, with the GB/s over each pass's algorithmic bytes:
  - the feature pack (fp32 NCHW -> bf16 [P, Cin]) at the bench shape 8 x 2048 x 64 x 128, the eval frame 1 x 2048 x 128 x 256
    and one domain of the adversarial step 4 x 2048 x 64 x 128;
  - the seam-tail forward (fp32 c + identity -> bf16 channels_last) at the bench shape;
  - the discriminator's gradient layout change 4 x 38 x 64 x 128 -> pitch 40;
  - the backward prologue of the fused train slice at the bench shape (C = 19, 512 x 1024 labels): the packed K2 finalize
    with the bias gradient (reads the K2 partial blocks and the bias partials, writes the bf16 class planes gOc) and the
    G'^t build (reads gOc, writes NJ x P bf16), each alone and both in sequence.
Passes of 100 us and more are timed with CUDA events around back-to-back calls; the prologue kernels are captured 20 times
into one CUDA graph that is replayed, so no host overhead enters.  Medians of alternating rounds.  The pack and tail
inputs are > 500 MB each (far more than the 126 MB L2); the prologue's 2.5 MB gOc is read from L2 by design (33 taps read
each class plane).  Prints and records the device name and power limit of the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from rnd_semantic_segmentation_b200 import _lib

RATES = [6, 12, 18, 24]
PEAK_TBS = 7.7                         # HBM3e data-sheet bandwidth of one B200


def device_info():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    info = {"device": torch.cuda.get_device_name(0), "library": os.path.relpath(_lib.LIB_PATH, root)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:                      # report, do not guess
        info["power_limit_and_max_sm_clock"] = f"unavailable ({e})"
    return info


def time_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def graphed(fn, reps=20):
    """fn captured `reps` times into one CUDA graph; returns (replay, calls per replay)."""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    return g.replay, reps


def alternate(fns, rounds=7, iters=10):
    """{name: (median ms per call, min, max)} over rounds that run every variant once, in turn."""
    got = {k: [] for k in fns}
    for k, (f, per) in fns.items():
        time_ms(f, 2)
    for _ in range(rounds):
        for k, (f, per) in fns.items():
            got[k].append(time_ms(f, iters) / per)
    return {k: (statistics.median(v), min(v), max(v)) for k, v in got.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "memory_passes_b200.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    res = {"info": device_info(), "passes": {}}
    print(json.dumps(res["info"]), flush=True)
    gen = torch.Generator(device="cuda").manual_seed(0)
    fns, nbytes = {}, {}

    feats = {"pack_bench_8x2048x64x128": (8, 2048, 64, 128), "pack_eval_1x2048x128x256": (1, 2048, 128, 256),
             "pack_adv_4x2048x64x128": (4, 2048, 64, 128)}
    xs = {}
    for name, shape in feats.items():
        xs[name] = torch.randn(shape, device="cuda", generator=gen)
        n = xs[name].numel()
        fns[name] = ((lambda x=xs[name]: _lib.aspp_pack_features(x)), 1)
        nbytes[name] = n * (4 + 2)

    shape = (8, 2048, 64, 128)
    c = xs["pack_bench_8x2048x64x128"]
    identity = torch.relu(torch.randn(shape, device="cuda", generator=gen))
    scale = 0.5 + torch.rand(2048, device="cuda", generator=gen)
    bias = 0.1 * torch.randn(2048, device="cuda", generator=gen)
    fns["seam_tail_fwd_8x2048x64x128"] = ((lambda: _lib.seam_tail_forward(c, identity, scale, bias)), 1)
    nbytes["seam_tail_fwd_8x2048x64x128"] = c.numel() * (4 + 4 + 2)

    gd = torch.randn(4, 38, 64, 128, device="cuda", generator=gen)
    fns["disc_grad_4x38x64x128_pitch40"] = graphed(lambda: _lib.nchw_to_nhwc_bf16(gd, 40))
    nbytes["disc_grad_4x38x64x128_pitch40"] = gd.numel() * 4 + 4 * 64 * 128 * 40 * 2

    # backward prologue at the bench shape
    N, C, h, w, H, W = 8, 19, 64, 128, 512, 1024
    logits = torch.randn(N, C, h, w, device="cuda", generator=gen)
    labels = torch.randint(0, C, (N, H, W), device="cuda", generator=gen)
    out2, ws = _lib.upsample_ce_forward(logits, labels)
    NJ = -(-(8 * len(RATES) + 1) * C // 128) * 128
    P = N * h * w
    WpT = torch.zeros(2048, NJ, dtype=torch.bfloat16, device="cuda")
    gOt, _ = _lib.upsample_ce_backward_packed(ws, out2, (N, C, h, w), (H, W))
    fin = lambda: _lib.upsample_ce_backward_packed(ws, out2, (N, C, h, w), (H, W), want_bias=True)
    gpr = lambda: _lib.aspp_backward_packed(gOt, None, WpT, RATES, N, h, w, C, need_grad_x=False, need_grad_w=False)
    fns["prologue_finalize_and_bias"] = graphed(fin)
    fns["prologue_gprime_build"] = graphed(gpr)
    fns["prologue_total"] = graphed(lambda: (fin(), gpr()))
    nblk = N * h * -(-w // 128)
    blocks_bytes = int(ws.numel()) - nblk * 32 * 4 - 256      # partial blocks + loss partials (upper bound of what is read)
    fin_bytes = blocks_bytes + nblk * 32 * 4 + P * C * 2
    gpr_bytes = NJ * P * 2 + P * C * 2
    nbytes["prologue_finalize_and_bias"] = fin_bytes
    nbytes["prologue_gprime_build"] = gpr_bytes
    nbytes["prologue_total"] = fin_bytes + gpr_bytes

    t = alternate(fns)
    for k, (med, lo, hi) in t.items():
        tbs = nbytes[k] / (med * 1e-3) / 1e12
        res["passes"][k] = {"us": round(med * 1e3, 1), "us_min_max": [round(lo * 1e3, 1), round(hi * 1e3, 1)],
                            "MB": round(nbytes[k] / 1e6, 1), "GB_s": round(tbs * 1e3), "of_7.7TB_s": round(tbs / PEAK_TBS, 3)}
        print(f"{k:34s} {med * 1e3:7.1f} us  [{lo * 1e3:.1f}, {hi * 1e3:.1f}]  {nbytes[k] / 1e6:7.1f} MB  {tbs * 1e3:6.0f} GB/s",
              flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()

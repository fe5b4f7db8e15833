#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native segmentation hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  Metric (BASELINE.json): ASPP+CE train Mpx/s -- label pixels per second
through  features -> ASPP head fwd -> upsample+CE fwd -> CE/upsample bwd -> head dgrad+wgrad (+ mean
all-reduce of the head gradients when N > 1) -- with eval img/s @1024x2048 (head fwd + upsample/argmax/
confusion matrix) reported in the same line under "eval".  Synthetic Cityscapes-shaped data, random-init head.

Under torchrun (N > 1) every rank runs the same per-GPU workload (weak scaling, batch sharded by image,
frames rank::world); time is the max over ranks, measured with CUDA events between barriers.

--dump-outputs DIR writes what the headline train step returned in its last timed step (loss, low-res logits, parameter
gradients, a fixed seeded sample of the feature gradient) as DIR/<name>.npy.  The inputs are seeded, so two builds can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

RATES = [6, 12, 18, 24]
F_FWD_PER_PX = 2 * 36 * 2048 * 19        # dense-tap convention, SURVEY.md section 8d (Cin=2048, C=19)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def workload_config(workload, world):
    """The `config` object of the JSON line: the workload only, byte-identical from both arms (``--impl ours`` / ``--impl
    reference``) so the driver's same_config check holds.  Everything measured lives in other keys."""
    from rnd_semantic_segmentation_b200 import synth
    n, cin, h, w, H, W, C = synth.WORKLOADS[workload]
    return {"workload": workload, "features": [n, cin, h, w], "labels": [n, H, W], "num_classes": C,
            "input": "fp32 NCHW layer4 features + int64 labels (the reference API contract), synthetic, seed 1234 + rank",
            "step": "ASPP head fwd + align-corners upsample + CrossEntropyLoss(ignore_index=255) fwd + backward (dX, dW, db)"
                    " [aspp_trainer.py:88-92 after the backbone]; N > 1: + mean all-reduce of the head gradients",
            "l2": "inputs larger than L2 (features %d MB per step)" % (n * cin * h * w * 4 // 2 ** 20),
            "parallelism": "dp%d (batch sharded by image, weak scaling)" % world}


def load_traffic(kernel_key):
    """dram bytes per launch of the dominant kernel from the committed `ncu --set full` summary (profiles/), or None."""
    path = os.path.join(ROOT, "profiles", "ncu_summary.json")
    try:
        with open(path) as f:
            return json.load(f)["kernels"][kernel_key]["dram_bytes_per_launch"]
    except Exception:
        return None


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], bf16_tflops_sustained=p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (rank 0)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        busy = [v for v in sm if smax and v > 0.5 * smax] or sm
        med = busy[len(busy) // 2] if busy else None
        return {"sm_mhz": med, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def barrier():
    if dist.is_available() and dist.is_initialized():
        dist.barrier()


def max_over_ranks(ms: float) -> float:
    if dist.is_available() and dist.is_initialized():
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return ms


def timed(step_fn, steps, warmup, sampler=None):
    """W untimed warm-ups, then exactly K steps between barrier + synchronize, CUDA events on the launching stream.
    The clock sampler (an nvidia-smi subprocess on rank 0) is started BEFORE the warm-up: it then samples the same workload
    under load for the warm-up plus the timed region, and its fork cannot desynchronise the ranks between the barrier and
    the first timed step."""
    if sampler:
        sampler.start()
    for _ in range(warmup):
        step_fn()
    torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        step_fn()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop() if sampler else None
    return max_over_ranks(e0.elapsed_time(e1)), clocks


DUMP_SAMPLE = 1 << 22                    # elements kept of an output larger than this (16 MB in float32)
DUMP_LIMIT_BYTES = 64 << 20


def seeded_sample(t, n=DUMP_SAMPLE, seed=0):
    """n elements of t at positions drawn from a fixed CPU generator: the same positions on every run for the same shape."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= n:
        return flat
    idx = torch.randint(0, flat.numel(), (n,), generator=torch.Generator().manual_seed(seed))
    return flat[idx.to(flat.device)]


def dump_outputs(out_dir, arrays):
    """Writes each tensor as out_dir/<name>.npy: float64 stays float64, everything else becomes float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    host = {name: t.detach().to(torch.float64 if t.dtype == torch.float64 else torch.float32).cpu().numpy()
            for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"dumped {len(host)} arrays ({total / 2 ** 20:.1f} MB) to {out_dir}")


class HostPipelinedStep:
    """End-to-end step from HOST buffers: every call copies that call's inputs host->device from pinned memory and reads the
    step's scalar result back (both inside the caller's timed region).  Double-buffered: the copy of call k+1's inputs is
    issued on a copy stream before call k's compute, so PCIe transfer and compute overlap -- per-step time is
    max(H2D, compute + D2H) instead of their sum."""

    def __init__(self, dev, host_tensors, compute):
        self.dev, self.host, self.compute = dev, host_tensors, compute
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.bufs = [[torch.empty_like(t, device=dev) for t in host_tensors] for _ in range(2)]
        self.ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.free = [torch.cuda.Event(), torch.cuda.Event()]
        self.k = 0
        self._issue(0)

    def _issue(self, slot):
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.free[slot])            # the compute that last read this slot is done
            for d, h in zip(self.bufs[slot], self.host):
                d.copy_(h, non_blocking=True)
            self.ready[slot].record(self.copy_stream)

    def __call__(self):
        slot = self.k & 1
        self.k += 1
        self._issue(slot ^ 1)                                        # next call's inputs go in flight first
        cur = torch.cuda.current_stream()
        cur.wait_event(self.ready[slot])
        out = self.compute(*self.bufs[slot])
        self.free[slot].record(cur)
        return out.item() if torch.is_tensor(out) and out.numel() == 1 else out.cpu()


# ----------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------
def run_ours(args):
    import rnd_semantic_segmentation_b200 as b200
    from rnd_semantic_segmentation_b200 import _lib, distributed as D, synth
    rank, world, local = D.env_rank_world()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the b200seg path has no CPU fallback")
    torch.cuda.set_device(local)
    D.init_from_env("nccl")
    dev = torch.device("cuda", local)
    peaks = load_peaks()
    _lib.load()

    n, cin, h, w, H, W, C = synth.WORKLOADS[args.workload]
    # the loops below feed the SAME synthetic feature tensor every step; the cross-module conversion cache would turn the
    # per-step fp32 -> bf16 feature pack into a hit, i.e. skip work a real iteration (new features every step) performs
    b200.set_feature_pack_cache(0)
    torch.manual_seed(1234)
    head = b200.ASPP_Classifier_V2(cin, RATES, RATES, C).to(dev)
    x = synth.make_features(n, cin, h, w, seed=1234 + rank, device=dev)
    labels = synth.make_labels(n, H, W, C, seed=1234 + rank, device=dev)
    bucket = D.HeadGradBucket(head) if world > 1 else None
    label_px = n * H * W
    head_params = list(head.parameters())                  # (an optimizer holds this list; zero_grad() walks it)
    # --dump-outputs: what the last timed step returned, kept from that step only, so that no earlier step's outputs stay
    # alive into the next timed step (timed() makes warmup + steps calls)
    last = {} if args.dump_outputs else None
    calls_left = [args.warmup + args.steps]

    def train_step(x_in=x, labels_in=labels):
        xg = x_in.detach().requires_grad_(True)            # the backbone needs d loss / d features
        for p in head_params:
            p.grad = None
        # (the module is in training mode: the bf16 weight pack is rebuilt on every call, as after every optimizer step)
        # N > 1: weight gradients land in the flat bucket and its NCCL mean all-reduce runs on a second stream underneath
        # the data-gradient GEMM; wait() joins the streams (the all-reduce is inside the timed step)
        loss, logits_lr = head.forward_loss(xg, labels_in, grad_bucket=bucket)
        loss.backward()
        if bucket is not None:
            bucket.wait()
        if last is not None:
            calls_left[0] -= 1
            if calls_left[0] == 0:                           # (detached: a live autograd graph would break the graph-capture leg)
                last.update(loss=loss.detach(), logits_lr=logits_lr, grad_x=xg.grad)
        return loss, xg.grad

    launches0 = _lib.launch_count()
    sampler = ClockSampler(local) if rank == 0 else None
    ms, clocks = timed(train_step, args.steps, args.warmup, sampler)
    launches = _lib.launch_count() - launches0 - 0
    launches_timed = launches * args.steps // (args.steps + args.warmup)
    if last is not None and rank == 0:
        # the later legs call train_step again: dump the headline's last timed step now.  The feature gradient has as many
        # elements as the features (8 x 2048 x 64 x 128 by default): a fixed seeded sample of it is kept.
        dump_outputs(args.dump_outputs, {"loss": last["loss"], "logits_lr": last["logits_lr"], "grad_x_sample": seeded_sample(last["grad_x"]),
                                         **{"grad." + name: p.grad for name, p in head.named_parameters()}})
    last = None
    ms_per_step = ms / args.steps
    value = world * label_px / (ms_per_step * 1e-3) / 1e6

    # ---- per-kernel CUDA-event timing (separate pass; events on the launching stream) -> roofline
    _lib.profile_enable(True)
    for _ in range(args.steps):
        train_step()
    torch.cuda.synchronize()
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    P = n * h * w
    flops_per_launch = 2.0 * 36 * cin * C * P
    gemm_names = ("head_fwd_gemm", "head_dgrad_gemm", "head_wgrad_gemm")
    gemm_ms = sum(prof[k][0] for k in gemm_names if k in prof)
    gemm_n = sum(prof[k][1] for k in gemm_names if k in prof)
    avg_ms = gemm_ms / max(gemm_n, 1)
    achieved = flops_per_launch / (avg_ms * 1e-3) / 1e12 if avg_ms > 0 else 0.0
    # peak: the measured cuBLAS bf16 number for the clock regime this run was in -- BURST (1653 TFLOP/s, SMs at their maximum
    # clock) when the sampled SM clock stayed within 10 % of the maximum (a 16 ms timed region does), else SUSTAINED.  Both
    # fractions are printed.  FLOPs are the dense 36-tap convention of SURVEY 8d; the kernel executes 33 taps (the four centre taps
    # are pre-summed), i.e. 33/36 of the credited FLOPs.
    sm_mhz, sm_max = (clocks or {}).get("sm_mhz"), (clocks or {}).get("sm_max_mhz")
    at_max_clock = bool(sm_mhz and sm_max and sm_mhz >= 0.9 * sm_max)
    peak = peaks["bf16_tflops"] if at_max_clock else peaks["bf16_tflops_sustained"]
    kernels = {k: {"ms_per_launch": round(v[0] / v[1], 4), "launches_per_step": v[1] / args.steps} for k, v in prof.items()}
    for k in gemm_names:
        if k in kernels:
            kernels[k]["tflops"] = round(flops_per_launch / (kernels[k]["ms_per_launch"] * 1e-3) / 1e12, 1)
    k2_ms = prof["upsample_ce_main"][0] / prof["upsample_ce_main"][1] if "upsample_ce_main" in prof else None
    k2_bytes = 16 * n * H * W + 12 * n * C * h * w                  # SURVEY 8d: int64 labels fwd + bwd, low-res logits r / r / w
    roofline = {"kernel": "gemm_bf16_kernel (tcgen05; head fwd / dgrad / wgrad launches)", "bound": "tensor",
                "achieved": round(achieved, 1), "peak": peak, "unit": "TFLOP/s", "frac": round(achieved / peak, 4),
                "traffic": load_traffic("head_fwd_gemm") if args.workload == "train_b8_512x1024" else None,
                "peak_source": peaks["source"] + (", burst bf16 (SM clock at max during the timed region)" if at_max_clock else ", sustained bf16"),
                "frac_of_burst": round(achieved / peaks["bf16_tflops"], 4), "frac_of_sustained": round(achieved / peaks["bf16_tflops_sustained"], 4),
                "sm_mhz_during_timed_region": sm_mhz,
                "algorithmic_flops_per_launch": flops_per_launch, "executed_flops_per_launch": flops_per_launch * 33 / 36,
                "flops_convention": "credited: dense 36 taps (SURVEY 8d); executed: 33 taps (centre taps pre-summed)",
                "head_fwd_bwd_incl_helpers_tflops": round(3 * flops_per_launch / (sum(prof[k][0] for k in prof if k.startswith(("head_", "pack_", "grad_im2col", "wgrad_reduce"))) / args.steps * 1e-3) / 1e12, 1),
                "k2_upsample_ce_us": None if k2_ms is None else round(k2_ms * 1e3, 2),
                "k2_hbm_frac": None if k2_ms is None else round(k2_bytes / (k2_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                "kernels": kernels}

    # ---- the SAME step written as the reference's unmodified trainer lines (aspp_trainer.py:88-92): module call, the caller's
    #      own nn.CrossEntropyLoss, backward -- reaches the fused kernels through lazy.LazyLogits
    criterion = torch.nn.CrossEntropyLoss(ignore_index=255)

    def unmodified_trainer_step():
        xg = x.detach().requires_grad_(True)
        for p in head_params:
            p.grad = None
        size = labels.shape[-2:]
        output = head(xg, size)
        loss = criterion(output, labels)
        loss.backward()
        return loss

    # (under a multi-rank process group the modules default to materialised outputs, because the reference wraps them in
    #  DistributedDataParallel(find_unused_parameters=True), which inspects the output for tensors.  This leg runs the module
    #  un-wrapped and without gradient synchronisation, so it opts in explicitly.)
    head.lazy = True
    try:
        ms_unmod, _ = timed(unmodified_trainer_step, args.steps, args.warmup)
    finally:
        head.lazy = None
    roofline["unmodified_trainer_lines_ms_per_step"] = round(ms_unmod / args.steps, 4)
    roofline["forward_loss_ms_per_step"] = round(ms_per_step, 4)

    # ---- the same step captured once in a CUDA graph and replayed (no Python / launch overhead at all): equal to the eager
    #      number when the step is GPU-bound.  Single-rank only (the bucket's NCCL all-reduce stays out of graphs here).
    graph_ms = None
    if world == 1:
        try:
            for p in head.parameters():
                p.grad = None
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                train_step()
            ms_g, _ = timed(g.replay, args.steps, args.warmup)
            graph_ms = round(ms_g / args.steps, 4)
            del g
        except Exception as e:                                   # never let the extra leg break the headline line
            log("graph replay leg skipped:", repr(e))
            torch.cuda.synchronize()

    # ---- seam format (SURVEY 8f rank 2): bf16 channels_last features in, bf16 channels_last feature gradient out.
    #      Reported beside the headline, which stays on the reference's fp32 NCHW contract.
    xs = x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
    ms_seam, _ = timed(lambda: train_step(xs, labels), args.steps, args.warmup)
    seam = {"value": round(world * label_px / (ms_seam / args.steps * 1e-3) / 1e6, 2), "unit": "Mpx/s",
            "ms_per_step": round(ms_seam / args.steps, 4),
            "input": "bf16 channels_last features (zero-copy GEMM operand), bf16 channels_last feature gradient from the dgrad epilogue"}
    del xs

    # ---- end to end through the public API with HOST buffers (pinned), H2D + loss D2H inside the timed region
    xh = x.cpu().pin_memory()
    lh = labels.cpu().pin_memory()
    e2e_step = HostPipelinedStep(dev, (xh, lh), lambda xd, ld: train_step(xd, ld)[0])
    e2e_steps = max(2, min(args.steps, 10))
    ms_e2e, _ = timed(e2e_step, e2e_steps, 4)
    e2e = {"value": round(world * label_px / (ms_e2e / e2e_steps * 1e-3) / 1e6, 2), "unit": "Mpx/s",
           "h2d_bytes_per_step": xh.numel() * 4 + lh.numel() * 8, "d2h_bytes_per_step": 4,
           "note": "public API from pinned host buffers; every step's H2D and loss D2H are inside the timed region, the H2D of "
                   "step k+1 (copy stream, double-buffered) overlaps the compute of step k"}
    del xh, lh, e2e_step
    # the same from host buffers in the seam formats of SURVEY 8f rank 2: bf16 channels_last features + uint8 labels (2.1x fewer bytes)
    xh = x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last).cpu().pin_memory()
    lh = labels.to(torch.uint8).cpu().pin_memory()
    e2e_seam_step = HostPipelinedStep(dev, (xh, lh), lambda xd, ld: train_step(xd, ld)[0])
    ms_e2e_s, _ = timed(e2e_seam_step, e2e_steps, 4)
    e2e["seam_bf16_uint8_value"] = round(world * label_px / (ms_e2e_s / e2e_steps * 1e-3) / 1e6, 2)
    e2e["seam_h2d_bytes_per_step"] = xh.numel() * 2 + lh.numel()
    del xh, lh, e2e_seam_step

    # ---- eval img/s @1024x2048 (the tester loop of aspp_tester.py:57-72 after the backbone): per frame the head forward on
    #      1 x 2048 x 128 x 256 features; upsample + argmax + confusion matrix (K4) over 8 queued frames per launch
    #      (utility.BatchedEvaluator -- a single 1024 x 2048 frame cannot fill 148 SMs with tall tiles).
    en, ecin, eh, ew, eH, eW, eC = synth.WORKLOADS["eval_1024x2048"]
    ehead = synth.scale_head_for_unit_logits(b200.ASPP_Classifier_V2(ecin, RATES, RATES, eC)).to(dev).eval()
    nf, nl, kf = 4, 8, 8                                 # distinct feature maps (4 x 268 MB > L2) / label maps; frames per K4 launch
    ex = [synth.make_features(1, ecin, eh, ew, seed=99 + rank * 16 + i, device=dev) for i in range(nf)]
    ey = [synth.make_labels(1, eH, eW, eC, seed=199 + rank * 16 + i, device=dev) for i in range(nl)]
    ey8 = [t.to(torch.uint8) for t in ey]
    esteps = max(args.steps * 4, 24) // kf * kf
    k4_bytes = 8 * eH * eW + 4 * eC * eh * ew + 8 * eC * eC
    k4_bytes_u8 = eH * eW + 4 * eC * eh * ew + 8 * eC * eC

    def eval_leg(features, labels, frames_per_launch):
        ev = b200.BatchedEvaluator(ehead, eC, frames=frames_per_launch)
        k = [0]

        def step():
            i = k[0]
            k[0] += 1
            ev.step(features[i % nf], labels[i % nl])

        ms_leg, _ = timed(step, esteps, (args.warmup + kf - 1) // kf * kf)
        _lib.profile_enable(True)
        for _ in range(2 * kf):
            step()
        torch.cuda.synchronize()
        prof_leg = _lib.profile_read()
        _lib.profile_enable(False)
        k4 = prof_leg["eval_argmax_confusion"]
        return ms_leg, ev.finish(), prof_leg, k4[0] / (2 * kf)             # K4 ms per FRAME

    ems, cm, eprof, k4_ms = eval_leg(ex, ey, kf)
    if world > 1:
        D.allreduce_confusion_(cm)
    ems_u8, _, _, k4_ms_u8 = eval_leg(ex, ey8, kf)
    ems_1, _, _, k4_ms_1 = eval_leg(ex, ey, 1)                             # one K4 launch per frame (the round-1 loop)
    exs = [t.to(torch.bfloat16).contiguous(memory_format=torch.channels_last) for t in ex]
    ems_seam, _, _, _ = eval_leg(exs, ey8, kf)                             # seam formats: bf16 channels_last features + uint8 labels
    del exs
    exh = ex[0].cpu().pin_memory()
    eyh = ey[0].cpu().pin_memory()

    def eval_from_device(xd, yd):
        with torch.no_grad():
            lg = ehead.logits(xd)
        c, _ = b200.segmentation_eval_step(lg, yd)
        return c

    eval_e2e_step = HostPipelinedStep(dev, (exh, eyh), eval_from_device)
    ems_e2e, _ = timed(eval_e2e_step, 10, 1)
    eval_obj = {"metric": "eval_img_per_s_1024x2048", "value": round(world * esteps / (ems * 1e-3), 1), "unit": "img/s",
                "ms_per_frame": round(ems / esteps, 4), "frames": esteps * world, "frames_per_k4_launch": kf,
                "confusion_total": int(cm.sum().item()),
                "e2e": {"value": round(world * 10 / (ems_e2e * 1e-3), 1), "unit": "img/s",
                        "h2d_bytes_per_step": exh.numel() * 4 + eyh.numel() * 8, "d2h_bytes_per_step": 8 * eC * eC},
                "roofline": {"kernel": "k4_upsample_argmax_confusion", "bound": "hbm", "achieved": round(k4_bytes / (k4_ms * 1e-3) / 1e9, 1),
                             "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": round(k4_bytes / (k4_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                             "traffic": load_traffic("eval_argmax_confusion"), "algorithmic_bytes_per_frame": k4_bytes,
                             "us_per_frame": round(k4_ms * 1e3, 2),
                             "uint8_labels": {"us_per_frame": round(k4_ms_u8 * 1e3, 2), "algorithmic_bytes_per_frame": k4_bytes_u8,
                                              "frac": round(k4_bytes_u8 / (k4_ms_u8 * 1e-3) / 1e9 / peaks["hbm_gbs"], 4)},
                             "one_frame_per_launch_us": round(k4_ms_1 * 1e3, 2)},
                "kernels": {k: round(v[0] / v[1], 4) for k, v in eprof.items()},
                "uint8_labels": {"value": round(world * esteps / (ems_u8 * 1e-3), 1), "unit": "img/s"},
                "one_k4_launch_per_frame": {"value": round(world * esteps / (ems_1 * 1e-3), 1), "unit": "img/s"},
                "seam_bf16_nhwc_uint8": {"value": round(world * esteps / (ems_seam * 1e-3), 1), "unit": "img/s",
                                         "ms_per_frame": round(ems_seam / esteps, 4)}}
    roofline.update({"eval_img_per_s": eval_obj["value"], "eval_ms_per_frame": eval_obj["ms_per_frame"],
                     "k4_us_per_frame": round(k4_ms * 1e3, 2), "k4_hbm_frac": eval_obj["roofline"]["frac"],
                     "k4_uint8_us_per_frame": round(k4_ms_u8 * 1e3, 2), "eval_uint8_img_per_s": eval_obj["uint8_labels"]["value"]})
    del ex, ey, ey8

    # ---- the other loss kernels of the scope table (SURVEY 8a5-a7) at the adversarial config: N=4, 2C=38, 512x1024
    from rnd_semantic_segmentation_b200 import ops as bops
    an, _, ah, aw, aH, aW, aC = synth.WORKLOADS["deeplabv2_r101_adv"]
    gen = torch.Generator(device=dev).manual_seed(4321 + rank)
    sets3 = []
    for _ in range(2):                                    # 2 x (319 + 319 MB) > L2
        pred = torch.randn(an, 2 * aC, aH, aW, device=dev, generator=gen)
        soft = torch.softmax(torch.randn(an, 2 * aC, aH, aW, device=dev, generator=gen), 1)
        sets3.append((pred, soft))
    i3 = [0]

    def k3_step():
        pred, soft = sets3[i3[0] & 1]
        i3[0] += 1
        pr = pred.requires_grad_(True)
        pr.grad = None
        bops.soft_label_cross_entropy(pr, soft).backward()

    k3_ms, _ = timed(k3_step, 6, 3)
    k3_bytes = 20 * 2 * aC * an * aH * aW
    del sets3
    d_lr = torch.randn(an, 2 * aC, ah, aw, device=dev, generator=gen)
    s_lr = torch.randn(an, aC, ah, aw, device=dev, generator=gen)

    def k5_step():
        dl = d_lr.requires_grad_(True)
        dl.grad = None
        bops.fada_soft_label_loss(dl, s_lr, (aH, aW), slot=0).backward()

    k5_ms, _ = timed(k5_step, 10, 3)
    aux = {"k3_soft_label_ce_fwd_bwd": {"ms": round(k3_ms / 6, 4), "algorithmic_bytes": k3_bytes, "bound": "hbm",
                                        "achieved_gbs": round(k3_bytes / (k3_ms / 6 * 1e-3) / 1e9, 1),
                                        "frac": round(k3_bytes / (k3_ms / 6 * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                                        "shape": [an, 2 * aC, aH, aW]},
           "k5_fused_fada_loss_tail_fwd_bwd": {"ms": round(k5_ms / 10, 4), "replaces_bytes_of_materialised_path": k3_bytes + 16 * 2 * aC * an * aH * aW,
                                               "shape_lowres": [an, 2 * aC, ah, aw], "size": [aH, aW],
                                               "note": "compute-bound: only low-resolution tensors are read"}}

    del d_lr, s_lr
    aux.update(run_tta_and_optim(b200, _lib, dev, rank, peaks))
    adv = run_adv_step(b200, _lib, synth, dev, rank, world, peaks, args)
    cfgs = run_baseline_configs(b200, _lib, synth, dev, rank, peaks, args) if world == 1 else {}
    dp_check = run_dp_check(b200, D, synth, dev, rank, world, head, bucket, x, labels) if world > 1 else "n/a (single rank)"

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = run_cpu_reference(args.workload, steps=2, warmup=1)["cpu_baseline"]
        eval_obj["cpu_baseline"] = run_cpu_eval_reference()
        adv["cpu_baseline"] = run_cpu_adv_reference()

    if rank == 0:
        # scalars the driver keeps (it drops nested objects outside the contract keys): everything a reader needs to judge the
        # other legs rides in `roofline`
        roofline.update({"dp_check": dp_check, "adv_step_Mpx_per_s": adv["value"], "adv_step_ms": adv["ms_per_step"],
                         "adv_conv_frac_of_sustained": adv["roofline"]["frac"], "seam_bf16_nhwc_ms_per_step": seam["ms_per_step"]})
        for key, c in cfgs.items():
            roofline.update({f"{key}_Mpx_per_s": c["Mpx_per_s"], f"{key}_ms_per_step": c["ms_per_step"],
                             f"{key}_graph_replay_ms_per_step": c["graph_replay_ms_per_step"],
                             f"{key}_gemm_frac_of_burst": c["gemm_frac_of_burst"], f"{key}_step_hbm_frac": c["step_hbm_frac"]})
        line = {"metric": "aspp_ce_train_Mpx_per_s", "value": round(value, 2), "unit": "Mpx/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "config": workload_config(args.workload, world),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches_timed), "roofline": roofline, "eval": eval_obj,
                "seam_bf16_nhwc": seam, "aux_kernels": aux, "adv_step": adv, "baseline_configs": cfgs, "dp_check": dp_check,
                "cuda_graph_replay_ms_per_step": graph_ms}
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        emit(line)
    if dist.is_initialized():
        dist.destroy_process_group()


def run_baseline_configs(b200, _lib, synth, dev, rank, peaks, args):
    """BASELINE.json's literal train configs on one GPU (each is a parity-test case at full size in tests/test_gpu_round2.py; here
    their throughput): cfg1 deeplabv2_r101_src (2 x 2048 x 65 x 129, C = 19), cfg2 deeplabv2_r101_src_kvasir (16 x 2048 x 44 x 44,
    C = 2 -- arithmetic intensity 72 FLOP/B, so judged against HBM, SURVEY 8d) and cfg4 deeplabv2_r101_tgt_self_distill (1 image
    per GPU).  Eager public-API step and the same step replayed from a CUDA graph (what the ~10 stream launches cost on the host:
    the small configs are host-bound in eager mode)."""
    out = {}
    for key, name, p_ign in (("cfg1", "deeplabv2_r101_src", 0.10), ("cfg2", "deeplabv2_r101_src_kvasir", 0.05),
                             ("cfg4", "deeplabv2_r101_tgt_self_distill", 0.10)):
        n, cin, h, w, H, W, C = synth.WORKLOADS[name]
        torch.manual_seed(1234)
        head = b200.ASPP_Classifier_V2(cin, RATES, RATES, C).to(dev)
        xs = [synth.make_features(n, cin, h, w, seed=31 + rank + 7 * i, device=dev) for i in range(2)]    # 2 x >= 137 MB: > L2 for cfg1 / cfg2
        labels = synth.make_labels(n, H, W, C, p_ignore=p_ign, seed=32 + rank, device=dev)
        k = [0]
        params = list(head.parameters())

        def step(x_in=None):
            x_in = xs[k[0] & 1] if x_in is None else x_in
            k[0] += 1
            xg = x_in.detach().requires_grad_(True)
            for p in params:
                p.grad = None
            loss, _ = head.forward_loss(xg, labels)
            loss.backward()
            return loss

        # (two alternating inputs = two address sets: each is seen once, then captured by the one-call entries' graph cache,
        #  so six warm-up steps put the timed region in the steady state a training loop runs in)
        ms, _ = timed(step, args.steps, max(args.warmup, 6))
        _lib.profile_enable(True)
        for _ in range(4):
            step()
        torch.cuda.synchronize()
        prof = _lib.profile_read()
        _lib.profile_enable(False)
        graph_ms = None
        try:
            for p in head.parameters():
                p.grad = None
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                step(xs[0])
            ms_g, _ = timed(g.replay, args.steps, args.warmup)
            graph_ms = ms_g / args.steps
            del g
        except Exception as e:
            log(f"{key}: graph replay leg skipped:", repr(e))
            torch.cuda.synchronize()
        flops = 2.0 * 36 * cin * C * n * h * w
        gms = sum(prof[q][0] for q in ("head_fwd_gemm", "head_dgrad_gemm", "head_wgrad_gemm") if q in prof) / 4
        gemm_tf = 3 * flops / (gms * 1e-3) / 1e12 if gms > 0 else 0.0
        step_bytes = 8.0 * n * cin * h * w + 16.0 * n * H * W            # fp32 features read + feature gradient written, int64 labels twice
        best_ms = min(ms / args.steps, graph_ms) if graph_ms else ms / args.steps
        out[key] = {"workload": name, "Mpx_per_s": round(n * H * W / (ms / args.steps * 1e-3) / 1e6, 1), "ms_per_step": round(ms / args.steps, 4),
                    "graph_replay_ms_per_step": None if graph_ms is None else round(graph_ms, 4),
                    "gemm_tflops": round(gemm_tf, 1), "gemm_frac_of_burst": round(gemm_tf / peaks["bf16_tflops"], 4),
                    "step_hbm_gbs": round(step_bytes / (best_ms * 1e-3) / 1e9, 1), "step_hbm_frac": round(step_bytes / (best_ms * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                    "bound": "hbm" if C == 2 else "tensor"}
        del head, xs, labels
    return out


def run_dp_check(b200, D, synth, dev, rank, world, head, bucket, x, labels):
    """Data-parallel correctness inside the driver-run path (SURVEY 4, "distributed" tier), after the timed region:
    (1) the gradients the overlapped bucket leaves in .grad are bit-identical on every rank and equal the mean of the per-rank
    gradients computed WITHOUT the bucket (plain autograd path); (2) the all-reduced int64 confusion matrix equals the matrix one
    rank computes over the union of all ranks' frames.  Returns "ok" or raises."""
    import torch.distributed as dist
    for p in head.parameters():
        p.grad = None
    xg = x.detach().requires_grad_(True)
    loss, _ = head.forward_loss(xg, labels, grad_bucket=bucket)
    loss.backward()
    bucket.wait()
    reduced = torch.cat([p.grad.reshape(-1) for p in head.parameters()]).clone()
    for p in head.parameters():
        p.grad = None
    xg = x.detach().requires_grad_(True)
    loss, _ = head.forward_loss(xg, labels)
    loss.backward()
    local = torch.cat([p.grad.reshape(-1) for p in head.parameters()]).clone()
    for p in head.parameters():
        p.grad = None
    all_reduced = [torch.empty_like(reduced) for _ in range(world)]
    all_local = [torch.empty_like(local) for _ in range(world)]
    dist.all_gather(all_reduced, reduced)
    dist.all_gather(all_local, local)
    for r in range(1, world):
        if not torch.equal(all_reduced[r], all_reduced[0]):
            raise RuntimeError(f"dp_check: bucket gradients differ between rank 0 and rank {r}")
    mean = torch.stack([t.double() for t in all_local]).mean(0)
    err = ((reduced.double() - mean).abs().max() / mean.abs().max()).item()
    if not err <= 1e-6:
        raise RuntimeError(f"dp_check: all-reduced gradients != mean of per-rank gradients (rel err {err:.3e})")
    # eval: frames rank::world of a common list; every rank can regenerate any frame (seeded CUDA generators)
    C, frames_total = 19, 2 * world

    def frame(i):
        g = torch.Generator(device=dev).manual_seed(9000 + i)
        lg = torch.randn(1, C, 64, 128, device=dev, generator=g)
        y = torch.randint(0, C, (1, 512, 1024), device=dev, generator=g)
        y[:, : 64 * (i % 3)] = 255
        return lg, y

    cm = torch.zeros(C, C, dtype=torch.int64, device=dev)
    for i in D.shard_indices(frames_total, rank, world):
        lg, y = frame(i)
        b200.segmentation_eval_step(lg, y, cm=cm)
    D.allreduce_confusion_(cm)
    union = torch.zeros_like(cm)
    for i in range(frames_total):
        lg, y = frame(i)
        b200.segmentation_eval_step(lg, y, cm=union)
    if not torch.equal(cm, union):
        raise RuntimeError("dp_check: all-reduced confusion matrix != single-rank matrix over the union of the shards")
    return "ok"


def run_tta_and_optim(b200, _lib, dev, rank, peaks):
    """SURVEY 8f ranks 3 and 4: K7 (flip test-time augmentation fused with argmax + confusion matrix, one 1024x2048 frame per
    launch, members = head logits of the frame and of its mirror image at 128x256) and K8 (one-launch optimizer steps of the head's
    SGD and the discriminator's Adam parameter groups; device time from back-to-back raw C-ABI calls, host-inclusive time through
    the torch.optim-compatible classes)."""
    import ctypes
    gen = torch.Generator(device=dev).manual_seed(777 + rank)
    C, H, W, h, w = 19, 1024, 2048, 128, 256
    frames = [([torch.randn(1, C, h, w, device=dev, generator=gen) for _ in range(2)],
               torch.randint(0, C, (1, H, W), device=dev, generator=gen)) for _ in range(8)]       # 8 x 16.8 MB of labels > L2
    cm = torch.zeros(C, C, dtype=torch.int64, device=dev)
    k = [0]

    def k7_step():
        members, labels = frames[k[0] & 7]
        k[0] += 1
        _lib.tta_argmax_confusion(members, [False, True], (H, W), labels=labels, divisors=(2,), cm=cm)

    k7_ms, _ = timed(k7_step, 16, 4)
    k7_bytes = 8 * H * W + 2 * 4 * C * h * w
    out = {"k7_flip_tta_argmax_confusion": {"ms_per_frame": round(k7_ms / 16, 4), "frames_per_s": round(16 / (k7_ms * 1e-3), 1),
                                            "algorithmic_bytes": k7_bytes, "members": [[C, h, w]] * 2, "size": [H, W],
                                            "replaces_bytes_of_materialised_path": 2 * 4 * C * H * W * 6,
                                            "note": "compute-bound (2 x 19 expf + correctly rounded divisions per label pixel); "
                                                    "bit-exact against the torch CUDA op sequence of utility.py:179-191"}}
    del frames
    lib = _lib.load()
    for name, shapes, kind in (("k8_head_sgd_step", [(19, 2048, 3, 3), (19,)] * 4, "sgd"),
                               ("k8_discriminator_adam_step", [(256, 2048, 3, 3), (256,), (128, 256, 3, 3), (128,), (19, 128, 3, 3), (19,),
                                                               (19, 128, 3, 3), (19,)], "adam")):
        ps = [torch.nn.Parameter(torch.randn(s, device=dev, generator=gen) * 0.01) for s in shapes]
        for p_ in ps:
            p_.grad = torch.randn(p_.shape, device=dev, generator=gen) * 0.01
        opt = b200.FusedSGD(ps, lr=2.5e-3, momentum=0.9, weight_decay=5e-4) if kind == "sgd" else b200.FusedAdam(ps, lr=1e-4, betas=(0.9, 0.99))
        api_ms, _ = timed(opt.step, 50, 5)
        n = len(ps)
        arr = lambda ts: (ctypes.c_void_p * n)(*[t.data_ptr() for t in ts])  # noqa: E731
        numels = (ctypes.c_int64 * n)(*[p_.numel() for p_ in ps])
        pa, ga = arr(ps), arr([p_.grad for p_ in ps])
        stream = torch.cuda.current_stream().cuda_stream
        if kind == "sgd":
            ba = arr([opt.state[p_]["momentum_buffer"] for p_ in ps])
            raw = lambda: lib.b200seg_sgd_step(n, pa, ga, ba, numels, 2.5e-3, 0.9, 0.0, 5e-4, 0, 0, 1.0, stream)  # noqa: E731
        else:
            ma, va = arr([opt.state[p_]["exp_avg"] for p_ in ps]), arr([opt.state[p_]["exp_avg_sq"] for p_ in ps])
            raw = lambda: lib.b200seg_adam_step(n, pa, ga, ma, va, numels, 1e-4, 0.9, 0.99, 1e-8, 0.0, 100, 1.0, stream)  # noqa: E731
        dev_ms, _ = timed(raw, 50, 5)
        nbytes = sum(p_.numel() for p_ in ps) * (20 if kind == "sgd" else 28)
        out[name] = {"us_device": round(dev_ms / 50 * 1e3, 2), "us_through_optimizer_api": round(api_ms / 50 * 1e3, 2),
                     "elements": sum(p_.numel() for p_ in ps), "algorithmic_bytes": nbytes, "bound": "hbm",
                     "achieved_gbs": round(nbytes / (dev_ms / 50 * 1e-3) / 1e9, 1),
                     "frac": round(nbytes / (dev_ms / 50 * 1e-3) / 1e9 / peaks["hbm_gbs"], 4),
                     "note": "parameter group of the size of L2 or smaller, re-touched every step: largely L2-resident (a fraction above 1 means L2 hits), launch-bound; one launch per group"}
    return out


def run_adv_step(b200, _lib, synth, dev, rank, world, peaks, args):
    """BASELINE.json configs[2] (deeplabv2_r101_adv): everything after the backbone of one FADA iteration, aspp_fada.py:91-125 --
    head fwd + CE fwd/bwd on the source batch, head fwd on the target batch, and three PixelDiscriminator passes with their
    soft-label losses (adversarial: gradient to the target features; discriminator update: weight gradients on detached
    features).  Optimizer steps excluded.  The discriminator convolutions run on the tcgen05 implicit-GEMM kernel (K6)."""
    an, cin, ah, aw, aH, aW, aC = synth.WORKLOADS["deeplabv2_r101_adv"]
    torch.manual_seed(4321)
    head = b200.ASPP_Classifier_V2(cin, RATES, RATES, aC).to(dev)
    model_D = b200.PixelDiscriminator(cin, 256, num_classes=aC).to(dev)
    src = synth.make_features(an, cin, ah, aw, seed=555 + rank, device=dev)
    tgt = synth.make_features(an, cin, ah, aw, seed=777 + rank, device=dev)
    lab = synth.make_labels(an, aH, aW, aC, seed=555 + rank, device=dev)
    size = (aH, aW)
    b200.set_feature_pack_cache(2)

    freeze = [False]
    with_opt = [False]
    opt_cls = b200.FusedSGD(head.parameters(), lr=2.5e-3, momentum=0.9, weight_decay=5e-4)     # aspp_trainer.py:26
    opt_d = b200.FusedAdam(model_D.parameters(), lr=1e-4, betas=(0.9, 0.99))                   # fada_adapter.py:24
    # N > 1: DDP semantics for both modules (train_adv.py shards the data but never synchronises, SURVEY 2a).  Head gradients:
    # flat bucket, mean all-reduce underneath the head's data-gradient GEMM.  Discriminator gradients (20.2 MB): flat bucket the
    # two discriminator backward passes accumulate into, mean all-reduce started after the second one on the bucket's stream and
    # joined only before the discriminator is used again -- i.e. it overlaps the NEXT iteration's source-domain head step.
    from rnd_semantic_segmentation_b200 import distributed as D
    hb = D.HeadGradBucket(head) if world > 1 else None
    db = D.OverlappedGradBucket(model_D.parameters()) if world > 1 else None

    def adv_step():
        b200.clear_feature_pack_cache()                       # new features every iteration: 2 conversions per step, not 0
        if hb is not None:
            hb.wait()                                         # (last iteration's head all-reduce / optimizer step)
        for p in head.parameters():
            p.grad = None
        if db is None:
            for p in model_D.parameters():
                p.grad = None
        # (both modules are in training mode: their bf16 weight packs are rebuilt on every call)
        src_fea = src.detach().requires_grad_(True)
        tgt_fea = tgt.detach().requires_grad_(True)
        loss_seg, src_lr = head.forward_loss(src_fea, lab, temperature=1.8, grad_bucket=hb)   # aspp_fada.py:91-96
        loss_seg.backward()
        with torch.no_grad():
            tgt_lr = head.logits(tgt_fea)                                                # :101-104 (soft labels are detached)
        if db is not None:
            db.wait()                                         # last iteration's discriminator all-reduce (+ Adam step) is done
        if freeze[0]:                                         # variant: D's own gradients of this pass are discarded at :117 anyway
            for p in model_D.parameters():
                p.requires_grad_(False)
        loss_adv = 0.001 * model_D.forward_soft_loss(tgt_fea, tgt_lr, size, slot=0)      # :110-112
        loss_adv.backward()
        if with_opt[0]:
            if hb is not None:
                hb.step(opt_cls)                                                         # :115 behind the head all-reduce
            else:
                opt_cls.step()                                                           # :115 (K8)
        for p in model_D.parameters():                                                   # optimizer_D.zero_grad(), :117
            p.requires_grad_(True)
        if db is not None:
            db.zero_grads_()
        else:
            for p in model_D.parameters():
                p.grad = None
        loss_d_src = 0.5 * model_D.forward_soft_loss(src_fea.detach(), src_lr, size, slot=0)   # :119-121
        loss_d_src.backward()
        loss_d_tgt = 0.5 * model_D.forward_soft_loss(tgt_fea.detach(), tgt_lr, size, slot=1)   # :123-125
        loss_d_tgt.backward()
        if db is not None:
            db.begin_allreduce_()
            if with_opt[0]:
                db.step(opt_d)                                                           # :127 behind the all-reduce
        elif with_opt[0]:
            opt_d.step()                                                                 # :127 (K8)
        return loss_seg, loss_adv, loss_d_src, loss_d_tgt

    def adv_step_sync():                                      # the timed unit: the iteration AND the collectives it started
        out = adv_step()
        return out

    l0 = _lib.launch_count()
    ms, _ = timed(adv_step, args.steps, args.warmup)
    if db is not None:
        db.wait()
    if hb is not None:
        hb.wait()
    launches = (_lib.launch_count() - l0) * args.steps // (args.steps + args.warmup)
    ms_step = ms / args.steps
    _lib.profile_enable(True)
    for _ in range(4):
        adv_step()
    torch.cuda.synchronize()
    prof = _lib.profile_read()
    _lib.profile_enable(False)
    freeze[0] = True
    ms_frozen, _ = timed(adv_step, args.steps, args.warmup)
    freeze[0] = False
    with_opt[0] = True                                       # the same iteration with the head's SGD and the discriminator's Adam step
    ms_opt, _ = timed(adv_step, args.steps, args.warmup)
    with_opt[0] = False
    # the whole iteration (~100 launches) captured once in a CUDA graph and replayed: what the launch gaps cost
    graph_ms = None
    try:
        if world > 1:
            raise RuntimeError("single-rank leg (the NCCL collectives stay out of the graph)")
        for p in list(head.parameters()) + list(model_D.parameters()):
            p.grad = None
        b200.clear_feature_pack_cache()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            adv_step()
        b200.clear_feature_pack_cache()                      # drop the references into the graph's memory pool
        ms_g, _ = timed(g.replay, args.steps, args.warmup)
        graph_ms = round(ms_g / args.steps, 4)
        del g
    except Exception as e:
        log("adv graph replay leg skipped:", repr(e))
        torch.cuda.synchronize()
    b200.set_feature_pack_cache(0)
    P = an * ah * aw
    # algorithmic FLOPs of one discriminator conv-stack pass (true channel counts, dense 3x3 taps)
    f_pass = 2.0 * 9 * P * (cin * 256 + 256 * 128 + 128 * 2 * aC)
    conv_names = ("conv3x3_fwd", "conv3x3_dgrad", "conv3x3_wgrad")
    conv_ms = sum(prof[k][0] for k in conv_names if k in prof) / 4
    # per step: 3 forward passes, 3 weight-gradient passes, 3 data-gradient passes of layers 3/2 and one of layer 1
    f_step = f_pass * 6 + 2.0 * 9 * P * (3 * (256 * 128 + 128 * 2 * aC) + cin * 256)
    tf = f_step / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    return {"metric": "fada_adv_step_Mpx_per_s", "value": round(world * 2 * an * aH * aW / (ms_step * 1e-3) / 1e6, 2), "unit": "Mpx/s",
            "ms_per_step": round(ms_step, 4), "gpu_launches": int(launches),
            "config": {"workload": "deeplabv2_r101_adv", "features_per_domain": [an, cin, ah, aw], "labels": [an, aH, aW],
                       "num_classes": aC, "discriminator": "PixelDiscriminator(2048, ndf=256) -> 2 x 19",
                       "step": "aspp_fada.py:91-125 after the backbone, optimizer steps excluded; source + target label pixels counted"
                               + ("; mean all-reduce of the head gradients (5.6 MB, under the head dgrad GEMM) and of the discriminator"
                                  " gradients (20.2 MB, overlapping the next iteration's head step) inside the timed region" if world > 1 else "")},
            "roofline": {"kernel": "conv_gemm_kernel (tcgen05 implicit GEMM; discriminator fwd / dgrad / wgrad launches)", "bound": "tensor",
                         "achieved": round(tf, 1), "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                         "frac": round(tf / peaks["bf16_tflops_sustained"], 4), "traffic": load_traffic("conv3x3_fwd"),
                         "algorithmic_flops_per_step": f_step, "conv_ms_per_step": round(conv_ms, 4)},
            "cuda_graph_replay_ms_per_step": graph_ms,
            "variants": {"with_optimizer_steps": {
                "ms_per_step": round(ms_opt / args.steps, 4),
                "note": "plus optimizer_cls.step() (aspp_fada.py:115, FusedSGD) and optimizer_D.step() (:127, FusedAdam): one K8 launch each"},
                         "discriminator_frozen_in_adversarial_pass": {
                "ms_per_step": round(ms_frozen / args.steps, 4),
                "note": "model_D parameters set requires_grad=False around aspp_fada.py:110-112: the weight gradients that pass "
                        "would compute are zeroed at :117 before anyone reads them, so the parameter updates are identical"}},
            "kernels": {k: {"ms_per_step": round(v[0] / 4, 4), "launches_per_step": v[1] / 4} for k, v in prof.items()}}


# ----------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path (oracle port), all host threads
# ----------------------------------------------------------------------------------------------------
def run_cpu_reference(workload, steps, warmup):
    from oracle import torch_oracle as to
    from rnd_semantic_segmentation_b200 import synth
    n, cin, h, w, H, W, C = synth.WORKLOADS[workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(1234)
    head = to.AsppHeadOracle(cin, RATES, RATES, C)
    ns = 1                                                 # bounded sample: one image of the step's batch per CPU step
    x = synth.make_features(ns, cin, h, w, seed=1234)
    labels = synth.make_labels(ns, H, W, C, seed=1234)
    for _ in range(warmup):
        to.train_step_src(head, x, labels)
    t0 = time.perf_counter()
    for _ in range(steps):
        to.train_step_src(head, x, labels)
    dt = (time.perf_counter() - t0) / steps
    value = ns * H * W / dt / 1e6
    sample = f"{ns} of the {n} images of workload {workload} per step ({ns}x{cin}x{h}x{w} features, {ns}x{H}x{W} labels), torch {torch.__version__} CPU fp32"
    return {"value": value, "ms_per_step": dt * 1e3,
            "cpu_baseline": {"value": round(value, 4), "unit": "Mpx/s", "cores": cores, "kind": "port", "sample": sample}}


def run_cpu_eval_reference():
    """SURVEY 8d (iii): the reference's eval frame on the host cores -- head forward, interpolate + softmax + max(1)[1]
    (utility.py:183-186, aspp_tester.py:63), then the confusion matrix: the reference's literal per-pixel Python loop
    (utility.py:347-359) timed on a 1/64 crop and extrapolated, and the vectorised bincount equivalent as the fair CPU row."""
    from oracle import torch_oracle as to
    from rnd_semantic_segmentation_b200 import synth
    n, cin, h, w, H, W, C = synth.WORKLOADS["eval_1024x2048"]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(99)
    head = synth.scale_head_for_unit_logits(to.AsppHeadOracle(cin, RATES, RATES, C))
    x = synth.make_features(1, cin, h, w, seed=99)
    y = synth.make_labels(1, H, W, C, seed=199)
    to.eval_frame(head, x, y, C)                                            # warm-up
    t0 = time.perf_counter()
    pred, _, _ = to.eval_frame(head, x, y, C)
    dt = time.perf_counter() - t0
    crop = (slice(None), slice(0, H // 8), slice(0, W // 8))
    t0 = time.perf_counter()
    to.confusion_matrix_loop(C, pred[crop].flatten(), y[crop].flatten())
    dt_loop = (time.perf_counter() - t0) * 64
    return {"value": round(1.0 / dt, 3), "unit": "img/s", "cores": cores, "kind": "port",
            "sample": f"1 frame 1x{cin}x{h}x{w} -> {H}x{W}: head fwd + interpolate/softmax/argmax + bincount confusion matrix + intersectionAndUnion",
            "with_reference_python_loop_confusion_matrix": {"value": round(1.0 / (dt + dt_loop), 4), "unit": "img/s",
                                                            "note": "utility.py:347-359 per-pixel loop timed on a 1/64 crop, x64"}}


def run_cpu_adv_reference():
    """SURVEY 8d (ii): the full aspp_fada.py:91-125 sequence after the backbone (forward AND backward) on the host cores, on a
    bounded sample: 1 source + 1 target image of the 4 + 4 of BASELINE configs[2]."""
    from oracle import torch_oracle as to
    from rnd_semantic_segmentation_b200 import synth
    n, cin, h, w, H, W, C = synth.WORKLOADS["deeplabv2_r101_adv"]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(4321)
    head = to.AsppHeadOracle(cin, RATES, RATES, C)
    model_D = to.PixelDiscriminatorOracle(cin, 256, num_classes=C)
    src = synth.make_features(1, cin, h, w, seed=555)
    tgt = synth.make_features(1, cin, h, w, seed=777)
    lab = synth.make_labels(1, H, W, C, seed=555)
    to.fada_step(head, model_D, src, tgt, lab)                              # warm-up
    t0 = time.perf_counter()
    to.fada_step(head, model_D, src, tgt, lab)
    dt = time.perf_counter() - t0
    return {"value": round(2 * H * W / dt / 1e6, 4), "unit": "Mpx/s", "cores": cores, "kind": "port", "ms_per_step": round(dt * 1e3, 1),
            "sample": f"1 + 1 of the {n} + {n} images of workload deeplabv2_r101_adv per step, torch {torch.__version__} CPU fp32"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from rnd_semantic_segmentation_b200 import synth
    n, cin, h, w, H, W, C = synth.WORKLOADS[args.workload]
    r = run_cpu_reference(args.workload, steps=max(1, args.steps), warmup=max(1, min(args.warmup, 2)))
    line = {"impl": "reference", "metric": "aspp_ce_train_Mpx_per_s", "value": round(r["value"], 4), "unit": "Mpx/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(r["ms_per_step"], 2),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.workload, args.gpus),
            "note": "reference's CPU path (oracle port of classifier.py:26-32 + CrossEntropyLoss + backward) on the host cores; "
                    "each step is a bounded one-image sample of the workload (per-pixel normalised)",
            "cpu_baseline": r["cpu_baseline"],
            "e2e": {"value": round(r["value"], 4), "unit": "Mpx/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


_REAL_STDOUT = None


def _claim_stdout():
    """Everything libraries print (NCCL banners, warnings) goes to stderr; stdout carries exactly one JSON line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20,
                    help="timed steps K of the headline train step and of the unmodified-trainer, graph-replay, seam, adversarial and "
                         "per-config legs.  Side legs derive or fix their own counts: end to end from host buffers "
                         "max(2, min(K, 10)) steps, eval max(4K, 24) frames rounded down to a multiple of 8, the single-kernel legs "
                         "fixed counts")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train_b8_512x1024")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the headline train step returned in its last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()

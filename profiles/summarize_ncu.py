"""Turn an `ncu --set full` report into the small CSV that is committed under profiles/.

    python profiles/summarize_ncu.py gpurun_out/prof_r1d.ncu-rep profiles/r1d_full_summary.csv

Runs here (no GPU needed): `ncu -i <rep> --page raw --csv` and keeps, per profiled launch, the metrics the roofline
statements in DESIGN.md / bench.py rest on.  `traffic_MB` = dram__bytes_read.sum + dram__bytes_write.sum (per launch).
"""
import csv
import os
import io
import subprocess
import sys

KEEP = [
    ("gpu__time_duration.sum", "time"),
    ("dram__bytes_read.sum", "dram_read"),
    ("dram__bytes_write.sum", "dram_write"),
    ("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "dram_pct"),
    ("sm__throughput.avg.pct_of_peak_sustained_elapsed", "sm_pct"),
    ("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "tensor_pipe_pct"),
    ("sm__inst_executed_pipe_tensor.sum", "tensor_inst"),
    ("smsp__issue_active.avg.pct_of_peak_sustained_active", "issue_active_pct"),
    ("sm__warps_active.avg.pct_of_peak_sustained_active", "warps_active_pct"),
    ("smsp__inst_executed.sum", "warp_inst"),
    ("launch__registers_per_thread", "regs"),
    ("launch__grid_size", "grid"),
    ("launch__block_size", "block"),
    ("launch__shared_mem_per_block_dynamic", "dyn_smem"),
    ("lts__t_bytes.sum", "l2_bytes"),
    ("lts__t_sector_hit_rate.pct", "l2_hit_pct"),
    ("l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum", "smem_bank_conflicts"),
    ("sm__cycles_elapsed.max", "sm_cycles"),
]

UNIT_SCALE = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}


def main(rep, out):
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], check=True, capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(raw)))
    head, units, body = rows[0], rows[1], rows[2:]
    col = {name: i for i, name in enumerate(head)}
    kname = col["Kernel Name"]
    fields = ["id", "kernel"] + [short for _, short in KEEP] + ["traffic_MB", "time_us"]
    with open(out, "w", newline="") as f:
        wr = csv.writer(f)
        wr.writerow(fields)
        for r in body:
            vals = {}
            for metric, short in KEEP:
                if metric in col and r[col[metric]] != "":
                    v = float(r[col[metric]].replace(",", ""))
                    v *= UNIT_SCALE.get(units[col[metric]], 1.0)
                    vals[short] = v
            traffic = (vals.get("dram_read", 0.0) + vals.get("dram_write", 0.0)) / 1e6
            name = r[kname].split("(")[0].replace("void ", "")
            wr.writerow([r[col["ID"]], name] + [("%.6g" % vals[s]) if s in vals else "" for _, s in KEEP]
                        + ["%.3f" % traffic, "%.2f" % vals.get("time", float("nan"))])
    print("wrote", out, len(body), "launches")


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])


def write_bench_json(summary_csv, out_json, source):
    """profiles/ncu_summary.json: per-launch DRAM traffic of the kernels bench.py quotes in `roofline.traffic`.
    The capture is profiles/prof_step.py (one train step of the bench workload, then one eval frame), so the first
    launch of each kernel below belongs to the train step unless it is the eval kernel."""
    import json
    keys = [("head_fwd_gemm", "gemm::gemm_bf16_kernel<0, 0, 2>", 0), ("head_dgrad_gemm", "gemm::gemm_bf16_kernel<0, 1, 1>", 0),
            ("head_wgrad_gemm", "gemm::gemm_bf16_kernel<0, 1, 2>", 0), ("pack_features", "nchw_to_nhwc_tile_kernel<false", 0),
            ("head_gather", "head_gather_kernel", 0), ("grad_im2col", "build_gprime", 0),
            ("upsample_ce_main", "k2_upsample_ce_main", 0), ("wgrad_reduce", "wgrad_reduce_kernel", 0),
            ("eval_argmax_confusion", "k4_upsample_argmax_confusion", 0), ("eval_head_fwd_gemm", "gemm::gemm_bf16_kernel<0, 0, 2>", 1),
            ("eval_pack_features", "nchw_to_nhwc_tile_kernel<false", 1), ("eval_head_gather", "head_gather_kernel", 1)]
    rows = list(csv.DictReader(open(summary_csv)))
    out = {"source": source, "kernels": {}}
    for key, pat, nth in keys:
        hits = [r for r in rows if pat in r["kernel"]]
        if len(hits) > nth:
            r = hits[nth]
            out["kernels"][key] = {"kernel": r["kernel"], "dram_bytes_per_launch": int(float(r["traffic_MB"]) * 1e6),
                                   "ncu_time_us": float(r["time_us"]), "registers": int(float(r["regs"])) if r["regs"] else None}
    with open(out_json, "w") as f:
        json.dump(out, f, indent=1)
    print("wrote", out_json)


def merge_disc_json(summary_csv, out_json, source):
    """Add the discriminator conv-stack launches (capture of profiles/prof_disc.py: layer 1 is the first forward launch,
    the last weight-gradient launch and the last data-gradient launch) to profiles/ncu_summary.json."""
    import json
    rows = list(csv.DictReader(open(summary_csv)))
    conv = [r for r in rows if "conv_gemm_kernel<0" in r["kernel"]]
    wg = [r for r in rows if "conv_gemm_kernel<1" in r["kernel"]]
    out = json.load(open(out_json)) if os.path.exists(out_json) else {"kernels": {}}
    out["source_disc"] = source
    for key, r in (("conv3x3_fwd", conv[0]), ("conv3x3_dgrad", conv[-1]), ("conv3x3_wgrad", wg[-1])):
        out["kernels"][key] = {"kernel": r["kernel"], "layer": "2048 -> 256 at 4 x 64 x 128 (layer 1 of the discriminator)",
                               "dram_bytes_per_launch": int(float(r["traffic_MB"]) * 1e6), "ncu_time_us": float(r["time_us"]),
                               "registers": int(float(r["regs"])) if r["regs"] else None,
                               "tensor_pipe_pct_of_active": float(r["tensor_pipe_pct"]) if r["tensor_pipe_pct"] else None}
    with open(out_json, "w") as f:
        json.dump(out, f, indent=1)
    print("merged", out_json)


if __name__ == "__main__" and len(sys.argv) > 4 and sys.argv[4] == "disc":
    merge_disc_json(sys.argv[2], sys.argv[3], os.path.basename(sys.argv[1]))
elif __name__ == "__main__" and len(sys.argv) > 3:
    write_bench_json(sys.argv[2], sys.argv[3], os.path.basename(sys.argv[1]))

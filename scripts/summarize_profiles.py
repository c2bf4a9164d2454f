#!/usr/bin/env python
"""Turns the ncu artefacts a GPU visit left in gpurun_out/ into the tracked summaries under profiles/.

    python scripts/summarize_profiles.py r01a        -> profiles/r01a_launches.md, r01a_ncu_<name>.md, r01a_bench_n1.json
"""
import collections
import csv
import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "gpurun_out")
PROF = os.path.join(ROOT, "profiles")

KEYS = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__inst_executed_pipe_tensor_subpipe_hmma.avg.pct_of_peak_sustained_active",
        "sm__throughput.avg.pct_of_peak_sustained_elapsed", "sm__warps_active.avg.pct_of_peak_sustained_active",
        "smsp__issue_active.avg.pct_of_peak_sustained_active", "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__pipe_alu_cycles_active.avg.pct_of_peak_sustained_active", "sm__pipe_xu_cycles_active.avg.pct_of_peak_sustained_active",
        "lts__t_sector_hit_rate.pct", "launch__registers_per_thread", "sm__cycles_elapsed.avg.per_second",
        "launch__grid_size", "launch__block_size", "smsp__warp_issue_stalled_long_scoreboard_per_warp_active.pct",
        "smsp__warp_issue_stalled_barrier_per_warp_active.pct", "smsp__warp_issue_stalled_math_pipe_throttle_per_warp_active.pct",
        "smsp__warp_issue_stalled_short_scoreboard_per_warp_active.pct", "smsp__warp_issue_stalled_wait_per_warp_active.pct",
        "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum", "launch__shared_mem_per_block_dynamic"]


def launches(tag):
    path = os.path.join(OUT, "launches.csv")
    if not os.path.exists(path):
        return
    lines = [l for l in open(path) if not l.startswith("==")]
    agg = collections.OrderedDict()
    for row in csv.DictReader(lines):
        if row.get("Metric Name") != "gpu__time_duration.sum":
            continue
        name = re.sub(r"\(.*", "", row["Kernel Name"]).replace("void unnamed>::", "")
        v = float(row["Metric Value"].replace(",", ""))
        v *= {"ns": 1, "us": 1e3, "ms": 1e6, "s": 1e9}.get(row["Metric Unit"], 1)
        key = (name, row["Grid Size"], row["Block Size"])
        a = agg.setdefault(key, [0, 0.0])
        a[0] += 1
        a[1] += v
    tot = sum(a[1] for a in agg.values())
    with open(os.path.join(PROF, f"{tag}_launches.md"), "w") as f:
        f.write(f"# {tag}: ncu launch list (`--metrics gpu__time_duration.sum --clock-control none`) of `bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-e2e`\n\n")
        f.write("Per-launch times under ncu are cold-cache and serialised: compare SHARES, not absolutes.\n")
        f.write(f"Window: {sum(a[0] for a in agg.values())} launches, {tot / 1e6:.3f} ms total.\n\n")
        f.write("| kernel | grid | block | launches | total ms | share | avg us |\n|---|---|---|---:|---:|---:|---:|\n")
        for (name, grid, block), (n, t) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write(f"| `{name}` | {grid} | {block} | {n} | {t / 1e6:.3f} | {100 * t / tot:.1f}% | {t / n / 1e3:.1f} |\n")
    shutil.copy(path, os.path.join(PROF, f"{tag}_launches.csv"))


def full(tag, rep):
    path = os.path.join(OUT, rep + ".ncu-rep")
    if not os.path.exists(path):
        return
    r = subprocess.run(["ncu", "-i", path, "--page", "raw", "--csv"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    rows = list(csv.reader(r.stdout.splitlines()))
    if len(rows) < 3:
        return
    hdr, units = rows[0], rows[1]
    with open(os.path.join(PROF, f"{tag}_ncu_{rep.replace('prof_', '')}.md"), "w") as f:
        f.write(f"# {tag}: `ncu --set full --clock-control none --import-source on` — {rep}\n\n")
        for row in rows[2:]:
            d = dict(zip(hdr, row))
            f.write(f"## {d.get('Kernel Name', '')[:160]}\n\ngrid {d.get('Grid Size')} block {d.get('Block Size')}\n\n| metric | value | unit |\n|---|---:|---|\n")
            for i, h in enumerate(hdr):
                if h in KEYS:
                    f.write(f"| {h} | {row[i]} | {units[i]} |\n")
            f.write("\n")


def traffic(tag):
    """DRAM bytes per launch of the dominant GEMM (3584 -> 1792: the 2nd of the 3 captured gemm launches) for bench.py's
    roofline.traffic field."""
    import json
    path = os.path.join(OUT, "prof_gemm.ncu-rep")
    if not os.path.exists(path):
        return
    r = subprocess.run(["ncu", "-i", path, "--page", "raw", "--csv"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    rows = list(csv.reader(r.stdout.splitlines()))
    if len(rows) < 3:
        return
    hdr, units, row = rows[0], rows[1], rows[2]      # first captured launch = gemm_mlp_2 of block 1
    def val(name):
        i = hdr.index(name)
        v = float(row[i].replace(",", ""))
        return v * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(units[i], 1)
    out = {"kernel": row[hdr.index("Kernel Name")][:80], "dram_bytes_read": val("dram__bytes_read.sum"),
           "dram_bytes_write": val("dram__bytes_write.sum"), "source": f"profiles/{tag}_ncu_gemm.md (ncu --set full, B = 64)"}
    out["traffic_bytes_per_launch"] = out["dram_bytes_read"] + out["dram_bytes_write"]
    # stamp: bench.py quotes the figure only for the machine code and launch size it was captured on
    hp = os.path.join(OUT, "kernel_hash.txt")
    out["kernel_hash"] = open(hp).read().strip() if os.path.exists(hp) else None
    out["kernel_hash_of"] = "sha256 of the SASS of gemm_tc_kernel<ACT_MISH, 0, false, true> (vision_transformer_detector_b200.build.kernel_hash)"
    out["rows_per_launch"] = 64 * 1296
    with open(os.path.join(PROF, "gemm_mlp_2_traffic.json"), "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    tag = sys.argv[1]
    os.makedirs(PROF, exist_ok=True)
    launches(tag)
    traffic(tag)
    for rep in sorted(x[:-8] for x in os.listdir(OUT) if x.endswith(".ncu-rep") and x.startswith("prof_")):
        full(tag, rep)
    for name in ("bench_n1.json", "bench_metric.json", "pytest_gpu.log", "bench_reference_n1.json", "smoke.log", "bench_fp32.json"):
        if os.path.exists(os.path.join(OUT, name)):
            shutil.copy(os.path.join(OUT, name), os.path.join(PROF, f"{tag}_{name}"))
    print(sorted(os.listdir(PROF)))

#!/usr/bin/env python
"""Turn the raw ncu outputs in profile_out/ into the small tracked summaries under profiles/.

    python scripts/summarize_profiles.py r1
"""
import csv
import io
import json
import os
import re
import subprocess
import sys
from collections import defaultdict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "profile_out")
PROF = os.path.join(ROOT, "profiles")

KEYS = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "sm__pipe_tensor_op_hmma_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__inst_executed_pipe_tensor.sum", "sm__warps_active.avg.pct_of_peak_sustained_active", "launch__registers_per_thread",
        "launch__grid_size", "launch__block_size", "sm__throughput.avg.pct_of_peak_sustained_elapsed", "sm__cycles_elapsed.avg",
        "smsp__inst_executed.sum", "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum", "lts__t_sector_hit_rate.pct",
        "sm__pipe_xu_cycles_active.avg.pct_of_peak_sustained_active", "smsp__cycles_active.avg", "dram__cycles_active.avg.pct_of_peak_sustained_elapsed"]


def short(name):
    m = re.search(r"(gemm_tc_kernel<[^>]*>|attn_fwd_kernel<[^>]*>|[a-z0-9_]+_kernel(<[^>]*>)?)", name)
    return m.group(1) if m else name[:60]


def launches(tag):
    path = os.path.join(OUT, f"launches_{tag}.csv")
    if not os.path.exists(path):
        return
    rows = []
    with open(path) as f:
        lines = [l for l in f if not l.startswith("==")]
    rd = csv.DictReader(io.StringIO("".join(lines)))
    for r in rd:
        if r.get("Metric Name") == "gpu__time_duration.sum":
            v = float(r["Metric Value"].replace(",", ""))
            unit = r.get("Metric Unit", "ns")
            scale = {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}.get(unit, 1e-3)
            rows.append((r["Kernel Name"], v * scale))
    agg = defaultdict(lambda: [0, 0.0])
    for k, us in rows:
        a = agg[short(k)]
        a[0] += 1
        a[1] += us
    tot = sum(a[1] for a in agg.values())
    os.makedirs(PROF, exist_ok=True)
    with open(os.path.join(PROF, f"{tag}_launch_list_summary.md"), "w") as f:
        f.write(f"# ncu launch list ({tag}): `ncu --metrics gpu__time_duration.sum --clock-control none` over bench.py --plms-steps 1\n\n")
        f.write(f"{len(rows)} launches, {tot/1e3:.2f} ms total (cold-cache, serialised: compare SHARES, not absolutes)\n\n")
        f.write("| kernel | launches | total us | share | mean us |\n|---|---:|---:|---:|---:|\n")
        for k, (n, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write(f"| `{k}` | {n} | {us:.1f} | {us/tot:.3f} | {us/n:.2f} |\n")
    print("wrote launch list summary:", len(rows), "launches")


def traffic(tag):
    """profiles/<tag>_gemm_dram_traffic.json from gpurun_out/traffic_<tag>.csv (ncu --metrics dram__bytes_read.sum,
    dram__bytes_write.sum -k regex:gemm_tc over bench.py --plms-steps 1); read by bench.py for roofline.traffic."""
    path = os.path.join(OUT, f"traffic_{tag}.csv")
    if not os.path.exists(path):
        return
    with open(path) as f:
        lines = [l for l in f if not l.startswith("==")]
    rd = csv.DictReader(io.StringIO("".join(lines)))
    rdb, wrb, ids = 0.0, 0.0, set()
    for r in rd:
        name = r.get("Metric Name", "")
        if not name.startswith("dram__bytes"):
            continue
        v = float(r["Metric Value"].replace(",", ""))
        unit = r.get("Metric Unit", "byte").lower()
        scale = {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, 1.0)
        ids.add(r["ID"])
        if "read" in name:
            rdb += v * scale
        else:
            wrb += v * scale
    n = max(len(ids), 1)
    alg = None
    bpo = os.path.join(OUT, "bench_per_op.json")
    if os.path.exists(bpo):
        ops = [o for o in json.load(open(bpo)) if o["kind"] in ("gemm", "conv3x3")]
        alg = sum(o["mbytes"] for o in ops) * 1e6 / max(len(ops), 1)
    out = {"kernel": "gemm_tc_kernel", "launches": n, "dram_bytes_read_per_launch": rdb / n, "dram_bytes_write_per_launch": wrb / n,
           "algorithmic_bytes_per_launch": alg,
           "how": "ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum --clock-control none -k regex:gemm_tc_kernel over bench.py --steps 1 "
                  "--warmup 1 --plms-steps 1 (B200; every launch serialised and replayed, caches flushed between replays)"}
    json.dump(out, open(os.path.join(PROF, f"{tag}_gemm_dram_traffic.json"), "w"), indent=1)
    print("wrote traffic:", out)


def full(tag, which):
    rep = os.path.join(OUT, f"prof_{which}_{tag}.ncu-rep")
    if not os.path.exists(rep):
        return
    r = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True)
    rd = list(csv.reader(io.StringIO(r.stdout)))
    if len(rd) < 3:
        print("empty report", rep, r.stderr[:500])
        return
    hdr, units = rd[0], rd[1]
    os.makedirs(PROF, exist_ok=True)
    with open(os.path.join(PROF, f"{tag}_ncu_full_{which}.md"), "w") as f:
        f.write(f"# ncu --set full --clock-control none ({tag}, {which}); values per launch\n\n")
        for row in rd[2:]:
            d = dict(zip(hdr, row))
            f.write(f"## {short(d.get('Kernel Name', '?'))}  grid {d.get('Grid Size', d.get('launch__grid_size', '?'))} block {d.get('Block Size', '?')}\n\n")
            for k in hdr:
                if any(k == key or k.startswith(key) for key in KEYS):
                    f.write(f"- {k} [{units[hdr.index(k)]}]: {d[k]}\n")
            f.write("\n")
    print("wrote", which)


if __name__ == "__main__":
    tag = sys.argv[1] if len(sys.argv) > 1 else "r1"
    launches(tag)
    traffic(tag)
    full(tag, "gemm")
    full(tag, "attn")

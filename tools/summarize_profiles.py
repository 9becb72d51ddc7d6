"""Turn the ncu artefacts in gpurun_out/ into the committed summaries under profiles/ (run in the build container).

    python tools/summarize_profiles.py r01
"""
import collections
import csv
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TAG = sys.argv[1] if len(sys.argv) > 1 else "r02"
OUT = os.path.join(ROOT, "profiles")
GO = os.path.join(ROOT, "gpurun_out")

METRICS = ["gpu__time_duration.sum", "launch__grid_size", "launch__block_size", "launch__registers_per_thread",
           "dram__bytes_read.sum", "dram__bytes_write.sum", "lts__t_bytes.sum", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
           "sm__throughput.avg.pct_of_peak_sustained_elapsed", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
           "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
           "smsp__inst_executed.sum", "l1tex__t_sectors_pipe_lsu_mem_global_op_ld.sum", "lts__t_sector_hit_rate.pct"]


def short(name):
    name = name.replace("gll::<unnamed>::", "").replace("void ", "").replace("unnamed>::", "")
    return name.split("(")[0]


def launches(path, out):
    rows = [r for r in csv.reader(open(path)) if len(r) > 10 and r[0].isdigit()]
    per = collections.OrderedDict()
    for r in rows:
        k = short(r[4])
        per.setdefault(k, []).append(float(r[-1]))
    tot = sum(sum(v) for v in per.values())
    with open(out, "w") as f:
        f.write(f"# ncu launch list ({os.path.basename(path)}): gpu__time_duration.sum per kernel, cold-cache and serialised\n")
        f.write("# command: python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-large-graph --no-sharded --no-cuda-graph (all launches, warm-up included)\n\n")
        f.write("| kernel | launches | mean us | total us | share |\n|---|---|---|---|---|\n")
        for k, v in sorted(per.items(), key=lambda kv: -sum(kv[1])):
            f.write(f"| {k} | {len(v)} | {sum(v) / len(v) / 1e3:.2f} | {sum(v) / 1e3:.1f} | {100 * sum(v) / tot:.1f}% |\n")
    print("wrote", out)


NAME_MAP = {"knn_gram_topk_tc_kernel": "knn_gram_topk_tcgen05", "knn_rerank_kernel": "knn_rerank", "cg_resident_kernel": "cg_persistent",
            "cg_persistent_kernel": "cg_persistent", "cg_small_kernel": "cg_persistent", "row_gather_kernel": "row_gather",
            "edge_grad_kernel": "edge_grad", "graph_weights_kernel": "graph_build"}
TRAFFIC = {}


def to_bytes(v, unit):
    scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)
    return float(v.replace(",", "")) * scale


def full(rep, out):
    txt = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(txt.splitlines()))
    hdr, units = rows[0], rows[1]
    wl = "c4" if "_c4_" in os.path.basename(rep) else "c2"
    for r in rows[2:]:
        nm = short(r[hdr.index("Kernel Name")]).split("<")[0]
        ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
        TRAFFIC.setdefault(wl, {}).setdefault(NAME_MAP.get(nm, nm), []).append(to_bytes(r[ir], units[ir]) + to_bytes(r[iw], units[iw]))
    with open(out, "w") as f:
        f.write(f"# ncu --set full summary of {os.path.basename(rep)} (one row block per captured launch)\n\n")
        for r in rows[2:]:
            f.write(f"## {short(r[hdr.index('Kernel Name')])}\n\n")
            for m in METRICS:
                if m in hdr:
                    i = hdr.index(m)
                    f.write(f"- {m} = {r[i]} {units[i]}\n")
            f.write("\n")
    print("wrote", out)


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    for nm in os.listdir(GO):
        if nm.startswith(TAG + "_launches") and nm.endswith(".csv"):
            launches(os.path.join(GO, nm), os.path.join(OUT, nm[:-4] + ".md"))
        if nm.startswith(TAG) and nm.endswith(".ncu-rep"):
            full(os.path.join(GO, nm), os.path.join(OUT, nm[:-8] + "_ncu_full.md"))
    if TRAFFIC:
        import json

        out = {wl: {k: sum(v) / len(v) for k, v in d.items()} for wl, d in TRAFFIC.items()}
        out["_source"] = f"dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full captures tagged {TAG}"
        json.dump(out, open(os.path.join(OUT, "ncu_traffic.json"), "w"), indent=1)
        print("wrote ncu_traffic.json", out)

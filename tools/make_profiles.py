"""Turn ncu output brought back in gpurun_out/ into the committed summaries under profiles/.

  python tools/make_profiles.py step  gpurun_out/step_metrics.csv   profiles/r01_step_launches.csv
      per-launch duration + DRAM bytes of ONE benchmark step (ncu --metrics gpu__time_duration.sum,
      dram__bytes_read.sum,dram__bytes_write.sum --csv), plus profiles/r01_traffic.json for bench.py
  python tools/make_profiles.py full  gpurun_out/prof.ncu-rep       profiles/r01_kernels_full.md
      headline metrics of an `ncu --set full` capture (tools/profile_kernels.py), one block per kernel launch
"""
import csv
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def short(name):
    n = name.replace("void ", "").replace("v100::", "")
    return n.split("(")[0]


def kind_of(name):
    if "conv_gemm" in name:
        return "gemm"
    if "dw_" in name:
        return "dwconv"
    if "logmel" in name:
        return "logmel"
    if "ctc_finalize" in name:
        return "ctc_finalize"
    return "other"


def step(src, dst):
    lines = [l for l in open(src) if not l.startswith("==")]
    rows = list(csv.DictReader(lines))
    # group the (kernel id -> metrics) triples
    by_id = {}
    for r in rows:
        d = by_id.setdefault(int(r["ID"]), {"name": r["Kernel Name"], "grid": r["Grid Size"], "block": r["Block Size"]})
        d[r["Metric Name"]] = float(r["Metric Value"].replace(",", "")) * {"ns": 1e-3, "us": 1.0, "ms": 1e3, "byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(r["Metric Unit"], 1.0)
    ids = sorted(by_id)
    mel = [i for i in ids if "logmel" in by_id[i]["name"]]
    start = mel[-2] if len(mel) >= 2 else mel[-1]          # one full step, away from the warm-up
    end = next((i for i in ids if i > start and "logmel" in by_id[i]["name"]), ids[-1] + 1)
    sel = [i for i in ids if start <= i < end]
    tot = sum(by_id[i]["gpu__time_duration.sum"] for i in sel)
    out = ["# one ASR step (asr_en_base, 256 x 15 s) under ncu: cold-cache, serialised -- compare SHARES, not absolutes",
           "kernel,grid,block,duration_us,share,dram_read_MB,dram_write_MB"]
    agg = {}
    for i in sel:
        d = by_id[i]
        us = d["gpu__time_duration.sum"]
        rd, wr = d.get("dram__bytes_read.sum", 0.0), d.get("dram__bytes_write.sum", 0.0)
        out.append(f'"{short(d["name"])}","{d["grid"]}","{d["block"]}",{us:.1f},{us / tot:.4f},{rd / 1e6:.1f},{wr / 1e6:.1f}')
        a = agg.setdefault(kind_of(d["name"]), dict(us=0.0, bytes=0.0, launches=0))
        a["us"] += us; a["bytes"] += rd + wr; a["launches"] += 1
    out.append("# total %.3f ms; " % (tot / 1e3) + "; ".join(f"{k}: share {v['us'] / tot:.3f}, {v['launches']} launches, DRAM {v['bytes'] / 1e9:.2f} GB" for k, v in agg.items()))
    open(dst, "w").write("\n".join(out) + "\n")
    traffic = {k: dict(dram_bytes_per_step=v["bytes"], launches=v["launches"], dram_bytes_per_launch=v["bytes"] / v["launches"],
                       share_of_step=v["us"] / tot) for k, v in agg.items()}
    tj = os.path.join(os.path.dirname(dst), os.path.basename(dst).split("_")[0] + "_traffic.json")   # r02_traffic.json
    json.dump({"source": os.path.basename(dst), "per_kernel_class": traffic}, open(tj, "w"), indent=1)
    print(out[-1])


WANT = [("gpu__time_duration.sum", "duration"), ("dram__bytes_read.sum", "DRAM read"), ("dram__bytes_write.sum", "DRAM write"),
        ("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "DRAM % of peak"),
        ("lts__throughput.avg.pct_of_peak_sustained_elapsed", "L2 % of peak"),
        ("l1tex__throughput.avg.pct_of_peak_sustained_elapsed", "L1/smem % of peak"),
        ("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "tensor pipe active %"),
        ("smsp__issue_active.avg.pct_of_peak_sustained_active", "issue active %"),
        ("sm__warps_active.avg.pct_of_peak_sustained_active", "warps active %"),
        ("launch__registers_per_thread", "registers/thread"),
        ("smsp__inst_executed.sum", "warp instructions"),
        ("l1tex__data_pipe_lsu_wavefronts_mem_shared.sum", "smem wavefronts"),
        ("sm__cycles_elapsed.avg", "SM cycles")]


def full(src, dst):
    raw = subprocess.run(["ncu", "-i", src, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(raw.splitlines()))
    hdr, units, data = rows[0], rows[1], rows[2:]
    col = {h: i for i, h in enumerate(hdr)}
    out = [f"# ncu --set full --clock-control none ({os.path.basename(src)}), kernels launched by tools/profile_kernels.py",
           "# shapes: asr_en_base layers at B=256, T=751 (1501 for the stride-2 block); one block per launch", ""]
    seen = {}
    for r in data:
        name = short(r[col["Kernel Name"]])
        key = (name, r[col["Grid Size"]])
        seen[key] = seen.get(key, 0) + 1
        if seen[key] > 1 and "gemm" not in name:
            continue                                   # identical repeat launches: keep one
        out.append(f"## {name}  grid {r[col['Grid Size']]} block {r[col['Block Size']]}")
        for m, label in WANT:
            if m in col:
                out.append(f"- {label}: {r[col[m]]} {units[col[m]]}")
        out.append("")
    open(dst, "w").write("\n".join(out))
    print("wrote", dst, len(data), "launches")


if __name__ == "__main__":
    {"step": step, "full": full}[sys.argv[1]](sys.argv[2], sys.argv[3])

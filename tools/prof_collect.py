"""Turns the ncu outputs of tools/prof_round.sh (gpurun_out/<tag>_*) into the tracked summaries under profiles/:
  profiles/<tag>_launches_summary.txt   per-kernel share of one bench pass from the launch list
  profiles/<tag>_ncu_<kernel>.txt       the numbers DESIGN.md quotes from each --set full capture
  profiles/roofline_traffic.json        dram bytes (read + write) per launch per bench kernel tag
usage: python tools/prof_collect.py r1"""
import csv
import glob
import json
import os
import subprocess
import sys

tag = sys.argv[1] if len(sys.argv) > 1 else "r1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
out_dir = os.path.join(ROOT, "profiles")
os.makedirs(out_dir, exist_ok=True)

# ---- launch list
path = os.path.join(ROOT, "gpurun_out", f"{tag}_launches.csv")
if os.path.exists(path):
    lines = [l for l in open(path) if l.startswith('"')]
    rows = list(csv.reader(lines))
if os.path.exists(path) and rows:
    hdr = rows[0]
    ik, iv, im = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Name")
    agg = {}
    for r in rows[1:]:
        if r[im] != "gpu__time_duration.sum":
            continue
        name = r[ik].split("(")[0].replace("void sb::<unnamed>::", "").replace("void sb::", "")
        n, t = agg.get(name, (0, 0.0))
        agg[name] = (n + 1, t + float(r[iv].replace(",", "")))
    tot = sum(t for _, t in agg.values()) or 1.0
    with open(os.path.join(out_dir, f"{tag}_launches_summary.txt"), "w") as f:
        f.write(f"# ncu --metrics gpu__time_duration.sum --clock-control none, one bench pass ({sum(n for n, _ in agg.values())} launches, "
                f"{tot / 1e6:.3f} ms summed; cold-cache serialised times: compare SHARES)\n")
        for name, (n, t) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write(f"{name:60s} launches={n:5d} total_us={t / 1e3:10.1f} avg_us={t / 1e3 / n:8.2f} share={t / tot:.4f}\n")
    print(open(os.path.join(out_dir, f"{tag}_launches_summary.txt")).read())

# ---- full captures
WANT = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "launch__registers_per_thread", "launch__grid_size", "launch__block_size",
        "smsp__inst_executed.sum", "smsp__issue_active.avg.pct_of_peak_sustained_active", "lts__throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__cycles_active.avg", "sm__cycles_active.max", "sm__cycles_elapsed.avg"]
TAGS = {"cross_attention_kernel": "dec_cross_attention", "out_argmax_kernel": "dec_gemm_out_argmax", "dec_ssru_kernel": "dec_ssru_q_fused",
        "self_attention_kernel": "enc_self_attention",
        "cross_attention_rc_kernel": "dec_cross_attention_rc", "cross_attention_rcl_kernel": "dec_cross_attention_rc",
        "enc_attention_kernel": "enc_qkv_attention_fused", "enc_attention_warp_kernel": "enc_qkv_attention_fused"}
traffic = {}
tpath = os.path.join(out_dir, "roofline_traffic.json")
if os.path.exists(tpath):
    traffic = json.load(open(tpath))
UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
for rep in sorted(glob.glob(os.path.join(ROOT, "gpurun_out", f"{tag}_*.ncu-rep"))):
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(raw.splitlines()))
    if len(rows) < 3:
        continue
    hdr, units = rows[0], rows[1]
    base = os.path.basename(rep)[:-len(".ncu-rep")]
    with open(os.path.join(out_dir, f"{base}.txt"), "w") as f:
        f.write(f"# ncu --set full --clock-control none --import-source on, from {os.path.basename(rep)} (python bench.py --steps 1 --warmup 3)\n")
        for r in rows[2:]:
            kname = r[hdr.index("Kernel Name")]
            f.write(f"kernel: {kname}\n")
            vals = {}
            for w in WANT:
                if w in hdr:
                    i = hdr.index(w)
                    vals[w] = (r[i], units[i])
                    f.write(f"  {w:72s} {r[i]} {units[i]}\n")
            st = []
            for i, h in enumerate(hdr):
                if "issue_stalled" in h and "per_issue_active" in h:
                    try:
                        st.append((float(r[i]), h.split("issue_stalled_")[1].split("_per_issue")[0]))
                    except ValueError:
                        pass
            f.write("  top stalls (warps per issue-active cycle): " + ", ".join(f"{n}={v:.2f}" for v, n in sorted(st, reverse=True)[:6]) + "\n")
            try:
                rd = float(vals["dram__bytes_read.sum"][0]) * UNIT[vals["dram__bytes_read.sum"][1]]
                wr = float(vals["dram__bytes_write.sum"][0]) * UNIT[vals["dram__bytes_write.sum"][1]]
                for pat, btag in TAGS.items():
                    if pat in kname:
                        traffic[btag] = rd + wr
                if "rows_ffn_kernel" in kname:
                    traffic["enc_wo_ffn_fused" if ", 128>" in kname or ", (int)128>" in kname else "dec_wo_ffn_fused"] = rd + wr
            except (KeyError, ValueError):
                pass
    print("wrote", base + ".txt")
json.dump(traffic, open(tpath, "w"), indent=1, sort_keys=True)
print(json.dumps(traffic))

#!/usr/bin/env python
"""Turn gpurun_out/launches_*.csv and prof_step_*.ncu-rep into the summaries committed under profiles/.
   python tools/summarise_profiles.py <launches.csv> <prof.ncu-rep> <tag>"""
import collections
import csv
import json
import re
import subprocess
import sys
from pathlib import Path

REPO = Path(__file__).resolve().parents[1]
launch_csv, rep, tag = sys.argv[1], sys.argv[2], sys.argv[3]


def short(name):
    for k in ("pipe_head_fwd_kernel", "pipe_head_bwd_dx_kernel", "head_dw2_kernel"):
        if k in name:
            return k
    if "rowgemm_ts_kernel" in name:
        return "rowgemm_ts<" + ("PipeFeatLoader,HeadFwdEpilogue" if "PipeFeat" in name else "DpreLoader,HeadBwdEpilogue") + ">"
    if "rowgemm_kernel" in name:
        return "rowgemm<RowLoader,StoreEpilogue>"
    if "tgrad_kernel" in name:
        return "tgrad<" + ("HeadDpre,HeadFeatOnes" if "HeadDpre" in name else "DgRows,GruInputRows" if "DgRows" in name
                           else "StackedRows,RowsThenOne" if "RowsThenOne" in name else "StackedRows") + ">"
    m = re.search(r"spmm_staged_kernel<(?:\(bool\))?(\d), (?:\(bool\))?(\d)>", name)
    if m:
        return f"spmm_staged_kernel<epi={m.group(1)},gate={m.group(2)}>"
    if "spmm_staged" in name:
        return "spmm_staged_kernel"
    for k in ("gru_fwd_kernel", "gru_bwd_hn_kernel", "node_init_fwd_kernel", "gate_extract_kernel", "mean_pool_kernel",
              "pool_bwd_fill_kernel", "reduce_parts_kernel", "colsum_reduce_kernel", "gather_partials_kernel",
              "spmm_gather_kernel"):
        if k in name:
            return k
    return "torch: " + name.split("(")[0][-60:]


rows = list(csv.reader(open(launch_csv)))
h = [i for i, r in enumerate(rows) if r and r[0] == "ID"][0]
hdr = rows[h]
ik, iv, iu = hdr.index("Kernel Name"), hdr.index("Metric Value"), hdr.index("Metric Unit")
ev = []
for r in rows[h + 1:]:
    if len(r) <= iv:
        continue
    t = float(r[iv].replace(",", "")) * {"nsecond": 1, "ns": 1, "usecond": 1e3, "us": 1e3, "msecond": 1e6, "ms": 1e6}.get(r[iu], 1)
    ev.append((short(r[ik]), t))
steps, i = [], 0
while i < len(ev):
    if ev[i][0].startswith("node_init_fwd"):
        j = i
        while j < len(ev) and not ev[j][0].startswith("gate_extract"):
            j += 1
        j = min(j + 6, len(ev) - 1)  # the sensor-row GEMMs and reductions that finish node_init_bwd
        seg = ev[i:j + 1]
        if not any("gru" in k for k, _ in seg):
            steps.append(seg)
        i = j + 1
    else:
        i += 1
agg = collections.OrderedDict()
for seg in steps:
    for k, t in seg:
        a = agg.setdefault(k, [0, 0.0])
        a[0] += 1
        a[1] += t
tot = sum(v[1] for v in agg.values())
out = [f"# ncu launch list, GNN-stack steps only (node_init_fwd .. end of node_init_bwd), {tag}",
       "# command: ncu --metrics gpu__time_duration.sum --clock-control none -c 1500 --csv python bench.py --steps 2 --warmup 3 --no-cpu-baseline",
       f"# {len(steps)} steps at B=4096, L-TOWN-A, P=764; cold-cache, serialised launches: compare SHARES with bench.py's live `kernels`",
       "kernel,launches,total_ms,ms_per_launch,share_of_step"]
for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1]):
    out.append(f"\"{k}\",{v[0]},{v[1] / 1e6:.3f},{v[1] / 1e6 / v[0]:.4f},{v[1] / tot:.4f}")
out.append(f"# total per step: {tot / 1e6 / max(len(steps), 1):.3f} ms")
(REPO / "profiles" / f"{tag}_launches_stack_steps.csv").write_text("\n".join(out) + "\n")
print("\n".join(out[3:20]), "\n", out[-1])

raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
rows = list(csv.reader(raw.splitlines()))
hdr, units = rows[0], rows[1]
want = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "launch__registers_per_thread", "launch__shared_mem_per_block_dynamic", "lts__t_sector_hit_rate.pct"]
want = [w for w in want if w in hdr]
name_map = {"spmm_staged_kernel<epi=1,gate=0>": "spmm_fused_fwd", "spmm_staged_kernel<epi=0,gate=1>": "spmm_fused_bwd",
            "rowgemm<RowLoader,StoreEpilogue>": "linear_tc", "rowgemm_ts<PipeFeatLoader,HeadFwdEpilogue>": "pipe_head_fwd",
            "rowgemm_ts<DpreLoader,HeadBwdEpilogue>": "pipe_head_bwd_dx", "tgrad<StackedRows>": "wgrad_tc",
            "tgrad<HeadDpre,HeadFeatOnes>": "pipe_head_bwd_w", "head_dw2_kernel": "pipe_head_bwd_w",
            "pipe_head_fwd_kernel": "pipe_head_fwd", "pipe_head_bwd_dx_kernel": "pipe_head_bwd_dx",
            "node_init_fwd_kernel": "node_init_fwd",
            "gate_extract_kernel": "node_init_bwd(gate_extract)", "mean_pool_kernel": "mean_pool_fwd",
            "pool_bwd_fill_kernel": "mean_pool_bwd"}
table = [["kernel"] + want]
traffic = collections.defaultdict(lambda: collections.defaultdict(list))  # op -> kernel -> bytes per launch
mult = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1}[units[hdr.index("dram__bytes_read.sum")]]
for r in rows[2:]:
    s = short(r[hdr.index("Kernel Name")])
    table.append([s] + [r[hdr.index(w)] for w in want])
    if s in name_map and float(r[hdr.index("gpu__time_duration.sum")]) * {"us": 1, "usecond": 1, "ms": 1e3, "msecond": 1e3, "ns": 1e-3, "nsecond": 1e-3}.get(units[hdr.index("gpu__time_duration.sum")], 1) > 60:
        traffic[name_map[s]][s].append((float(r[hdr.index("dram__bytes_read.sum")]) + float(r[hdr.index("dram__bytes_write.sum")])) * mult)
with open(REPO / "profiles" / f"{tag}_kernels_ncu_full.csv", "w", newline="") as f:
    w = csv.writer(f)
    w.writerow([f"# ncu --set full --clock-control none; one GNN-stack fwd+bwd at B=4096, L-TOWN-A, D=64, P=764 (tools/prof_step.py 4096 2); units "
                + str({x: units[hdr.index(x)] for x in want})])
    w.writerows(table)
tpath = REPO / "profiles" / "ncu_traffic.json"
t = json.loads(tpath.read_text()) if tpath.exists() else {"B4096_P764": {}}
for k, per_kernel in traffic.items():  # an op's traffic = sum over its kernels of the mean bytes per launch
    t["B4096_P764"][k.split("(")[0]] = sum(sum(v) / len(v) for v in per_kernel.values())
tpath.write_text(json.dumps(t, indent=1))
for row in table[1:]:
    print(row[:6])

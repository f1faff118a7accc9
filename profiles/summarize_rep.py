"""Turns an `ncu --set full` report into the committed text summary + the traffic.json entry bench.py reads.

usage: python profiles/summarize_rep.py gpurun_out/full_r1_c2.ncu-rep <workload> profiles/r1_full_c2.txt
Per launch: duration, DRAM bytes (read+write), L2 bytes, SM/FP64-pipe utilisation, issue-slot use, occupancy, regs."""
import collections
import csv
import io
import json
import os
import re
import subprocess
import sys

M = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum", "lts__t_bytes.sum",
     "sm__throughput.avg.pct_of_peak_sustained_elapsed", "gpu__compute_memory_throughput.avg.pct_of_peak_sustained_elapsed",
     "sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
     "sm__warps_active.avg.pct_of_peak_sustained_active", "launch__registers_per_thread", "launch__grid_size",
     "launch__block_size", "dram__throughput.avg.pct_of_peak_sustained_elapsed",
     "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum", "smsp__warp_issue_stalled_long_scoreboard_per_warp_active.pct",
     "smsp__warp_issue_stalled_barrier_per_warp_active.pct", "smsp__warp_issue_stalled_short_scoreboard_per_warp_active.pct",
     "sm__pipe_tensor_cycles_active_realtime.avg.pct_of_peak_sustained_elapsed", "sm__mem_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed",
     "l1tex__data_pipe_tc_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed", "lts__throughput.avg.pct_of_peak_sustained_elapsed",
     "l1tex__throughput.avg.pct_of_peak_sustained_elapsed"]
NAMES = {"smallnet_fwd_bwd_kernel<1, 0>": "smallnet_fwd_bwd_kernel(fused features)", "smallnet_fwd_bwd_kernel<2, 0>": "smallnet_fwd_bwd_kernel(fused features)",
         # (ncu runs on one GPU only: the <2, 1> instance seen there is the single-GPU prewait, not the data-parallel one)
         "smallnet_fwd_bwd_kernel<2, 1>": "smallnet_fwd_bwd_kernel(fused features, front end ahead of the wait)",
         "smallnet_fwd_bwd_kernel<0, 0>": "smallnet_fwd_bwd_kernel", "smallnet_wgrad_kernel<2>": "smallnet_wgrad_kernel(+SGD update)",
         "smallnet_wgrad_kernel<0>": "smallnet_wgrad_kernel", "smallnet_wgrad_kernel<1>": "smallnet_wgrad_kernel"}


def to_bytes(v, unit):
    v = float(v.replace(",", ""))
    return v * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(unit, 1)


def main(rep, workload, out_txt):
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True, check=True).stdout
    rows = list(csv.reader(io.StringIO(raw)))
    hdr, units = rows[0], rows[1]
    col = {h: i for i, h in enumerate(hdr)}
    agg = collections.OrderedDict()
    for r in rows[2:]:
        name = re.sub(r"^void ", "", r[col["Kernel Name"]])
        name = re.sub(r"\(.*", "", name)
        rec = agg.setdefault(name, collections.defaultdict(list))
        for m in M:
            if m not in col:
                cands = [h for h in hdr if h.endswith(m)]
                if cands:
                    col[m] = col[cands[0]]
            if m in col and r[col[m]] not in ("", "n/a", "no data"):
                v = r[col[m]]
                try:
                    rec[m].append(to_bytes(v, units[col[m]]) if "bytes" in m else float(v.replace(",", "")))
                except ValueError:
                    pass
    note = sys.argv[4] if len(sys.argv) > 4 else "ncu --set full --clock-control none"
    lines = [f"# {os.path.basename(rep)}  ({note})"]
    traffic = {}
    for name, rec in agg.items():
        n = len(rec["gpu__time_duration.sum"])
        lines.append(f"\n## {name}  launches={n}")
        for m in M:
            if rec[m]:
                lines.append(f"  {m:82s} {sum(rec[m]) / len(rec[m]):16.3f}")
        if rec["dram__bytes_read.sum"]:
            key = NAMES.get(name.split("(")[0], re.sub(r"<.*", "", name))
            traffic[key] = (sum(rec["dram__bytes_read.sum"]) + sum(rec["dram__bytes_write.sum"])) / n
    open(out_txt, "w").write("\n".join(lines) + "\n")
    tpath = os.path.join(os.path.dirname(os.path.abspath(__file__)), "traffic.json")
    t = json.load(open(tpath)) if os.path.exists(tpath) else {}
    t[workload] = traffic
    json.dump(t, open(tpath, "w"), indent=1, sort_keys=True)
    print("\n".join(lines))


if __name__ == "__main__":
    main(*sys.argv[1:4])

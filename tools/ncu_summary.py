#!/usr/bin/env python
"""Condense an `ncu --set full` report into the per-kernel table kept under profiles/.
usage: python tools/ncu_summary.py report.ncu-rep [--traffic-json profiles/rNN_traffic.json] > profiles/rNN_ncu_full_summary.txt

--traffic-json also writes {launch-site name: dram__bytes_read.sum + dram__bytes_write.sum per launch}, the file
bench.py reads for `roofline.traffic` (launch-site names as in csrc/api.cu: mlp_fused_fwd, mlp_fused_bwd, wgrad)."""
import json
import csv
import io
import subprocess
import sys

KEEP = [
    "gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
    "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
    "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
    "sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active",
    "sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active",
    "smsp__issue_active.avg.pct_of_peak_sustained_active", "sm__warps_active.avg.pct_of_peak_sustained_active",
    "launch__registers_per_thread", "launch__shared_mem_per_block_dynamic", "launch__grid_size", "launch__block_size",
    "lts__t_sectors_srcunit_tex_op_read.sum",
    "smsp__average_warps_issue_stalled_barrier_per_issue_active.ratio",
    "smsp__average_warps_issue_stalled_long_scoreboard_per_issue_active.ratio",
    "smsp__average_warps_issue_stalled_wait_per_issue_active.ratio",
    "smsp__average_warps_issue_stalled_mio_throttle_per_issue_active.ratio",
    "smsp__average_warps_issue_stalled_short_scoreboard_per_issue_active.ratio",
    "smsp__average_warps_issue_stalled_math_pipe_throttle_per_issue_active.ratio",
]


SITES = {"mlp_fused_pair_kernel": "mlp_fused_fwd", "mlp_fused_bwd_kernel": "mlp_fused_bwd", "wgrad_kernel": "wgrad"}
MULT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}


def main():
    rep = sys.argv[1]
    traffic_path = sys.argv[sys.argv.index("--traffic-json") + 1] if "--traffic-json" in sys.argv else None
    traffic = {}
    raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True, check=True).stdout
    rows = list(csv.reader(io.StringIO(raw)))
    hdr, units, data = rows[0], rows[1], rows[2:]
    col = {h: i for i, h in enumerate(hdr)}
    for r in data:
        print("---")
        print("%-90s %s" % ("Kernel Name", r[col["Kernel Name"]]))
        for k in KEEP:
            if k in col:
                print("%-90s %s %s" % (k, r[col[k]], units[col[k]]))
        name = r[col["Kernel Name"]]
        for pat, site in SITES.items():
            if pat in name and site not in traffic:
                tot = 0.0
                for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    tot += float(r[col[k]].replace(",", "")) * MULT.get(units[col[k]], 1.0)
                traffic[site] = tot
    if traffic_path:
        json.dump(traffic, open(traffic_path, "w"), indent=1)


if __name__ == "__main__":
    main()

"""profiles/<tag>_large_chain_kernels.md from the raw ncu pages written by tools/ncu_big.sh.
usage: python tools/large_chain_summary.py <tag>"""
import csv
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
tag = sys.argv[1]
G, P = os.path.join(ROOT, "gpurun_out"), os.path.join(ROOT, "profiles")
CASES = [("cfg4 x 0.05 (500 chains of 200-330 reads)", f"{tag}_cfg4_sparse_raw.csv"),
         ("cfg1 (one chain of 1,400 reads)", f"{tag}_cfg1_sparse_raw.csv")]


def val(hdr, row, name):
    return row[hdr.index(name)] if name in hdr else ""


def unit(hdr, units, name):
    return units[hdr.index(name)] if name in hdr else ""


lines = [f"# Large-chain cluster editing under `ncu --set full --clock-control none` ({tag}; tools/ncu_big.sh)", "",
         "| case | kernel | grid x block | ms | warp instructions | IPC (whole GPU) | lanes/inst | regs | warps active % | L2 hit % | dram R / W | top stalls (cycles per issue) |",
         "|---|---|---|---|---|---|---|---|---|---|---|---|"]
for what, fn in CASES:
    path = os.path.join(G, fn)
    if not os.path.exists(path):
        continue
    rows = list(csv.reader(open(path)))
    if len(rows) < 3:
        continue
    hdr, units = rows[0], rows[1]
    for r in rows[2:]:
        stalls = []
        for i, h in enumerate(hdr):
            if "issue_stalled" in h and h.endswith("per_issue_active.ratio") and "not_issued" not in h:
                try:
                    stalls.append((float(r[i]), h.replace("smsp__average_warps_issue_stalled_", "").replace("_per_issue_active.ratio", "")))
                except ValueError:
                    pass
        stalls.sort(reverse=True)
        top = ", ".join(f"{n} {v:.1f}" for v, n in stalls[:3])
        name = val(hdr, r, "Kernel Name").split("(")[0].replace("void ", "")
        dr = f"{val(hdr, r, 'dram__bytes_read.sum')} {unit(hdr, units, 'dram__bytes_read.sum')} / {val(hdr, r, 'dram__bytes_write.sum')} {unit(hdr, units, 'dram__bytes_write.sum')}"
        lines.append(f"| {what} | `{name}` | {val(hdr, r, 'Grid Size')} x {val(hdr, r, 'Block Size')} | {float(val(hdr, r, 'gpu__time_duration.sum')):.2f} | "
                     f"{float(val(hdr, r, 'smsp__inst_executed.sum')) / 1e6:.1f} M | {float(val(hdr, r, 'sm__inst_executed.avg.per_cycle_elapsed')):.3f} | "
                     f"{val(hdr, r, 'smsp__thread_inst_executed_per_inst_executed.ratio')} | {val(hdr, r, 'launch__registers_per_thread')} | "
                     f"{float(val(hdr, r, 'sm__warps_active.avg.pct_of_peak_sustained_active')):.0f} | {float(val(hdr, r, 'lts__t_sector_hit_rate.pct')):.0f} | {dr} | {top} |")
lines += ["", "IPC is per SM averaged over all 148: a one-chain launch (cfg1) occupies one SM, so its own IPC is 148 x the figure.", ""]
open(os.path.join(P, f"{tag}_large_chain_kernels.md"), "w").write("\n".join(lines))
print("\n".join(lines))

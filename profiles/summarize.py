"""Turn gpurun_out ncu artefacts into the small text summaries committed under profiles/.

    python profiles/summarize.py launches gpurun_out/launches_X.csv  > profiles/rN_launches.txt
    python profiles/summarize.py raw      gpurun_out/raw_X.csv       > profiles/rN_kernels.txt
    python profiles/summarize.py traffic  gpurun_out/launches_X.csv  > profiles/ncu_traffic.json
(raw csv = `ncu -i prof.ncu-rep --page raw --csv`)
"""
import collections
import csv
import sys

WANT = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "sm__throughput.avg.pct_of_peak_sustained_elapsed",
        "launch__grid_size", "launch__block_size", "launch__registers_per_thread",
        "launch__occupancy_limit_registers", "launch__occupancy_limit_shared_mem",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__inst_executed.sum",
        "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__inst_executed_pipe_xu.sum", "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum",
        "lts__t_sector_hit_rate.pct", "smsp__cycles_active.avg",
        "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed",
        "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
        "lts__throughput.avg.pct_of_peak_sustained_elapsed", "l1tex__throughput.avg.pct_of_peak_sustained_elapsed",
        "smsp__pcsamp_warps_issue_stalled_long_scoreboard", "smsp__pcsamp_warps_issue_stalled_wait",
        "smsp__pcsamp_warps_issue_stalled_barrier", "smsp__pcsamp_warps_issue_stalled_short_scoreboard",
        "smsp__pcsamp_warps_issue_stalled_selected", "smsp__pcsamp_warps_issue_stalled_math_pipe_throttle"]


def launches(path):
    lines = [l for l in open(path) if not l.startswith("==")]
    d = collections.defaultdict(list)
    for row in csv.DictReader(lines):
        if row.get("Metric Name", "gpu__time_duration.sum") != "gpu__time_duration.sum":
            continue
        d[row["Kernel Name"][:90]].append(float(row["Metric Value"].replace(",", "")))
    tot = sum(sum(v) for v in d.values())
    print("# ncu --metrics gpu__time_duration.sum --clock-control none (cold-cache, serialised: compare SHARES)")
    print("%-92s %5s %10s %10s %6s" % ("kernel", "n", "avg_us", "total_us", "share"))
    for k, v in sorted(d.items(), key=lambda kv: -sum(kv[1])):
        print("%-92s %5d %10.1f %10.1f %5.1f%%" % (k, len(v), sum(v) / len(v) / 1e3, sum(v) / 1e3, 100 * sum(v) / tot))


ENTRY_OF = [("readloss8_kernel", "pm_readloss_fwd8"), ("labels_pack_kernel", "pm_labels_pack"),
            ("conv1x1_nn_kernel", "pm_conv1x1_fwd"), ("conv1x1_wgrad_kernel", "pm_conv1x1_wgrad"),
            ("read_fwd_tiled_kernel", "pm_read_fwd"), ("read_fwd_kernel", "pm_read_fwd"),
            ("colsoftmax_apply_kernel", "pm_colsoftmax_apply"), ("readloss_kernel", "pm_readloss_fwd"),
            ("bn_stats_kernel", "pm_bn_stats"), ("bn_apply_kernel", "pm_bn_apply"),
            ("write_reduce_mma_kernel", "pm_write_reduce_fwd"), ("write_reduce_tiled_kernel", "pm_write_reduce_fwd"),
            ("update_fwd_kernel", "pm_update_fwd"), ("update_bwd_kernel", "pm_update_bwd"),
            ("write_bwd_tiled_kernel", "pm_write_bwd"), ("bn_bwd_reduce_rows_kernel", "pm_bn_bwd_reduce_rows"),
            ("readloss8_kernel", "pm_readloss_fwd8"), ("readloss_cells_kernel", "pm_readloss_fwd8"),
            ("bn_bwd_apply_kernel", "pm_bn_bwd_apply"), ("read_bwd_ds_tiled_kernel", "pm_read_bwd.ds"), ("read_bwd_ds_planes_kernel", "pm_read_bwd.ds"),
            ("read_bwd_dx_tiled_kernel", "pm_read_bwd.dx"), ("read_bwd_dx_tma_kernel", "pm_read_bwd.dx")]


def traffic(path, dtype="f32"):
    """{dtype: {C-ABI entry: dram bytes (read+write) per launch}} from a launch csv that carries
    dram__bytes_read.sum / dram__bytes_write.sum / gpu__time_duration.sum per launch (bench.py reads it)."""
    import json

    lines = [l for l in open(path) if not l.startswith("==")]
    per = collections.defaultdict(lambda: collections.defaultdict(float))  # launch id -> metric -> value
    name = {}
    for row in csv.DictReader(lines):
        v = float(row["Metric Value"].replace(",", ""))
        unit = row.get("Metric Unit", "")
        v *= {"Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "byte": 1.0, "us": 1e3, "ms": 1e6, "ns": 1.0, "usecond": 1e3,
              "nsecond": 1.0, "msecond": 1e6}.get(unit, 1.0)
        per[row["ID"]][row["Metric Name"]] = v
        name[row["ID"]] = row["Kernel Name"]
    agg = collections.defaultdict(list)
    for i, m in per.items():
        for pat, ent in ENTRY_OF:
            if pat in name[i]:
                agg[ent].append((m.get("dram__bytes_read.sum", 0.0) + m.get("dram__bytes_write.sum", 0.0),
                                 m.get("gpu__time_duration.sum", 0.0) / 1e3))
                break
    out, detail = {}, {}
    for ent, v in agg.items():
        out[ent] = sum(a for a, _ in v) / len(v)
        detail[ent] = {"traffic": out[ent], "ncu_us": sum(b for _, b in v) / len(v), "launches_averaged": len(v)}
    if "pm_read_bwd.ds" in out and "pm_read_bwd.dx" in out:
        out["pm_read_bwd"] = out["pm_read_bwd.ds"] + out["pm_read_bwd.dx"]
    for alias, ent in (("pm_read_fwd_planes", "pm_read_fwd"), ("pm_read_bwd_planes", "pm_read_bwd")):
        if ent in out:
            out[alias] = out[ent]
    print(json.dumps({dtype: out, "_detail_" + dtype: detail}, indent=1))


def raw(path):
    rows = list(csv.reader(open(path)))
    hdr, units, data = rows[0], rows[1], rows[2:]
    idx = {h: i for i, h in enumerate(hdr)}
    print("# ncu --set full --clock-control none, one launch per kernel")
    for d in data:
        print("== " + d[idx["Kernel Name"]][:110])
        for w in WANT:
            if w in idx:
                print("   %-66s %16s %s" % (w, d[idx[w]][:16], units[idx[w]]))


if __name__ == "__main__":
    {"launches": launches, "raw": raw, "traffic": traffic}[sys.argv[1]](*sys.argv[2:])

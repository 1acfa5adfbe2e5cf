#!/usr/bin/env python
"""Turns ncu artefacts under gpurun_out/ into the small tracked summaries under profiles/.

    python scripts/summarize_profiles.py launches gpurun_out/launches_r01.csv profiles/r01_launches.txt
    python scripts/summarize_profiles.py full gpurun_out/prof.ncu-rep profiles/r01_kernel_full.txt
    python scripts/summarize_profiles.py traffic profiles/r02_traffic.json        (from the round-2 .ncu-rep files)
"""
import collections
import csv
import subprocess
import sys

KEYS = [
    "gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum", "launch__grid_size",
    "launch__block_size", "launch__registers_per_thread", "launch__shared_mem_per_block_dynamic",
    "launch__occupancy_limit_registers", "launch__occupancy_limit_shared_mem",
    "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
    "smsp__inst_executed.sum", "sm__throughput.avg.pct_of_peak_sustained_elapsed",
    "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
    "sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active",
    "sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active",
    "sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active",
    "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
    "sm__inst_executed_pipe_tc.avg.pct_of_peak_sustained_active",
    "l1tex__data_pipe_lsu_wavefronts.avg.pct_of_peak_sustained_elapsed",
    "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum", "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum",
    "lts__t_sectors_op_read.sum", "lts__t_sectors_op_write.sum",
]


def launches(src, dst):
    rows = [r for r in csv.reader(open(src, errors="replace")) if len(r) > 14 and r[0].isdigit()]
    per = collections.OrderedDict()
    order = []
    for r in rows:
        name, val, unit = r[4], float(r[14]), r[13]
        scale = {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6}.get(unit, 1.0)
        short = name.split("(")[0].replace("void ", "")[:90]
        order.append((short, val * scale))
        c = per.setdefault(short, [0, 0.0])
        c[0] += 1
        c[1] += val * scale
    tot = sum(v[1] for v in per.values())
    with open(dst, "w") as f:
        f.write(f"# ncu --metrics gpu__time_duration.sum --clock-control none  ({src})\n")
        f.write("# per-launch times are cold-cache and serialised: compare SHARES, not absolutes\n")
        f.write(f"# {len(order)} launches, {tot:.1f} us total\n\n")
        f.write(f"{'kernel':92s} {'launches':>8s} {'total_us':>12s} {'share':>7s}\n")
        for k, (n, t) in sorted(per.items(), key=lambda kv: -kv[1][1]):
            f.write(f"{k:92s} {n:8d} {t:12.1f} {100 * t / tot:6.1f}%\n")
        f.write("\n# launch order\n")
        for k, t in order:
            f.write(f"{t:12.1f} us  {k}\n")


def full(src, dst):
    out = subprocess.run(["ncu", "-i", src, "--page", "raw", "--csv"], stdout=subprocess.PIPE, text=True).stdout
    rows = list(csv.reader(out.splitlines()))
    hdr, units = rows[0], rows[1]
    with open(dst, "w") as f:
        f.write(f"# ncu --set full --clock-control none ({src})\n")
        for vals in rows[2:]:
            d = dict(zip(hdr, zip(vals, units)))
            f.write(f"\nkernel: {d['Kernel Name'][0]}\n")
            for k in KEYS:
                if k in d:
                    f.write(f"  {k:70s} {d[k][0]:>18s} {d[k][1]}\n")
            for k in hdr:
                if k.startswith("smsp__average_warps_issue_stalled") and k.endswith("per_issue_active.ratio"):
                    f.write(f"  {k:70s} {d[k][0]:>18s}\n")


def _raw(src):
    out = subprocess.run(["ncu", "-i", src, "--page", "raw", "--csv"], stdout=subprocess.PIPE, text=True).stdout
    rows = list(csv.reader(out.splitlines()))
    hdr, units = rows[0], rows[1]
    res = []
    for vals in rows[2:]:
        d = dict(zip(hdr, zip(vals, units)))

        def num(key, to):
            v, u = d[key]
            x = float(v.replace(",", ""))
            scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6,
                     "%": 1.0}.get(u, 1.0)
            return x * scale
        res.append({"kernel": d["Kernel Name"][0][:60],
                    "dram_bytes": num("dram__bytes_read.sum", "byte") + num("dram__bytes_write.sum", "byte"),
                    "us": num("gpu__time_duration.sum", "us"),
                    "tensor_pct": num("sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "%")})
    return res


def traffic(dst, *_):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the dominant kernels, from the ncu --set full
    captures of the bench commands; bench.py reads this file for roofline.traffic."""
    import json
    out = {}
    fe = _raw("gpurun_out/prof_fe_r02.ncu-rep")[0]
    out["frontend"] = {"kernel": fe["kernel"], "dram_bytes_per_launch": fe["dram_bytes"], "gpu_time_us": fe["us"],
                       "source": "gpurun_out/prof_fe_r02.ncu-rep -> profiles/r02_frontend_ncu.txt (bench.py --workload "
                                 "frontend, 1024 x 10 s)"}
    pl = _raw("gpurun_out/prof_plda_r02.ncu-rep")[0]
    out["plda_score"] = {"kernel": pl["kernel"], "dram_bytes_per_launch": pl["dram_bytes"], "gpu_time_us": pl["us"],
                         "source": "gpurun_out/prof_plda_r02.ncu-rep -> profiles/r02_plda_score_ncu.txt (bench.py "
                                   "--workload plda, first score GEMM of the step)"}
    st = _raw("gpurun_out/prof_w2x_stack_r02.ncu-rep")
    seen, per = set(), []
    for k in st:                      # (ncu lists a kernel once per replayed section set: keep the first of each launch)
        key = (k["kernel"], round(k["us"], 3))
        if key in seen:
            continue
        seen.add(key)
        per.append(k)
    out["tdnn_stack"] = {"kernel": "gather_cmvn_splice_kernel + tdnn_tc_pair_kernel x5 + tdnn_tc_stats_kernel (one "
                                   "wav2xvec step)",
                         "dram_bytes_per_launch": sum(k["dram_bytes"] for k in per),
                         "gpu_time_us": sum(k["us"] for k in per), "per_kernel": per,
                         "source": "gpurun_out/prof_w2x_stack_r02.ncu-rep -> profiles/r02_wav2xvec_stack_ncu.txt (bench.py "
                                   "default workload, 7 consecutive launches of one step)"}
    with open(dst, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    {"launches": launches, "full": full, "traffic": traffic}[sys.argv[1]](*sys.argv[2:])

#!/usr/bin/env python
"""Turns the scratch captures of tools/profile_round2.sh (gpurun_out/r02_*) into the committed evidence under profiles/:
ncu summaries (tools/ncu_summary.py), per-source-line hot spots (tools/ncu_lines.py), launch-list summaries, bench lines, and
profiles/k3_traffic.json (the per-launch DRAM bytes / L2->L1 sectors bench.py quotes next to its live kernel time)."""
import csv, json, os, shutil, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G, P = os.path.join(ROOT, "gpurun_out"), os.path.join(ROOT, "profiles")
LIB = os.path.join(ROOT, "physimglobalpose_b200", "libpgp.so")


def run(cmd):
    return subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT).stdout


def raw_metrics(rep):
    rows = list(csv.reader(run(["ncu", "-i", rep, "--page", "raw", "--csv"]).splitlines()))
    return dict(zip(rows[0], rows[2]))


KERNELS = {"r02_k3": "k3_fine_kernelILb1ELi0E", "r02_k3w": "k3_fine_kernelILb0ELi1E", "r02_k2_query": "k2_join_queryILb0", "r02_k2_select": "k2_join_select",
           "r02_k2s_bases": "k2s_select_basesENS", "r02_k5": "k5_tricp_kernel"}
traffic = {}
for name, mangled in KERNELS.items():
    rep = os.path.join(G, name + ".ncu-rep")
    if not os.path.exists(rep):
        continue
    out = run([sys.executable, "tools/ncu_summary.py", rep])
    lines = run([sys.executable, "tools/ncu_lines.py", rep, LIB, mangled, "40"])
    if name in ("r02_k3", "r02_k3w"):
        env = dict(os.environ, NCU_LINES_MEM="1")
        lines += "\n---- per source line by memory traffic (gsect = L2 sectors requested by global loads, shwave = shared-memory wavefronts, lsect = local-memory sectors)\n" + \
            subprocess.run([sys.executable, "tools/ncu_lines.py", rep, LIB, mangled, "24"], capture_output=True, text=True, cwd=ROOT, env=env).stdout
    open(os.path.join(P, name + "_ncu_full_summary.txt"), "w").write(out + "\n---- per source line (tools/ncu_lines.py; inst = share of warp instructions, lanes = active threads per instruction, stall = share of stall samples)\n" + lines)
    if name in ("r02_k3", "r02_k3w"):
        m = raw_metrics(rep)
        f = lambda k: float(m[k].replace(",", ""))
        units_row = list(csv.reader(run(["ncu", "-i", rep, "--page", "raw", "--csv"]).splitlines()))[1]
        unit = lambda k: {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1, "ms": 1.0, "us": 1e-3, "usecond": 1e-3, "msecond": 1.0, "second": 1e3, "ns": 1e-6, "nsecond": 1e-6}[units_row[list(m).index(k)]]
        traffic["c2" if name == "r02_k3" else "c2w"] = {
            "kernel": m["Kernel Name"], "source": f"profiles/{name}_ncu_full_summary.txt (ncu --set full --clock-control none, one launch, C2 inputs via tools/run_mode.py; tools/profile_round2.sh)",
            "dram_bytes_read": int(f("dram__bytes_read.sum") * unit("dram__bytes_read.sum")), "dram_bytes_write": int(f("dram__bytes_write.sum") * unit("dram__bytes_write.sum")),
            "l2_to_l1_sectors": int(f("lts__t_sectors_srcunit_tex_op_read.sum")), "l1_global_load_sectors": int(f("l1tex__t_sectors_pipe_lsu_mem_global_op_ld.sum")),
            "issue_active_pct": f("smsp__issue_active.avg.pct_of_peak_sustained_active"), "l1tex_throughput_pct": f("l1tex__throughput.avg.pct_of_peak_sustained_active"),
            "l2_throughput_pct": f("lts__throughput.avg.pct_of_peak_sustained_elapsed"), "dram_throughput_pct": f("gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed"),
            "warp_instructions": int(f("smsp__inst_executed.sum")), "kernel_ms_under_ncu": f("gpu__time_duration.sum") * unit("gpu__time_duration.sum")}
if traffic:
    json.dump(traffic, open(os.path.join(P, "k3_traffic.json"), "w"), indent=1)
for name in ("r02_launches", "r02_k2_launches_m0", "r02_k2_launches_m1"):
    src = os.path.join(G, name + ".csv")
    if os.path.exists(src):
        shutil.copy(src, os.path.join(P, name + ".csv"))
        open(os.path.join(P, name + "_summary.txt"), "w").write(run([sys.executable, "tools/launch_summary.py", src]))
for f in sorted(os.listdir(G)):
    if f.startswith("r02_bench") and f.endswith(".json") and os.path.getsize(os.path.join(G, f)) > 10 and not any(c in f for c in ("_a.", "_b.", "_c.", "_d.")):
        shutil.copy(os.path.join(G, f), os.path.join(P, f))
for f in ("r02_c1_latency.json", "r02_gen_m0.log", "r02_gen_m1_100.log", "r02_gen_m1_13000.log", "r02_tricp.log"):
    if os.path.exists(os.path.join(G, f)):
        shutil.copy(os.path.join(G, f), os.path.join(P, f))
print("profiles/ updated:", sorted(x for x in os.listdir(P) if x.startswith("r02") or x == "k3_traffic.json"))

"""Turns gpurun_out/{launches.csv,*.ncu-rep} into the text summaries committed under profiles/ (run in the build
container; ncu reads the reports without a GPU)."""
import collections
import csv
import subprocess
import sys

TAG = sys.argv[1] if len(sys.argv) > 1 else "r01"
# the scoring workload of the captures: the bench bank with its neighbour table, four batches of 16 images
SCORE_RUN = ('python -c "import bench, torch; b = bench.build_bank(0, bench.BANK_ROWS, 0); b.finalize(); b.build_knn(); '
             'p = torch.stack(bench.test_patches(16)).cuda(); [b.score_batch(p, (28, 28), 224) for _ in range(4)]"')
KEYS = ["gpu__time_duration.sum", "sm__cycles_elapsed.max.per_second", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "dram__bytes_read.sum.per_second", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "lts__t_sector_hit_rate.pct",
        "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active", "sm__throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__inst_executed.sum.per_cycle_active", "smsp__inst_executed.sum", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "launch__registers_per_thread", "launch__grid_size",
        "launch__block_size", "launch__shared_mem_per_block_dynamic",
        "smsp__average_warps_issue_stalled_long_scoreboard_per_issue_active.ratio",
        "smsp__average_warps_issue_stalled_barrier_per_issue_active.ratio",
        "smsp__average_warps_issue_stalled_wait_per_issue_active.ratio",
        "smsp__average_warps_issue_stalled_math_pipe_throttle_per_issue_active.ratio",
        "smsp__average_warps_issue_stalled_short_scoreboard_per_issue_active.ratio"]


def launches(path, out, cmd):
    rows = list(csv.reader(open(path)))
    hi = [i for i, r in enumerate(rows) if "Kernel Name" in r][0]
    hdr = rows[hi]
    k, v = hdr.index("Kernel Name"), hdr.index("Metric Value")
    agg = collections.OrderedDict()
    for r in rows[hi + 1:]:
        if len(r) <= v:
            continue
        name = r[k].split("(")[0][:64]
        a = agg.setdefault(name, [0, 0.0])
        a[0] += 1
        a[1] += float(r[v].replace(",", ""))
    tot = sum(a[1] for a in agg.values())
    with open(out, "w") as f:
        f.write(f"# {cmd}\n# per-launch device times are cold-cache and serialised by ncu: compare SHARES, not absolutes\n")
        for n, (c, t) in sorted(agg.items(), key=lambda x: -x[1][1]):
            f.write(f"{n:66s} n={c:4d} avg={t / c / 1e3:12.2f} us total={t / 1e6:10.3f} ms share={t / tot * 100:5.1f}%\n")


def full(rep, out, title):
    txt = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(txt.splitlines()))
    hdr, units, vals = rows[0], rows[1], rows[2]
    with open(out, "w") as f:
        f.write(f"# {title}\n# kernel: {vals[hdr.index('Kernel Name')]}\n")
        for i, h in enumerate(hdr):
            if h in KEYS:
                f.write(f"{h:92s} {units[i]:16s} {vals[i]}\n")
    return {h: (units[i], vals[i]) for i, h in enumerate(hdr)}


def to_bytes(unit, val):
    scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[unit]
    return float(val.replace(",", "")) * scale


def gemm_traffic(metrics, images, source, out="profiles/gemm_traffic.json"):
    """bench.py reads roofline.traffic from this file: dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the
    dominant kernel, from the ncu --set full capture named in `source`"""
    import json
    rd = to_bytes(*metrics["dram__bytes_read.sum"])
    wr = to_bytes(*metrics["dram__bytes_write.sum"])
    json.dump({"kernel": metrics["Kernel Name"][1], "images_per_launch": images, "dram_bytes_read": rd, "dram_bytes_write": wr,
               "duration_ms_under_ncu": to_bytes("byte", metrics["gpu__time_duration.sum"][1]) * {"ms": 1, "us": 1e-3, "ns": 1e-6, "s": 1e3}[metrics["gpu__time_duration.sum"][0]],
               "source": source}, open(out, "w"), indent=1)


if __name__ == "__main__":
    import os
    g = "gpurun_out"
    if os.path.exists(f"{g}/launches.csv"):
        launches(f"{g}/launches.csv", f"profiles/{TAG}_launches_bench.txt",
                 "ncu --metrics gpu__time_duration.sum --clock-control none -c 2500 python bench.py --steps 2 --warmup 3 --skip-cpu "
                 "--skip-extras --skip-dropin")
    cap = "ncu --set full --clock-control none --import-source on -k regex:%s -s 1 -c 1 " + SCORE_RUN
    for rep, out, title in (
            ("prof_score_gemm", "prof_gemm", "score_gemm_kernel<1,2,1>, batch of 16 images x 784 patches vs 200k x 768 bank"),
            ("prof_gemm", "prof_gemm", "score_gemm_kernel<1,2,1>, batch of 16 images x 784 patches vs 200k x 768 bank"),
            ("prof_refine_cert", "prof_refine_cert", "refine_cert_kernel<8>, 12 544 queries x 296 producers, 200k x 768 bank"),
            ("prof_rescan_kernel", "prof_rescan", "rescan_kernel, ~100 (query, producer) pairs of a 16-image batch, 200k x 768 bank"),
            ("prof_upsample_hblur", "prof_hblur", "upsample_hblur_kernel, 16 images 28x28 -> 224x224"),
            ("prof_coreset", "prof_coreset", "coreset_kernel<__half,3>, 200k x 301, 300 picks"),
            ("prof_reweight", "prof_reweight", "reweight_kernel<6>, batch of 16, 200k x 768 bank")):
        if os.path.exists(f"{g}/{rep}.ncu-rep") and not (rep == "prof_gemm" and os.path.exists(f"{g}/prof_score_gemm.ncu-rep")):
            m = full(f"{g}/{rep}.ncu-rep", f"profiles/{TAG}_{out}.txt", (cap % rep[5:]) + " -- " + title)
            if out == "prof_gemm":
                gemm_traffic(m, 16, f"profiles/{TAG}_prof_gemm.txt (gpurun_out/{rep}.ncu-rep: " + (cap % "score_gemm") + ")")

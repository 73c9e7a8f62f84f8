#!/usr/bin/env python
"""Headline benchmark of the memory-bank anomaly-scoring hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1|2|3|4|5] [--dump-outputs DIR]

Default (--config 1, BASELINE cfg 5 headline).  A "step" scores one batch (--batch, default 16) of synthetic 784-patch
images (DINO ViT-B/8 shaped, 768-d) against an un-subsampled 200 000 x 768 float32 bank through the full path: distance
GEMM + min/argmin, s*/m*/top-3 re-weighting, bilinear upsample and Gaussian blur, one result set per image.
  value    patch-NN scores/s with the patches already resident in HBM (device pointer through the C ABI)
  e2e      the same through the C ABI with HOST buffers (pinned patches in, results out), copies inside the timed region
  parity   (outside the timed region) the scored batch against the CPU restatement of the reference at the SAME size;
           N > 1 additionally: row-sharded results == single-GPU results, bit for bit, scoring and coreset
  coreset_select_s    projection + greedy selection of 10 % of the same bank
  predict_batch_e2e   the drop-in API (methods.RGBFeatures.predict_batch: normalisation, scoring, late-fusion head on the device)
  large_bank / configs   the other BASELINE configurations in bounded form (full form: --config 2 / 3 / 4 / 5;
                         3 = the ten classes in sequence, class-parallel over the ranks)
N > 1 (torchrun, one rank per GPU): the bank is row-sharded; every step runs one round of the three-phase sharded
protocol (two small exchanges over peer-mapped memory fused into the kernels) with three rounds outstanding on two compute lanes (strong scaling: the job is still one 200k bank).
`--impl reference` times the CPU restatement of the reference path (oracle/, the one place it may be executed from here)
on ALL host cores, --steps images.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)

BANK_ROWS, DIM, P, FMAP, OUT_HW = 200_000, 768, 784, 28, 224
PIPELINE_DEPTH = 3   # submitted calls outstanding per handle (three result slots, two compute lanes)
METRIC = "patch-NN scores/sec at 200k x 768 bank"
WORKLOAD = ("cfg5 headline: score 784-patch images (28x28x768) against an un-subsampled 200000x768 fp32 bank "
            "(min/argmin + s*/m*/top-3 reweight + bilinear 224^2 + blur); coreset 10% of the same bank reported beside")
GEMM_PROFILE = os.path.join(ROOT, "profiles", "gemm_traffic.json")  # written by scripts/summarize_profiles.py from an ncu capture


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], bf16_tflops=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained"),
                    source="MEASURED_PEAKS.json")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def host_cores():
    """cores this process may run on (the launcher's OMP_NUM_THREADS=1 under torchrun is NOT a core count)"""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu, self.proc, self.lines = gpu, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
            time.sleep(0.3)  # let the sampler come up before the timed region starts
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------------
# synthetic data
# ---------------------------------------------------------------------------------------------------------------------
_HOST_BANK = {}


def host_bank_rows(c0, n):
    """rows [c0, c0 + n) of the headline bank (numpy PCG64 streams in chunks of 25 000 rows: identical on every rank)"""
    from cmdiad_b200 import synth
    cent = synth.centroids(DIM)
    chunk = 25_000
    out = []
    for k in range(c0 // chunk, (c0 + n + chunk - 1) // chunk):
        if k not in _HOST_BANK:
            _HOST_BANK[k] = synth.patches(chunk, DIM, seed=5000 + k, cent=cent)
        a, b = max(c0, k * chunk), min(c0 + n, (k + 1) * chunk)
        out.append(_HOST_BANK[k][a - k * chunk:b - k * chunk])
    return np.concatenate(out, 0)


def build_bank(lo, hi, device):
    from cmdiad_b200 import Bank
    bank = Bank(DIM, hi - lo, device=device, row_offset=lo)
    c0 = lo
    while c0 < hi:
        c1 = min(hi, c0 - c0 % 25_000 + 25_000)
        bank.append(host_bank_rows(c0, c1 - c0))
        c0 = c1
    return bank


def test_patches(n):
    from cmdiad_b200 import synth
    cent = synth.centroids(DIM)
    return [torch.from_numpy(synth.patches(P, DIM, seed=7000 + i, anomalous_frac=0.01, cent=cent)) for i in range(n)]


def device_patches(rows, dim, seed, device, k=2048, anomalous_frac=0.0):
    """clustered synthetic rows generated ON the device (the large configurations: 1M x 1920 would take minutes with
    numpy).  Same recipe as cmdiad_b200.synth ("C": centroid + 0.35 N(0,1)), torch's Philox streams."""
    g = torch.Generator(device=device)
    g.manual_seed(int(seed))
    gc = torch.Generator(device=device)
    gc.manual_seed(10_000 + dim)
    cent = torch.randn((k, dim), generator=gc, device=device)
    out = torch.empty((rows, dim), device=device)
    for r0 in range(0, rows, 100_000):
        n = min(100_000, rows - r0)
        j = torch.randint(0, k, (n,), generator=g, device=device)
        noise = torch.randn((n, dim), generator=g, device=device)
        scale = torch.full((n, 1), 0.35, device=device)
        if anomalous_frac > 0:
            scale[torch.rand((n, 1), generator=g, device=device) < anomalous_frac] = 3.0
        out[r0:r0 + n] = cent[j] + scale * noise
    return out


def sparse_csr(n_rows, dim, seed=0):
    from sklearn import random_projection
    tr = random_projection.SparseRandomProjection(eps=0.9, random_state=seed)
    tr.fit(np.broadcast_to(np.zeros((1, 1)), (n_rows, dim)))
    c = tr.components_
    return (c.indptr, c.indices, c.data, c.shape[0])


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline
# ---------------------------------------------------------------------------------------------------------------------
def cpu_reference_leg(steps, warmup, threads=None):
    """reference path restated on the CPU (oracle/restate.py: torch.cdist + min + topk + interpolate + PIL-exact blur);
    one step = one image against the full bank.  threads: torch intra-op threads, set EXPLICITLY (torch.distributed.run
    exports OMP_NUM_THREADS=1, which would otherwise silently turn this into a 1-core baseline); None = all host cores"""
    from oracle import restate as O
    threads = threads or host_cores()
    prev = torch.get_num_threads()
    torch.set_num_threads(threads)
    try:
        lib = torch.from_numpy(host_bank_rows(0, BANK_ROWS))
        patches = test_patches(max(1, min(4, steps + warmup)))
        for i in range(warmup):
            O.score_restated(patches[i % len(patches)], lib, (FMAP, FMAP), OUT_HW)
        t0 = time.perf_counter()
        for i in range(steps):
            O.score_restated(patches[i % len(patches)], lib, (FMAP, FMAP), OUT_HW)
        dt = time.perf_counter() - t0
    finally:
        torch.set_num_threads(prev)
    return P * steps / dt, dt / steps * 1e3, threads


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # one step = one 784-patch image on the host cores (~0.3 s on 16 cores).  value = ALL host cores at every N; the
    # reference's own default of 6 threads (main.py:149 --cpu_core_num) is timed beside it over the same step count.
    steps = args.steps
    warm = args.warmup
    val, ms, cores = cpu_reference_leg(steps, warm)
    val6, ms6, _ = cpu_reference_leg(steps, 1, threads=min(6, cores))
    line = {"metric": METRIC, "value": val, "unit": "patch-NN scores/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "bank_rows": BANK_ROWS, "dim": DIM, "patches_per_image": P,
                       "images_per_step": 1},
            "cpu_baseline": {"value": val, "unit": "patch-NN scores/s", "cores": cores, "kind": "port",
                             "sample": f"{steps} images x {P} patches against the full {BANK_ROWS}x{DIM} bank, "
                                       f"torch.set_num_threads({cores}) (all host cores; OMP_NUM_THREADS ignored)",
                             "reference_default_threads": {"cores": min(6, cores), "value": val6, "ms_per_image": ms6,
                                                           "note": "main.py:149 --cpu_core_num 6"}},
            "e2e": {"value": val, "unit": "patch-NN scores/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# parity (outside every timed region)
# ---------------------------------------------------------------------------------------------------------------------
def lsb_histogram(mine, ref):
    """post-blur map differences in units of the reference map's 8-bit quantisation step (max / 255)"""
    lsb = float(ref.max()) / 255.0
    d = np.abs(mine.astype(np.float64) - ref.astype(np.float64)) / lsb
    steps = np.rint(d).astype(np.int64)
    return {"pixels": int(d.size), "eq_bits": int((mine == ref).sum()), "ge_1_lsb": int((steps >= 1).sum()),
            "ge_2_lsb": int((steps >= 2).sum()), "ge_3_lsb": int((steps >= 3).sum()), "max_lsb": float(d.max())}


def _rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-30)))


def parity_vs_oracle(results, patches_host, n_images=2, exact_bank=None):
    """our results of the first n_images of a scored batch against oracle.score_restated on the SAME 200k x 768 bank.
    exact_bank: an un-sharded Bank of the same rows -- additionally compares min_val / min_idx bit for bit with the exact
    float32 scan of the whole bank on the device (the arithmetic of the re-check kernels; test hook cmdb_debug_exact_min),
    which separates our error from the float32 noise of the host's mm-form cdist."""
    from oracle import restate as O
    from tests.cases import tie_aware_idx_ok
    prev = torch.get_num_threads()
    torch.set_num_threads(host_cores())
    try:
        lib = torch.from_numpy(host_bank_rows(0, BANK_ROWS))
        out = {"images": n_images, "bank_rows": BANK_ROWS, "checker": "oracle.restate.score_restated (torch.cdist mm-form on the host)",
               "min_idx_strict_mismatch": 0, "min_idx_tie_aware_ok": True, "min_val_max_rel": 0.0, "s_max_rel": 0.0,
               "s_star_max_rel": 0.0, "s_idx_equal": True, "nn_idx_set_equal": True, "pre_blur_max_rel": 0.0,
               "u8_image_pixels_differing": 0, "blur_given_same_u8_bit_exact": True,
               "post_blur": {"pixels": 0, "eq_bits": 0, "ge_1_lsb": 0, "ge_2_lsb": 0, "ge_3_lsb": 0, "max_lsb": 0.0}}
        for i in range(n_images):
            r = results[i]
            ref = O.score_restated(patches_host[i], lib, (FMAP, FMAP), OUT_HW)
            ok, nbad = tie_aware_idx_ok(r.min_idx, ref["min_idx"], ref["dist"].numpy())
            out["min_idx_strict_mismatch"] += int(nbad)
            out["min_idx_tie_aware_ok"] &= bool(ok)
            rel_p = np.abs(r.min_val.astype(np.float64) - ref["min_val"]) / ref["min_val"]
            if float(rel_p.max()) > out["min_val_max_rel"]:
                w = int(rel_p.argmax())
                out["min_val_worst"] = {"image": i, "patch": w, "ours": float(r.min_val[w]), "oracle": float(ref["min_val"][w]),
                                        "row": int(r.min_idx[w]), "oracle_row": int(ref["min_idx"][w])}
            if exact_bank is not None:
                ex_val, ex_idx = np.empty(P, np.float32), np.empty(P, np.int64)
                q = np.ascontiguousarray(patches_host[i].numpy())
                rc = exact_bank._lib.cmdb_debug_exact_min(exact_bank._h, q.ctypes.data, P, ex_val.ctypes.data, ex_idx.ctypes.data)
                out["equals_exact_device_scan"] = bool(out.get("equals_exact_device_scan", True) and rc == 0
                                                       and (ex_val == r.min_val).all() and (ex_idx == r.min_idx).all())
                out["oracle_vs_exact_scan_max_rel"] = max(out.get("oracle_vs_exact_scan_max_rel", 0.0), _rel(ref["min_val"], ex_val))
            out["min_val_max_rel"] = max(out["min_val_max_rel"], _rel(r.min_val, ref["min_val"]))
            out["s_max_rel"] = max(out["s_max_rel"], _rel(r.s[0], ref["s"]))
            out["s_star_max_rel"] = max(out["s_star_max_rel"], _rel(r.s_star[0], ref["s_star"]))
            out["s_idx_equal"] &= int(r.s_idx[0]) == ref["s_idx"]
            out["nn_idx_set_equal"] &= (set(r.nn_idx[1:].tolist()) == set(ref["nn_idx"][1:].tolist())
                                        and int(r.nn_idx[0]) == int(ref["nn_idx"][0]))
            out["pre_blur_max_rel"] = max(out["pre_blur_max_rel"], _rel(r.s_map_pre, ref["s_map_pre"]))
            out["u8_image_pixels_differing"] += int((r.s_map_u8 != ref["s_map_u8"]).sum())
            mine_blur, _ = O.knn_blur_restated(r.s_map_pre)
            out["blur_given_same_u8_bit_exact"] &= bool((mine_blur == r.s_map).all())
            h = lsb_histogram(r.s_map, ref["s_map"])
            for k, v in h.items():
                out["post_blur"][k] = max(out["post_blur"][k], v) if k == "max_lsb" else out["post_blur"][k] + v
        pb = out["post_blur"]
        pb["frac_ge_1_lsb"] = pb["ge_1_lsb"] / max(1, pb["pixels"])
        out["within_contract"] = bool(out["min_idx_tie_aware_ok"] and out["min_val_max_rel"] <= 1e-4 and out["s_max_rel"] <= 1e-4
                                      and out["pre_blur_max_rel"] <= 1e-4 and out["s_idx_equal"] and out["nn_idx_set_equal"]
                                      and out["blur_given_same_u8_bit_exact"])
    finally:
        torch.set_num_threads(prev)
    return out


def results_equal(a, b, names=("min_idx", "min_val", "s", "s_star", "s_idx", "nn_idx", "m_star_knn", "w", "s_map")):
    return all(bool((getattr(a, n) == getattr(b, n)).all()) for n in names)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, result):
    """Writes every array of a BatchResult (what the caller of score_batch_async receives) as <directory>/<name>.npy, so
    that two builds run with the same arguments can be compared output for output.  float32 arrays are written as they
    are; integer arrays (indices) as float64, which holds them exactly.  Every array is indexed by image first; when
    the batch would exceed DUMP_LIMIT_BYTES, a fixed seeded sample of the images is written.  image_index.npy lists the
    images written."""
    arrays = {n: np.asarray(a) for n, a in result.arrays.items() if a is not None}
    arrays = {n: a if a.dtype == np.float32 else a.astype(np.float64) for n, a in arrays.items()}
    n_img = len(result)
    per_image = sum(a.nbytes for a in arrays.values()) // n_img + 8
    keep = np.arange(n_img)
    if n_img * per_image > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n_img, DUMP_LIMIT_BYTES // per_image, replace=False))
        arrays = {n: a[keep] for n, a in arrays.items()}
    arrays["image_index"] = keep.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


# ---------------------------------------------------------------------------------------------------------------------
# the other BASELINE configurations (bounded forms inside the default run, full forms behind --config)
# ---------------------------------------------------------------------------------------------------------------------
def event_time(stream, fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    w0 = time.perf_counter()
    out = fn()
    e1.record(stream)
    e1.synchronize()
    return out, max(e0.elapsed_time(e1) * 1e-3, time.perf_counter() - w0)


def coreset_point(bank, n_total, n_sel, csr, comm=None, mode=None):
    """one timed coreset selection on `bank` (whole call: projection + greedy loop; the caller takes the max over ranks)"""
    from cmdiad_b200 import _lib as L
    mode = L.CORESET_FP16 if mode is None else mode
    run = (lambda n: bank.coreset_select(n, csr, mode)) if comm is None else \
        (lambda n: bank.coreset_select_sharded(comm, n_total, n, csr, mode))
    run(min(64, n_sel))
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    idx = run(n_sel)
    torch.cuda.synchronize()
    return idx, time.perf_counter() - t0


def coreset_report(n_total, d_proj, n_sel, seconds, pk, world, elem_bytes=2):
    byts = (n_sel - 1) * float(n_total) * d_proj * elem_bytes
    return {"rows": n_total, "d_proj": d_proj, "picks": n_sel, "seconds": seconds, "us_per_pick": seconds / max(1, n_sel - 1) * 1e6,
            "achieved_gbs": byts / seconds / 1e9, "frac_of_hbm": byts / seconds / 1e9 / (pk["hbm_gbs"] * world)}


def large_bank_leg(rank, world, local, pk, steps, rows=1_000_000, picks=10_000, comm=None):
    """BASELINE cfg 5, the regime where row-sharding is meant to pay (SURVEY 8e): a `rows` x 768 bank generated on the
    device, row-sharded over the ranks; scoring of 16-image batches and a bounded coreset selection (FP16 mode)."""
    import torch.distributed as dist
    from cmdiad_b200 import Bank
    dev = torch.device("cuda", local)
    lo, hi = rows * rank // world, rows * (rank + 1) // world
    bank = Bank(DIM, hi - lo, device=local, row_offset=lo)
    c0 = lo
    while c0 < hi:  # global rows in chunks of 100k with their own seeds: identical whatever the world size
        c1 = min(hi, c0 - c0 % 100_000 + 100_000)
        chunk = device_patches(100_000, DIM, 9000 + c0 // 100_000, dev)
        bank.append(chunk[c0 % 100_000:c0 % 100_000 + (c1 - c0)])
        c0 = c1
    del chunk
    csr = sparse_csr(rows, DIM)
    idx, cs = coreset_point(bank, rows, picks, csr, comm)
    t = torch.tensor([cs], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    out = {"rows": rows, "coreset": coreset_report(rows, csr[3], picks, float(t), pk, world)}
    out["coreset"]["idx_checksum"] = int(np.bitwise_xor.reduce(idx * np.arange(1, len(idx) + 1)))
    bank.finalize()
    t0 = time.perf_counter()
    if world > 1:
        bank.build_knn_sharded()
        bank.attach_comm(comm)
    else:
        bank.build_knn()
    torch.cuda.synchronize()
    out["knn_table_build_s"] = time.perf_counter() - t0
    B = 16
    imgs = device_patches(B * P, DIM, 9900, dev, anomalous_frac=0.01).view(B, P, DIM)
    st = bank.stream()

    def run(k):
        pending = []   # up to PIPELINE_DEPTH calls outstanding: the host never gates the next distance GEMM
        for _ in range(k):
            pending.append(bank.score_sharded_async(imgs, (FMAP, FMAP), OUT_HW, distribute=True) if world > 1 else
                           bank.score_batch_async(imgs, (FMAP, FMAP), OUT_HW))
            if len(pending) >= PIPELINE_DEPTH:
                pending.pop(0).wait()
        while len(pending) > 1:
            pending.pop(0).wait()
        return pending.pop(0).wait()

    run(3)
    if world > 1:
        dist.barrier()
    res, sec = event_time(st, lambda: run(steps))
    t = torch.tensor([sec], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t)
    flop = 2.0 * B * P * rows * DIM * steps
    out["scoring"] = {"images_per_step": B, "value": B * P * steps / sec, "unit": "patch-NN scores/s",
                      "ms_per_step": sec / steps * 1e3, "tflops_algorithmic": flop / sec / 1e12,
                      "frac_of_bf16_peak": flop / sec / 1e12 / (pk["bf16_tflops"] * world),
                      "s_checksum": float(np.sum(res.arrays["s"]))}
    bank.close()
    return out


def dual_bank_leg(local, pk, n_img=200, score_images=16, seed_base=0):
    """BASELINE cfg 2: DINO + Point-MAE dual bank -- XYZ 200 x 3136 x 1152 (627 200 rows, d' = 329, n = 62 720) and RGB
    200 x 784 x 768 (156 800 rows, n = 15 680), 10 % coreset each (multiple_features.py:873-895), then scoring of
    `score_images` test images against both coresets through the device-side late-fusion head (:967-994)."""
    from cmdiad_b200 import Bank
    from cmdiad_b200.fusion import LateFusion
    dev = torch.device("cuda", local)
    out = {}
    banks = {}
    for name, Pm, D, seed in (("xyz", 3136, 1152, 21 + seed_base), ("rgb", 784, 768, 22 + seed_base)):
        rows = n_img * Pm
        b = Bank(D, rows, device=local)
        for r0 in range(0, rows, 100_000):
            b.append(device_patches(min(100_000, rows - r0), D, seed * 100 + r0 // 100_000, dev))
        mean, std, _, _ = b.stats()
        b.normalize(mean, std)
        csr = sparse_csr(rows, D)
        n_sel = rows // 10
        idx, cs = coreset_point(b, rows, n_sel, csr)
        out[f"coreset_{name}"] = coreset_report(rows, csr[3], n_sel, cs, pk, 1)
        b.gather(idx)
        b.finalize()
        t0 = time.perf_counter()
        b.build_knn()
        torch.cuda.synchronize()
        out[f"coreset_{name}"]["knn_table_build_s"] = time.perf_counter() - t0
        b.set_query_norm(mean, std, True)
        banks[name] = (b, Pm, D, seed)
    out["coreset_select_s"] = out["coreset_xyz"]["seconds"] + out["coreset_rgb"]["seconds"]
    fus = LateFusion([banks["xyz"][0], banks["rgb"][0]], [1.0, 0.1], [1.0, 0.1], [0.8, 0.9], [2.0], [0.7, 1.1], [3.0])
    q = [device_patches(score_images * Pm, D, seed * 100 + 77, dev, anomalous_frac=0.01).view(score_images, Pm, D)
         for (_, Pm, D, seed) in (banks["xyz"], banks["rgb"])]
    dims = [(56, 56), (28, 28)]
    fus.score_batch(q, dims, OUT_HW)
    st = banks["xyz"][0].stream()
    n_rep = 5
    _, sec = event_time(st, lambda: [fus.score_batch(q, dims, OUT_HW) for _ in range(n_rep)][-1])
    n_scores = score_images * (3136 + 784) * n_rep
    flop = 2.0 * score_images * n_rep * (3136 * 62720 * 1152 + 784 * 15680 * 768)
    out["scoring"] = {"images_per_step": score_images, "ms_per_step": sec / n_rep * 1e3, "value": n_scores / sec,
                      "unit": "patch-NN scores/s (3136 xyz + 784 rgb per image, fused late-fusion head on the device)",
                      "tflops_algorithmic": flop / sec / 1e12}
    for b, *_ in banks.values():
        b.close()
    return out


def ten_class_leg(rank, world, local, pk, n_classes=10):
    """BASELINE cfg 3: the 10 MVTec-3D-shaped classes, one synthetic dual bank each (the cfg 2 pipeline: 10 % coreset of the
    XYZ and RGB banks, neighbour tables, scoring through the late-fusion head), handled in sequence as cmdiad_runner.py does
    per class.  Classes are independent objects: with N GPUs class c runs on rank c % N, no collective on the data path."""
    import torch.distributed as dist
    dev = torch.device("cuda", local)
    mine = [c for c in range(n_classes) if c % world == rank]
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    per_class = {}
    for c in mine:
        tc = time.perf_counter()
        r = dual_bank_leg(local, pk, seed_base=40 * (c + 1))
        torch.cuda.synchronize()
        per_class[c] = {"rank": rank, "coreset_select_s": r["coreset_select_s"], "us_per_pick_xyz": r["coreset_xyz"]["us_per_pick"],
                        "us_per_pick_rgb": r["coreset_rgb"]["us_per_pick"], "scoring_value": r["scoring"]["value"],
                        "scoring_ms_per_step": r["scoring"]["ms_per_step"], "class_wall_s": time.perf_counter() - tc}
    wall = time.perf_counter() - t0
    t = torch.tensor([wall], device=dev, dtype=torch.float64)
    gathered = [per_class]
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gathered = [None] * world
        dist.all_gather_object(gathered, per_class)
    allc = {}
    for g in gathered:
        allc.update(g)
    wall = float(t)
    n = len(allc)
    return {"classes": n, "assignment": "class c on rank c % N (independent objects, no data-path collective)",
            "wall_s_all_classes": wall, "classes_per_s": n / wall,
            "coreset_select_s_sum": sum(v["coreset_select_s"] for v in allc.values()),
            "coreset_select_s_mean_per_class": sum(v["coreset_select_s"] for v in allc.values()) / max(1, n),
            "scoring_value_mean_per_gpu": sum(v["scoring_value"] for v in allc.values()) / max(1, n),
            "unit_scoring": "patch-NN scores/s (3136 xyz + 784 rgb per image)",
            "per_class": {str(k): allc[k] for k in sorted(allc)},
            "note": "wall time covers bank generation on the device, statistics, both coresets (627 200 -> 62 720 and 156 800 -> "
                    "15 680 rows), gather, finalize, neighbour tables and 6 scoring steps of 16 images per class"}


def fused_bank_leg(local, pk, fracs=(0.01,), rows=1_000_000, D=1920):
    """BASELINE cfg 4: fused-feature bank 1M x 1920 (d' = 341), coreset sweep"""
    from cmdiad_b200 import Bank
    dev = torch.device("cuda", local)
    b = Bank(D, rows, device=local)
    for r0 in range(0, rows, 100_000):
        b.append(device_patches(100_000, D, 4100 + r0 // 100_000, dev))
    csr = sparse_csr(rows, D)
    out = {"rows": rows, "dim": D, "d_proj": csr[3], "sweep": []}
    for f in fracs:
        n_sel = int(f * rows)
        idx, cs = coreset_point(b, rows, n_sel, csr)
        rep = coreset_report(rows, csr[3], n_sel, cs, pk, 1)
        rep["fraction"] = f
        rep["unique"] = int(len(set(idx.tolist())))
        out["sweep"].append(rep)
    b.close()
    return out


# ---------------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from cmdiad_b200 import Bank
    from cmdiad_b200 import _lib as L
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the results of one GPU: run it without torchrun")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(*vals):
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    pk = peaks()
    lo, hi = BANK_ROWS * rank // world, BANK_ROWS * (rank + 1) // world
    bank = build_bank(lo, hi, local)
    bank.finalize()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    if world == 1:  # SURVEY 8f-1: neighbour table of the bank (one-off, like finalize); the re-weighting is then a lookup
        bank.build_knn()
    else:           # row-sharded: replicated table, built cooperatively (R/world x R distance work per rank)
        bank.build_knn_sharded()
    torch.cuda.synchronize()
    knn_build_s = max_over_ranks(time.perf_counter() - t0)[0]
    comm = None
    if world > 1:
        # peer-mapped buffers (CUDA IPC over NVLink): the sharded rounds exchange through them inside the kernels (no NCCL in
        # the scoring data path); the sharded coreset loop uses the same object
        from cmdiad_b200 import Comm
        comm = Comm(local, d_proj_max=512)
        bank.attach_comm(comm)
    bank.set_timing(world == 1)
    st = bank.stream()
    B = args.batch
    imgs = test_patches(max(B, 16))
    n_img = 3  # distinct batches cycled through
    host = [torch.stack([imgs[(k * 5 + i) % len(imgs)] for i in range(B)]).pin_memory() for k in range(n_img)]
    devb = [p.cuda() for p in host]
    dims = (FMAP, FMAP)

    def submit(patches, **kw):
        if world == 1:
            return bank.score_batch_async(patches, dims, OUT_HW, **kw)
        return bank.score_sharded_async(patches, dims, OUT_HW, distribute=True, **kw)

    def timed(patches, steps, collect_stage=False, pipelined=True):
        """K steps between barriers; device time from CUDA events on the bank's stream, max over ranks.  pipelined: up to
        PIPELINE_DEPTH batches outstanding -- every step still copies its inputs from the host block and its results back inside the timed
        region, the copies just overlap the other batch's kernels.  Also returns the results of the last step."""
        stage_ms = []
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        w0 = time.perf_counter()
        pending = []
        last = None
        for i in range(steps):
            t = submit(patches[i % len(patches)])
            if not pipelined:
                last = t.wait()
                if collect_stage:
                    stage_ms.append(bank.timings())
                continue
            pending.append(t)
            if len(pending) >= PIPELINE_DEPTH:
                pending.pop(0).wait()
        while pending:
            last = pending.pop(0).wait()
        e1.record(st)
        e1.synchronize()
        wall = time.perf_counter() - w0
        barrier()
        ms, wall_ms = max_over_ranks(e0.elapsed_time(e1), wall * 1e3)
        return ms, wall_ms, stage_ms, last

    for i in range(args.warmup):
        submit(devb[i % n_img]).wait()
        submit(host[i % n_img]).wait()
    line = {}
    if world == 1:  # single-image latency of the reference's call pattern, reported beside the batch throughput
        one = devb[0][0].contiguous()
        for _ in range(3):
            bank.score(one, dims, OUT_HW)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(20):
            bank.score(one, dims, OUT_HW)
        single_ms = (time.perf_counter() - t0) / 20 * 1e3
        single_stage = bank.timings()
    # the plain synchronous call, for the per-stage times and as a reference point beside the pipelined numbers
    n_s = max(5, args.steps // 2)
    ms_s, wall_s, stages, _ = timed(devb, n_s, collect_stage=(world == 1), pipelined=False)
    ms_h, wall_h, _, _ = timed(host, n_s, pipelined=False)
    sync_call = {"value": B * P * n_s / (max(ms_s, wall_s) * 1e-3), "e2e": B * P * n_s / (max(ms_h, wall_h) * 1e-3),
                 "unit": "patch-NN scores/s", "note": "one batch / round at a time (the host waits for every batch)"}
    for i in range(3):
        timed(host, 2)
    with ClockSampler(local) as clk:
        ms_dev, wall_dev, _, last = timed(devb, args.steps)
        ms_e2e, wall_e2e, _, _ = timed(host, args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last)
    # results are host-visible when the loop ends, so the event span equals the wall span; report the larger (safer) one
    t_dev, t_e2e = max(ms_dev, wall_dev), max(ms_e2e, wall_e2e)
    value = B * P * args.steps / (t_dev * 1e-3)
    e2e = B * P * args.steps / (t_e2e * 1e-3)
    maps_d2h = -(-B // world) if world > 1 else B  # images whose maps this rank copies back
    line.update({"metric": METRIC, "value": value, "unit": "patch-NN scores/s", "n_gpus": world, "steps": args.steps,
                 "warmup": args.warmup, "ms_per_step": t_dev / args.steps, "higher_is_better": True, "scaling": "strong",
                 "vs_baseline": None,
                 "dtype": "f32 (fp16 tensor-core pre-filter with an error-bound certificate, exact fp32 re-check, FP32-equivalent "
                          "fp16 hi/lo fallback)",
                 "data": "synthetic",
                 "config": {"workload": WORKLOAD, "bank_rows": BANK_ROWS, "dim": DIM, "patches_per_image": P,
                            "images_per_step": B,
                            "call": ("cmdb_score_batch_submit / _wait, three batches outstanding (two compute lanes)" if world == 1 else
                                     "cmdb_score_shard_round_submit + cmdb_score_shard_wait, three rounds outstanding (two compute lanes)"),
                            "sharding": "single GPU" if world == 1 else
                            f"bank row-sharded over {world} GPUs, neighbour table replicated; per step 2 exchanges over peer-mapped "
                            f"memory fused into the kernels (MIN over {B * P} packed int64 keys, SUM over {2 * B} floats; no NCCL call in "
                            f"the scoring path) + the NCCL all-gather of the cooperatively staged host queries (e2e only); map + "
                            f"device->host of image i on rank i % {world}",
                            "l2": "inputs larger than L2: the fp16 bank streams 307 MB per step and the candidate lists 59 MB vs 126 MB of L2"},
                 "e2e": {"value": e2e, "unit": "patch-NN scores/s",
                         "h2d_bytes_per_step": B * P * DIM * 4 // world if world > 1 else B * P * DIM * 4,
                         "d2h_bytes_per_step": maps_d2h * OUT_HW * OUT_HW * 4 + B * (P * 12 + 64),
                         "note": "per rank" if world > 1 else "pinned host block in, results out, inside the timed region"},
                 # kernels per step (N = 1): q_split, GEMM, certificate (takes the tier decision), rescan (publishes its
                 # results), tier-2 chain on the side stream (q_split, GEMM, refine: sized on the device, empty unless very many
                 # certificates fail), select + neighbour-table lookup, 3 map kernels (band maxima, horizontal, vertical) = 12;
                 # sharded round: the same 7 of local_min, push / reduce keys, select, lookup, push / sum of the neighbour
                 # distances, final, 3 map kernels = 17.  Two timed loops (device-resident and host inputs).
                 "gpu_launches": args.steps * 2 * (12 if world == 1 else 17),
                 "clocks": clk.summary(), "sync_call": sync_call})
    flop = 2.0 * B * P * BANK_ROWS * DIM
    if world == 1:
        gemm_ms = float(np.mean([s["gemm"] for s in stages]))
        achieved = flop / (gemm_ms * 1e-3) / 1e12
        stats = bank.score_stats()
        traffic, traffic_src = None, None
        if os.path.exists(GEMM_PROFILE):  # DRAM bytes of one launch from the committed ncu --set full capture of this workload
            gp = json.load(open(GEMM_PROFILE))
            if gp.get("images_per_launch") == B:
                traffic, traffic_src = gp["dram_bytes_read"] + gp["dram_bytes_write"], gp.get("source")
        line["roofline"] = {"bound": "tensor", "achieved": achieved, "peak": pk["bf16_tflops"], "unit": "TFLOP/s",
                            "frac": achieved / pk["bf16_tflops"], "traffic": traffic, "traffic_source": traffic_src,
                            "algorithmic_bytes": BANK_ROWS * DIM * 2 + B * P * DIM * 2 + 2 * 148 * B * P * 16,
                            "algorithmic_bytes_note": "fp16 bank once + fp16 queries once (inputs) + the producers' candidate lists "
                                                      "written once (output of the kernel: 296 x queries x 16 B)",
                            "kernel": "score_gemm_kernel<1,2,1>",
                            "kernel_ms": gemm_ms,
                            "frac_of_sustained": achieved / pk["bf16_sustained"] if pk.get("bf16_sustained") else None,
                            "note": f"algorithmic 2*P*R*D FLOP per launch / CUDA-event time of the kernel on its stream; the "
                                    f"certified pre-filter issues exactly these FLOPs as fp16 tcgen05 MMAs, so peak = dense "
                                    f"16-bit tensor throughput of {pk['source']} (burst, kernel timed alone)"}
        line["prefilter"] = {"mode": stats["mode"], "queries_per_step": stats["queries"],
                             "uncertified_queries_last_step": stats["fallback_queries"],
                             "rescan_pairs_last_step": stats["rescan_pairs"], "gemm_fallback_last_step": stats["gemm_fallback"],
                             "note": "mode 0 = certified hi.hi pre-filter; where the error-bound certificate fails the rows it could not "
                                     "exclude are rescanned exactly (or, for many failures, the queries are redone with the "
                                     "FP32-equivalent 3-term GEMM) inside the same call; results identical to mode 3"}
        line["stage_ms"] = {k: float(np.mean([s[k] for s in stages])) for k in stages[0]}
        line["single_image"] = {"ms_per_image": single_ms, "value": P / (single_ms * 1e-3), "unit": "patch-NN scores/s",
                                "stage_ms": single_stage}
    line["knn_table"] = {"build_s": knn_build_s, "tflops": 2.0 * BANK_ROWS * BANK_ROWS * DIM / knn_build_s / 1e12,
                         "note": "exact 3 nearest rows of every bank row (pre-filter GEMM + certificate + exact re-check), one-off per "
                                 "bank; N > 1: every rank computes the entries of its own rows against the all-gathered bank and the "
                                 "24-byte-per-row table is replicated"}

    # ---- parity, outside the timed regions -------------------------------------------------------------------------
    par = {}
    full_res = submit(host[0], full=True).wait()
    single_r0 = None
    if world > 1:
        # device time of one round at a time (CUDA events on the handle's stream): the peer-memory protocol as timed above, and
        # the NCCL form of the same round (torch.distributed all-reduces between separate phase calls) with its phases
        rounds = []
        for _ in range(5):
            evs = []
            bank.score_sharded_async(devb[0], dims, OUT_HW, distribute=True, phase_events=evs).wait()
            rounds.append(evs[1].elapsed_time(evs[-1]))
        bank.attach_comm(None)
        ph = []
        for _ in range(4):
            evs = []
            bank.score_sharded_async(devb[0], dims, OUT_HW, distribute=True, phase_events=evs).wait()
            ph.append(evs)
        bank.attach_comm(comm)
        torch.cuda.synchronize()
        line["round_ms"] = {"peer_memory_exchange": float(np.median(rounds)),
                            "nccl_exchange": float(np.median([p[1].elapsed_time(p[-1]) for p in ph[1:]]))}
        line["phase_ms_nccl_form"] = {n: float(np.median([p[i].elapsed_time(p[i + 1]) for p in ph[1:]])) for i, n in enumerate(Bank.PHASES)}
        # sharded == single GPU: every rank holds a full replica of the bank for this check and compares the images it owns
        replica = build_bank(0, BANK_ROWS, local)
        replica.finalize()
        replica.build_knn()
        single = replica.score_batch(host[0], dims, OUT_HW, full=True)
        ok = all(results_equal(full_res[i], single[i]) for i in range(B) if full_res[i] is not None)
        sc = bool((full_res.arrays["s"] == single.arrays["s"]).all() and (full_res.arrays["min_idx"] == single.arrays["min_idx"]).all())
        t = torch.tensor([int(ok and sc)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        par["sharded_equals_single"] = bool(int(t))
        par["sharded_check"] = (f"{B} images of one batch: min_idx, min_val, s, s*, s_idx, nn_idx, m_star_knn, w, s_map compared bit for "
                                f"bit on the rank that finished the image, s / min_idx of all images on every rank; single-GPU result "
                                f"from a full replica of the bank on every rank")
        # image-parallel replicas: when the bank fits one GPU, every rank can also score DIFFERENT images against a full
        # replica with no collective at all; reported beside the row-sharded headline (north_star asks for row sharding)
        for _ in range(2):
            replica.score_batch_async(host[0], dims, OUT_HW).wait()
        barrier()
        w0 = time.perf_counter()
        pending = None
        for i in range(args.steps):
            tk = replica.score_batch_async(host[i % n_img], dims, OUT_HW)
            if pending is not None:
                pending.wait()
            pending = tk
        pending.wait()
        sec = max_over_ranks(time.perf_counter() - w0)[0]
        line["image_parallel_replicas"] = {"e2e_value": world * B * P * args.steps / sec, "unit": "patch-NN scores/s",
                                           "note": f"{world} independent replicas of the 200k bank, each rank scores its own batches from "
                                                   f"host buffers (no collective); NOT the headline: north_star shards the bank row-wise"}
        single_r0 = single if rank == 0 else None
        if rank != 0:
            replica.close()
    if rank == 0:
        src = full_res if world == 1 else single_r0
        par.update(parity_vs_oracle(src, [host[0][i] for i in range(B)], n_images=1 if args.skip_cpu else 2,
                                    exact_bank=bank if world == 1 else replica))
        if world > 1:
            replica.close()
    line["parity"] = par

    # ---- the drop-in API: methods.predict_batch with everything behind the ABI (SURVEY 8f-2) -------------------------
    if world == 1 and not args.skip_dropin:
        line["predict_batch_e2e"] = dropin_leg(bank, imgs, B)

    # ---- coreset selection of 10 % of the same bank (BASELINE.json: "coreset-select seconds") ------------------------
    if not args.skip_coreset:
        csr = sparse_csr(BANK_ROWS, DIM)
        n_sel = BANK_ROWS // 10
        idx, cs = coreset_point(bank, BANK_ROWS, n_sel, csr, comm)
        cs = max_over_ranks(cs)[0]
        d_proj = csr[3]
        rep = coreset_report(BANK_ROWS, d_proj, n_sel, cs, pk, world)
        line["coreset_select_s"] = cs
        line["coreset_roofline"] = {"bound": "hbm", "achieved": rep["achieved_gbs"], "peak": pk["hbm_gbs"] * world, "unit": "GB/s",
                                    "frac": rep["frac_of_hbm"], "kernel": "coreset_kernel<__half,3>", "us_per_pick": rep["us_per_pick"],
                                    "note": f"(n-1)*N*d'*2 B with N={BANK_ROWS}, d'={d_proj}, n={n_sel}; wall time of the whole "
                                            f"call incl. projection (max over ranks); peak = {world} x HBM; the projected bank "
                                            f"({BANK_ROWS * d_proj * 2 / 1e6:.0f} MB) is pinned in L2 as far as it fits, so "
                                            f"achieved/HBM-peak may exceed 1", "unique": int(len(set(idx.tolist())))}
        if world > 1:  # sharded picks == single-GPU picks (a prefix: the loop is sequential, so a prefix checks the exchange fully)
            n_chk = 2000
            replica = build_bank(0, BANK_ROWS, local)
            one = replica.coreset_select(n_chk, csr, L.CORESET_FP16)
            replica.close()
            t = torch.tensor([int((one == idx[:n_chk]).all())], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            line["parity"]["coreset_sharded_equals_single"] = bool(int(t))
            line["parity"]["coreset_check"] = f"first {n_chk} picks of the {world}-rank loop == single-GPU loop on a full replica, on every rank"
    if world == 1:
        # the FP32-equivalent 3-term GEMM for every query (CMDB_OPT_PREFILTER_TERMS=3), same results, for comparison
        bank.set_prefilter_terms(3)
        for i in range(3):
            submit(devb[i % n_img]).wait()
        n_full = max(5, args.steps // 2)
        ms_full, wall_full, st_full, _ = timed(devb, n_full, collect_stage=True, pipelined=False)
        bank.set_prefilter_terms(0)
        g3 = float(np.mean([x["gemm"] for x in st_full]))
        line["fp32_equivalent_3term_mode"] = {"value": B * P * n_full / (max(ms_full, wall_full) * 1e-3), "unit": "patch-NN scores/s",
                                              "gemm_ms": g3, "gemm_tflops_algorithmic": flop / (g3 * 1e-3) / 1e12,
                                              "frac_of_tf32_equivalent_peak": flop / (g3 * 1e-3) / 1e12 / (pk["bf16_tflops"] / 2.0),
                                              "note": "CMDB_OPT_PREFILTER_TERMS=3: hi.hi + hi.lo + lo.hi for every query; 3x the "
                                                      "tensor work; identical outputs"}
    if world == 1 and rank == 0 and not args.skip_cpu and not args.skip_coreset:
        line["coreset_baselines"] = coreset_baselines(bank, csr, idx, n_sel)
    # free the headline bank before the larger configurations
    torch.cuda.synchronize()
    del devb, host, imgs
    bank.close()
    # ---- BASELINE cfg 5 at 1M rows (every N), cfg 2 and cfg 4 in bounded form (N = 1) --------------------------------
    if not args.skip_extras:
        line["large_bank"] = large_bank_leg(rank, world, local, pk, steps=max(5, args.steps // 2), comm=comm)
        if world == 1:
            line["configs"] = {"cfg2_dual_bank": dual_bank_leg(local, pk), "cfg4_fused_bank_1pct": fused_bank_leg(local, pk),
                               "note": "bounded forms measured in this run; full sweeps: bench.py --config 2 / 3 / 4 / 5 "
                                       "(logs under profiles/)"}
    if comm is not None:
        comm.close()
    if world == 1 and rank == 0 and not args.skip_cpu:  # after every GPU measurement: it keeps all host cores busy
        v, ms, cores = cpu_reference_leg(3, 1)
        line["cpu_baseline"] = {"value": v, "unit": "patch-NN scores/s", "cores": cores, "kind": "port",
                                "sample": f"3 images x {P} patches against the full {BANK_ROWS}x{DIM} bank (oracle/restate.py "
                                          f"score_restated: torch.cdist + min + topk + bilinear + blur), {ms:.0f} ms/image"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def coreset_baselines(bank, csr, idx, n_sel):
    """the reference's own coreset path on the same projected bank (SURVEY 8d): its torch loop on this GPU ("reference GPU"
    line, features.py:401-420 as shipped) and on the host cores, both timed on a bounded number of picks and extrapolated
    linearly (per-pick cost is constant); sklearn's projection timed on a row sample"""
    from oracle import restate as O
    prev = torch.get_num_threads()
    torch.set_num_threads(host_cores())
    try:
        z = torch.from_numpy(bank.project(csr))
        picks_gpu, picks_cpu = 200, 12
        O.coreset_torch_literal(z[:4096], 8, "FP16", device="cuda")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ref_idx = O.coreset_torch_literal(z, picks_gpu + 1, "FP16", device="cuda")
        torch.cuda.synchronize()
        t_gpu = (time.perf_counter() - t0) / picks_gpu
        t0 = time.perf_counter()
        O.coreset_torch_literal(z, picks_cpu + 1, "FP16", device="cpu")
        t_cpu = (time.perf_counter() - t0) / picks_cpu
        sample = bank.read(0, 20_000)
        from sklearn import random_projection as _rp
        t0 = time.perf_counter()
        _rp.SparseRandomProjection(n_components=csr[3], random_state=0).fit_transform(sample)
        t_proj = (time.perf_counter() - t0) * (BANK_ROWS / 20_000)
        return {"reference_torch_cuda_loop_s": t_gpu * (n_sel - 1), "reference_torch_cpu_loop_s": t_cpu * (n_sel - 1),
                "sklearn_projection_s": t_proj, "cores": host_cores(),
                "first_picks_equal_ours": bool((ref_idx.numpy() == idx[:picks_gpu + 1]).all()),
                "note": "free-running equality against the reference loop run on CUDA (oracle.restate.coreset_torch_literal: the "
                        "loop of features.py:372-425 re-typed with the same torch calls; the unmodified file cannot travel to the "
                        "offline GPU box). Against the CPU-run reference golden only teacher-forced agreement is possible.",
                "sample": f"torch loop: {picks_gpu} picks on cuda / {picks_cpu} picks on cpu of the same {BANK_ROWS}x{csr[3]} projected "
                          f"bank, extrapolated to {n_sel - 1}; projection: 20000 rows extrapolated to {BANK_ROWS}"}
    finally:
        torch.set_num_threads(prev)


def dropin_leg(bank, imgs, B):
    """methods.RGBFeatures.predict_batch on the SAME 200k bank (f_coreset = 1: no subsampling): per-sample tensors in,
    fused float64 maps + image scores out; the late-fusion head is fitted on 4 training images with sklearn as in the
    reference (features.py:352-358)."""
    from cmdiad_b200 import RGBFeatures, default_args
    from cmdiad_b200.methods import DeviceLib
    m = RGBFeatures(default_args(f_coreset=1.0))
    m._banks["rgb"] = bank
    m.rgb_mean, m.rgb_std = torch.tensor(0.0), torch.tensor(1.0)  # the synthetic bank is used as is
    m.patch_rgb_lib = DeviceLib(bank)
    train = [{"rgb": imgs[i]} for i in range(4)]
    m.add_samples_to_late_fusion_mem_bank(train)
    m.run_late_fusion()
    n_images = 4 * B
    samples = [{"rgb": imgs[i % len(imgs)]} for i in range(n_images)]
    masks = [torch.zeros(1, OUT_HW, OUT_HW)] * n_images
    out = {}
    for name, smp in (("host_samples", samples), ("device_samples", [{"rgb": s["rgb"].cuda()} for s in samples])):
        m.predict_batch(smp, masks, [0] * n_images, [["w.png"]] * n_images)   # warm-up: pinned staging blocks, scratch
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.predict_batch(smp, masks, [0] * n_images, [["x.png"]] * n_images)
        sec = time.perf_counter() - t0
        out[name] = {"value": n_images * P / sec, "ms_per_image": sec / n_images * 1e3}
    # the reference's call pattern through the same API: one image per predict() call
    one = samples[:8]
    m.predict(one[0], masks[0], 0, ["y.png"])
    t0 = time.perf_counter()
    for smp in one:
        m.predict(smp, masks[0], 0, ["y.png"])
    sec = time.perf_counter() - t0
    out["predict_one_by_one"] = {"value": len(one) * P / sec, "ms_per_image": sec / len(one) * 1e3}
    # host-side head for comparison (what round 1 did: sklearn score_samples on 50 176 x m rows per image)
    m.device_head = False
    m.predict(one[0], masks[0], 0, ["y.png"])
    t0 = time.perf_counter()
    for smp in one:
        m.predict(smp, masks[0], 0, ["y.png"])
    sec = time.perf_counter() - t0
    out["predict_one_by_one_host_head"] = {"value": len(one) * P / sec, "ms_per_image": sec / len(one) * 1e3}
    out["unit"] = "patch-NN scores/s"
    out["images"] = n_images
    out["note"] = ("RGBFeatures.predict_batch / predict (cmdiad_b200/methods.py): raw per-sample patches in (host: gathered into a "
                   "pinned block; device: stacked on the GPU), (patch - mean) / std, scoring, lambda scaling and both linear "
                   "One-Class-SVM heads on the device (cmdb_score_fused_batch_submit / _wait), float64 fused map + score per image "
                   "out, result bookkeeping of multiple_features.py:996-1003 included")
    m._banks = {}  # the bank belongs to the caller
    return out


def run_config(args):
    """--config 2 / 3 / 4 / 5: the full forms of the other BASELINE configurations (one JSON line each)"""
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    pk = peaks()
    out = {"config": args.config, "n_gpus": world, "data": "synthetic (generated on the device)"}
    if args.config == 2:
        assert world == 1
        out["cfg2_dual_bank"] = dual_bank_leg(local, pk)
    elif args.config == 3:
        out["cfg3_ten_classes"] = ten_class_leg(rank, world, local, pk)
    elif args.config == 4:
        assert world == 1
        out["cfg4_fused_bank"] = fused_bank_leg(local, pk, fracs=(0.01, 0.10, 0.25))
    elif args.config == 5:
        comm = None
        if world > 1:
            from cmdiad_b200 import Comm
            comm = Comm(local, d_proj_max=512)
        out["cfg5_sweep"] = []
        for rows in (50_000, 200_000, 1_000_000, 4_000_000):
            picks = min(rows // 10, 20_000)  # bounded: per-pick cost is constant, us_per_pick is the figure of merit
            out["cfg5_sweep"].append(large_bank_leg(rank, world, local, pk, steps=10, rows=rows, picks=picks, comm=comm))
        if comm is not None:
            comm.close()
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16, help="images per step")
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4, 5],
                    help="1 = headline (default); 2 / 3 / 4 / 5 = full form of BASELINE.json configs[1] / [2] / [3] / [4]")
    ap.add_argument("--skip-coreset", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="skip the 1M-row bank and the bounded cfg 2 / cfg 4 legs")
    ap.add_argument("--skip-dropin", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the results of the last step of the headline loop to DIR/<name>.npy "
                         "(one GPU, --config 1, --impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config != 1):
        ap.error("--dump-outputs needs --impl ours and --config 1")
    args.warmup = max(3, args.warmup)
    if args.impl == "reference":
        return run_reference(args)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: cmdiad_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    if args.config != 1:
        return run_config(args)
    run_ours(args)


if __name__ == "__main__":
    main()

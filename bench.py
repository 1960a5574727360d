#!/usr/bin/env python
"""bench.py — boosting iterations/sec of the histogram tree-learner hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's own CPU path

One "step" = one boosting iteration (L2 gradients -> Train one tree -> score update) on the synthetic
10M x 1024, 255-bin, 127-leaf regression workload of BASELINE.json (C3 in SURVEY.md §8d).
  value : whole-job it/s with label/score/grad/hess already resident in HBM (device-resident boosting),
          timed with CUDA events on the learner's stream, max over ranks.
  e2e   : the same iteration through the reference-facing C-ABI call with HOST buffers: grad/hess are
          copied host->device inside Train (from pinned memory) and the per-row leaf ids device->host
          inside AddPredictionToScore, every step, inside the timed region.
  roofline : dominant kernel = k_hist_a (+ its k_hist_reduce); algorithmic bytes = n_leaf*(C*1 + 8 [+4 index]) +
          C*256*16 per launch, divided by the CUDA-event time of those launches (measured live, profiling pass).
  cpu_baseline : the UNMODIFIED reference (oracle/_ref/lib_lightgbm.so) on the host cores, bounded two-sample estimate;
          the measured full-workload numbers are the `--impl reference` / `--impl reference_cuda` arms.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "boosting iters/sec, 10M x 1K synthetic, 255 bins, 127 leaves"
# BASELINE.json configs (SURVEY.md §8d).  kind: how the feature values are drawn; shard: how N > 1 GPUs split the work.
WORKLOADS = {
    "C3": dict(rows=10_000_000, cols=1024, leaves=127, seed=44, kind="dense", objective="regression", shard="features"),
    "C2": dict(rows=1_000_000, cols=256, leaves=63, seed=42, kind="dense", objective="regression", shard="features"),
    # 2048 sparse features, mutually exclusive inside blocks of 4 => EFB bundles them into 512 uint8 columns (<= 253 bins)
    "C4": dict(rows=5_000_000, cols=2048, leaves=127, seed=45, kind="efb4", objective="binary", shard="features"),
    # Higgs-shaped: 21 low-level + 7 derived features, GOSS (docs/Experiments.rst settings: 255 leaves), row-sharded
    "C5": dict(rows=11_000_000, cols=28, leaves=255, seed=46, kind="higgs", objective="binary", shard="rows", goss=(0.2, 0.1)),
}
GEN_CHUNK = 65536
EFB_P = 0.02           # P(feature != 0); features of one block of 4 are mutually exclusive
EFB_VALUES = 63        # non-zero values 1..63 => 64 bins per feature, 1 + 4 * 63 = 253 stored values per bundle column


def wl_columns(wl):
    """stored uint8 columns of THIS repo's layout"""
    return wl["cols"] // 4 if wl["kind"] == "efb4" else wl["cols"]


def _chunk_jobs(rows, row_lo, row_hi, nblocks_lo, nblocks_hi):
    return [(s, b) for s in range(row_lo, row_hi, GEN_CHUNK) for b in range(nblocks_lo, nblocks_hi)]


def _run_jobs(work, jobs, threads):
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=threads or min(32, os.cpu_count() or 8)) as ex:
        list(ex.map(work, jobs))


def gen_bins(rows, cols, seed, col_lo=0, col_hi=None, threads=None, row_lo=0, row_hi=None):
    """Seeded synthetic bin matrix (SURVEY.md §8d): one Philox stream per (64K-row chunk, 128-column block), so the
    matrix — and any column slice or 64K-aligned row range of it — is identical whatever the thread count or the number
    of ranks, and a rank only generates the column blocks it owns."""
    col_hi = cols if col_hi is None else col_hi
    row_hi = rows if row_hi is None else min(rows, row_hi)
    assert row_lo % GEN_CHUNK == 0
    out = np.empty((row_hi - row_lo, col_hi - col_lo), dtype=np.uint8)
    cblock = 128

    def work(job):
        s, b = job
        e = min(rows, s + GEN_CHUNK)        # the chunk's extent in the FULL matrix fixes the stream length
        c0, c1 = b * cblock, min(cols, (b + 1) * cblock)
        rng = np.random.Generator(np.random.Philox(key=seed, counter=[0, 0, b, s // GEN_CHUNK]))
        blk = rng.integers(0, 255, (e - s, c1 - c0), dtype=np.uint8)
        lo, hi = max(c0, col_lo), min(c1, col_hi)
        e2 = min(e, row_hi)
        out[s - row_lo:e2 - row_lo, lo - col_lo:hi - col_lo] = blk[:e2 - s, lo - c0:hi - c0]
    _run_jobs(work, _chunk_jobs(rows, row_lo, row_hi, col_lo // cblock, (col_hi + cblock - 1) // cblock), threads)
    return out


def gen_efb4(rows, cols, seed, bundle_lo=0, bundle_hi=None, threads=None, row_lo=0, row_hi=None, raw=False):
    """C4: `cols` sparse features in exclusive blocks of 4.  Per (row, block): with probability 1 - (1 - p)^4 exactly one of
    the four features is non-zero, uniform in 1..63.  Returns either the BUNDLED uint8 columns [rows, bundles] exactly as
    the reference's EFB stores such a block (feature_group.h:253-267: 0 = all four at their most frequent bin 0, else
    1 + 63 * j + (v - 1) for feature j with value v => bin v), or (raw=True) the raw feature values [rows, 4 * bundles]."""
    nb_total = cols // 4
    bundle_hi = nb_total if bundle_hi is None else bundle_hi
    row_hi = rows if row_hi is None else min(rows, row_hi)
    assert row_lo % GEN_CHUNK == 0
    nb = bundle_hi - bundle_lo
    out = np.zeros((row_hi - row_lo, nb * (4 if raw else 1)), dtype=np.uint8)
    bblock = 32                                   # bundles per Philox stream
    p_any = 1.0 - (1.0 - EFB_P) ** 4

    def work(job):
        s, b = job
        e = min(rows, s + GEN_CHUNK)
        b0, b1 = b * bblock, min(nb_total, (b + 1) * bblock)
        rng = np.random.Generator(np.random.Philox(key=seed, counter=[0, 1, b, s // GEN_CHUNK]))
        act = rng.random((e - s, b1 - b0), dtype=np.float32) < p_any
        j = rng.integers(0, 4, (e - s, b1 - b0), dtype=np.uint8)
        v = rng.integers(1, EFB_VALUES + 1, (e - s, b1 - b0), dtype=np.uint8)
        lo, hi = max(b0, bundle_lo), min(b1, bundle_hi)
        e2 = min(e, row_hi)
        act, j, v = act[:e2 - s, lo - b0:hi - b0], j[:e2 - s, lo - b0:hi - b0], v[:e2 - s, lo - b0:hi - b0]
        if raw:
            r, c = np.nonzero(act)
            out[s - row_lo + r, 4 * (lo - bundle_lo + c) + j[r, c]] = v[r, c]
        else:
            out[s - row_lo:e2 - row_lo, lo - bundle_lo:hi - bundle_lo] = np.where(act, 1 + EFB_VALUES * j + (v - 1), 0).astype(np.uint8)
    _run_jobs(work, _chunk_jobs(rows, row_lo, row_hi, bundle_lo // bblock, (bundle_hi + bblock - 1) // bblock), threads)
    return out


def gen_higgs(rows, seed, threads=None, row_lo=0, row_hi=None):
    """C5: 28 columns — 21 "low-level" features uniform in 0..254 and 7 "high-level" ones = quantised means of three
    low-level features (SURVEY.md §8d)."""
    row_hi = rows if row_hi is None else min(rows, row_hi)
    assert row_lo % GEN_CHUNK == 0
    out = np.empty((row_hi - row_lo, 28), dtype=np.uint8)

    def work(job):
        s, _ = job
        e = min(rows, s + GEN_CHUNK)
        rng = np.random.Generator(np.random.Philox(key=seed, counter=[0, 2, 0, s // GEN_CHUNK]))
        low = rng.integers(0, 255, (e - s, 21), dtype=np.uint8)
        hi7 = np.stack([(low[:, 3 * k].astype(np.uint16) + low[:, 3 * k + 1] + low[:, 3 * k + 2]) // 3 for k in range(7)], axis=1)
        blk = np.concatenate([low, hi7.astype(np.uint8)], axis=1)
        e2 = min(e, row_hi)
        out[s - row_lo:e2 - row_lo] = blk[:e2 - s]
    _run_jobs(work, _chunk_jobs(rows, row_lo, row_hi, 0, 1), threads)
    return out


def gen_columns(wl, col_lo=0, col_hi=None, threads=None, row_lo=0, row_hi=None):
    """this repo's stored columns [rows, col_hi - col_lo] for any workload"""
    if wl["kind"] == "dense":
        return gen_bins(wl["rows"], wl["cols"], wl["seed"], col_lo, col_hi, threads, row_lo, row_hi)
    if wl["kind"] == "efb4":
        return gen_efb4(wl["rows"], wl["cols"], wl["seed"], col_lo, col_hi, threads, row_lo, row_hi)
    b = gen_higgs(wl["rows"], wl["seed"], threads, row_lo, row_hi)
    return np.ascontiguousarray(b[:, col_lo:col_hi]) if (col_lo, col_hi) not in ((0, None), (0, 28)) else b


def gen_raw_float(wl, threads=None, row_lo=0, row_hi=None):
    """the raw feature matrix [rows, cols] float32 the reference arms are fed (its own binning / bundling reproduces the
    stored columns above)"""
    if wl["kind"] == "efb4":
        b = gen_efb4(wl["rows"], wl["cols"], wl["seed"], 0, None, threads, row_lo, row_hi, raw=True)
    else:
        b = gen_columns(wl, 0, None, threads, row_lo, row_hi)
    out = np.empty(b.shape, dtype=np.float32)
    nt = max(1, min(16, threads or 8))
    per = (len(b) + nt - 1) // nt
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=nt) as ex:       # numpy casts release the GIL
        list(ex.map(lambda t: np.copyto(out[t * per:(t + 1) * per], b[t * per:(t + 1) * per], casting="unsafe"), range(nt)))
    return out


LABEL_COLS = {"dense": 32, "efb4": 16, "higgs": 28}      # stored columns the label depends on


def gen_label_wl(wl, label_cols, row_lo=0):
    """Labels of rows row_lo .. row_lo + len(label_cols) from the first LABEL_COLS stored columns.  regression: linear +
    N(0, 0.5); binary: Bernoulli(sigmoid(linear)).  The per-row random stream is drawn for the whole workload and sliced."""
    rng = np.random.Generator(np.random.Philox(key=wl["seed"] + 1000))
    n = len(label_cols)
    if wl["kind"] == "dense":
        w = rng.normal(size=32)
        noise = rng.normal(size=wl["rows"]).astype(np.float32)[row_lo:row_lo + n]
        return ((label_cols.astype(np.float32) / 127.0 - 1.0) @ w.astype(np.float32) + 0.5 * noise).astype(np.float32)
    w = rng.normal(size=label_cols.shape[1])
    u = rng.random(wl["rows"], dtype=np.float32)[row_lo:row_lo + n]
    if wl["kind"] == "efb4":
        x = (label_cols > 0).astype(np.float32) * (((label_cols.astype(np.int32) - 1) % EFB_VALUES + 1) / float(EFB_VALUES))   # value / 63 of the active feature
        logit = 3.0 * (x @ w.astype(np.float32))
    else:
        logit = (label_cols.astype(np.float32) / 127.0 - 1.0) @ (0.5 * w).astype(np.float32)
    return (u < 1.0 / (1.0 + np.exp(-logit))).astype(np.float32)


def gen_label(rows, cols, seed, bins_first32):
    return gen_label_wl(dict(kind="dense", rows=rows, cols=cols, seed=seed), bins_first32)


def make_layout(lgb, wl, columns, col_lo=0):
    """Layout of a column slice [col_lo, col_lo + columns.shape[1]) of the workload"""
    nc = columns.shape[1]
    if wl["kind"] != "efb4":
        lay = lgb.Layout.identity(columns)
        lay.feat_real_index = np.arange(col_lo, col_lo + nc, dtype=np.int32)
        return lay
    f = np.arange(4 * nc, dtype=np.int32)
    z = np.zeros(4 * nc, np.int32)
    return lgb.Layout(np.ascontiguousarray(columns, dtype=np.uint8), f // 4, (1 + EFB_VALUES * (f % 4)).astype(np.int32),
                      np.full(4 * nc, EFB_VALUES + 1, np.int32), z.copy(), z.copy(), z.copy(), (4 * col_lo + f).astype(np.int32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self.gpu = gpu_index
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.max_mhz = float(out[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), out[2:6]):
                    if v.strip().lower() == "active":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self.t.start(); return self

    def __exit__(self, *a):
        self._stop.set(); self.t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def effective_cores():
    """Host threads this process can really use: min(affinity, cgroup quota)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def dist_env():
    rank = int(os.environ.get("RANK", 0)); world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    return rank, world, local


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


def ncu_traffic(workload, world):
    """DRAM bytes per k_hist_a launch from the committed ncu capture (profiles/hist_traffic.json) — only when that
    capture was taken on THIS workload at THIS GPU count; otherwise null (a number copied across configs is wrong)."""
    p = os.path.join(ROOT, "profiles", "hist_traffic.json")
    if os.path.exists(p):
        t = json.load(open(p))
        if t.get("workload") == workload and int(t.get("n_gpus", 0)) == world and t.get("kernel") == "k_hist_a":
            return t
    return None


# ----------------------------------------------------------------------------------------------------
# Reference arms.  Both run the UNMODIFIED reference through its own C API (oracle/refapi.py), never this repo's code:
#   --impl reference       the reference's OpenMP CPU learner (oracle/_ref/lib_lightgbm.so, built by oracle/Makefile.ref)
#   --impl reference_cuda  the reference's own CUDA learner compiled for sm_100 (oracle/_ref/cuda/lib_lightgbm.so, built by
#                          oracle/Makefile.refcuda): the rival on the same box
# They train on the FULL workload that config.workload prints (the matrix is streamed into the reference Dataset in
# row blocks, so the 41 GB fp32 copy of C3 never exists); `value` and `ms_per_step` are what was measured, unscaled.
REF_BLOCK_ROWS = 4 * GEN_CHUNK


def _ref_params(wl, threads, device="cpu", quantized=0):
    # Dataset parameters.  C4: the Dataset is CONSTRUCTED with the cuda rules (dense storage, bundles capped at 256 bins,
    # dataset.cpp:119,141,357-372) for every arm, so that the CPU learner trains on the same bundled columns.
    dsp = dict(max_bin=255, min_data_in_bin=1, enable_bundle="true" if wl["kind"] == "efb4" else "false", feature_pre_filter="false",
               verbosity=-1, num_threads=threads, device_type="cuda" if wl["kind"] == "efb4" else device)
    if device == "cuda":
        dsp.update(gpu_device_id=0, num_gpu=1)
    bp = dict(dsp, objective=wl["objective"], num_leaves=wl["leaves"], learning_rate=0.1, min_data_in_leaf=20, device_type=device)
    if wl.get("goss"):
        bp.update(data_sample_strategy="goss", top_rate=wl["goss"][0], other_rate=wl["goss"][1])
    if quantized:
        bp.update(use_quantized_grad="true", num_grad_quant_bins=quantized)
    return dsp, bp


def _ref_dataset(refapi, wl, rows, dsp, threads):
    """Reference Dataset over rows [0, rows) of the workload, streamed in REF_BLOCK_ROWS blocks of raw float features."""
    lc = LABEL_COLS[wl["kind"]]
    label_cols = np.empty((rows, lc), dtype=np.uint8)

    def block(lo, hi):
        label_cols[lo:hi] = gen_columns(wl, 0, lc, threads=min(32, threads), row_lo=lo, row_hi=hi)
        return gen_raw_float(wl, threads=min(32, threads), row_lo=lo, row_hi=hi)
    t0 = time.time()
    ds = refapi.RefDatasetStreamed(block, rows, wl["cols"], None, dsp, block_rows=REF_BLOCK_ROWS,
                                   sample_rows=REF_BLOCK_ROWS if wl["kind"] == "efb4" else 65_536,
                                   sampled_columns=wl["kind"] == "efb4")       # EFB needs the real training-set construction
    ds.set_label(gen_label_wl(wl, label_cols))
    return ds, time.time() - t0


def _time_iters(bst, warmup, steps):
    for _ in range(warmup):
        bst.update()
    t0 = time.time()
    for _ in range(steps):
        bst.update()
    return (time.time() - t0) / max(steps, 1)


def _calibrate_threads(refapi, ds, wl, cores, device, quantized):
    """Shared GPU boxes advertise more logical CPUs than a tenant gets; OpenMP spin-waits then collapse (measured in
    round 1: 49 s/iter at 128 threads vs ~16 usable cores).  Time one iteration on a small Dataset at cores, cores/2,
    cores/4 threads and keep the fastest: the reference gets the best thread count the box offers."""
    if device != "cpu":
        return cores
    best, best_dt, t = cores, None, cores
    while t >= 4:
        _, bp = _ref_params(wl, t, device, quantized)
        b = refapi.RefBooster(ds, bp)
        dt = _time_iters(b, 1, 2)
        b.free()
        if best_dt is None or dt < best_dt:
            best, best_dt = t, dt
        t //= 2
        if t < cores // 4:
            break
    return best


def host_mem_available():
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 1 << 62
    try:
        lim = open("/sys/fs/cgroup/memory.max").read().strip()
        if lim != "max":
            cur = int(open("/sys/fs/cgroup/memory.current").read().strip())
            avail = min(avail, int(lim) - cur)
    except Exception:
        pass
    return avail


def run_reference(args, wl, rank, world, device="cpu", dropin=False):
    """Full-workload arm through the LGBM_* C API: the reference CPU learner, the reference CUDA learner, or (dropin)
    THIS repo's learner behind the unmodified reference host code (integration/_build/lib_lightgbm.so, device_type=cuda:
    LGBM_BoosterUpdateOneIter -> GBDT::TrainOneIter -> B200TreeLearner -> liblgbm_b200.so).  None on ranks != 0."""
    if rank != 0:
        return None
    if dropin:
        os.environ["LGBM_REF_LIB"] = os.path.join(ROOT, "integration", "_build_cuda" if dropin == "device" else "_build", "lib_lightgbm.so")
    elif device == "cuda":
        os.environ["LGBM_REF_LIB"] = os.path.join(ROOT, "oracle", "_ref", "cuda", "lib_lightgbm.so")
    from oracle import refapi
    if not os.path.exists(refapi.REF_LIB):
        return {"unavailable": f"{refapi.REF_LIB} not built (oracle/Makefile.ref{'cuda' if device == 'cuda' else ''}, integration/Makefile)"}
    cores = effective_cores()
    rows = wl["rows"]
    need = 3.2 * rows * wl["cols"] + (2 << 30)      # column-wise + row-wise bin copies + one fp32 block, bytes
    note = ""
    if host_mem_available() < need:
        rows = max(REF_BLOCK_ROWS, int(host_mem_available() / (3.2 * wl["cols"])) // GEN_CHUNK * GEN_CHUNK)
        note = f"; host memory allows only {rows} rows"
    dsp, _ = _ref_params(wl, cores, device, args.quantized)
    cal_ds, _ = _ref_dataset(refapi, wl, min(rows, REF_BLOCK_ROWS), dsp, cores)
    threads = _calibrate_threads(refapi, cal_ds, wl, cores, device, args.quantized)
    cal_ds.free()
    dsp, bp = _ref_params(wl, threads, device, args.quantized)
    ds, t_ds = _ref_dataset(refapi, wl, rows, dsp, cores)
    bst = refapi.RefBooster(ds, bp)
    dt = _time_iters(bst, args.warmup, args.steps)
    trees = bst.trees()
    bst.free()
    ds.free()
    kind = ("this repo's learner behind the reference's LGBM_* C API, linked against the -DUSE_CUDA reference host code "
            "(integration/_build_cuda/lib_lightgbm.so): the reference's CUDA objective and score updater keep gradients and scores "
            "in HBM (boosting_on_gpu_), nothing crosses PCIe per iteration" if dropin == "device" else
            "this repo's learner behind the reference's LGBM_* C API (integration/_build/lib_lightgbm.so, device_type=cuda; "
            "host objective and score, gradients H2D and leaf ids D2H every iteration)" if dropin else
            "the reference's own CUDA learner (src/treelearner/cuda, -DUSE_CUDA, sm_100), boosting on the GPU" if device == "cuda"
            else "the reference's OpenMP CPU learner, col/row-wise chosen by its own auto-timing")
    sample = f"all {rows} rows x {wl['cols']} cols, {wl['leaves']} leaves, {kind}, {threads} host threads; " \
             f"dataset construction {t_ds:.1f}s excluded{note}"
    return dict(value=1.0 / dt, ms_per_step=dt * 1e3, cores=threads, sample=sample, rows=rows,
                first_tree=ref_tree_signature(trees[args.warmup]) if len(trees) > args.warmup else None)


def tree_signature(t):
    """Structure hash of one tree (split leaf / feature / threshold bin / default_left / child counts, in split order):
    equal hashes across N = 1, 2, 4, 8 prove that every configuration grew the same tree."""
    import hashlib
    h = hashlib.sha1()
    for k in ("leaf", "feature", "threshold", "default_left", "left_count", "right_count"):
        h.update(np.ascontiguousarray(t.splits[k]).tobytes())
    hv = hashlib.sha1(np.ascontiguousarray(t.leaf_value).tobytes()).hexdigest()[:16]
    return {"num_leaves": int(t.num_leaves), "root_feature": int(t.splits["feature"][0]) if t.num_leaves > 1 else -1,
            "root_threshold_bin": int(t.splits["threshold"][0]) if t.num_leaves > 1 else 0,
            "structure_sha1": h.hexdigest()[:16], "leaf_values_sha1": hv}


def ref_tree_signature(t):
    return {"num_leaves": int(t.num_leaves), "root_feature": int(t.split_feature[0]) if t.num_leaves > 1 else -1,
            "root_threshold": float(t.threshold[0]) if t.num_leaves > 1 else 0.0}


def run_reference_fit(args, wl):
    """Bounded CPU baseline for the b200 arm's `cpu_baseline` key (about 10-30 s of CPU work): the reference CPU
    learner timed on TWO row samples of the workload, t(rows) = a + b*rows fitted through them and evaluated at the
    full row count.  The per-split work that does not depend on the row count (the scan of 2 x T bins, the per-thread
    histogram merge) lands in `a` and is NOT multiplied up.  An estimate, labelled as such: the measured full-size
    number is `bench.py --impl reference`."""
    from oracle import refapi
    if not os.path.exists(refapi.REF_LIB):
        return None
    cores = effective_cores()
    s1, s2 = 2 * GEN_CHUNK, 8 * GEN_CHUNK
    s2 = min(s2, wl["rows"] // GEN_CHUNK * GEN_CHUNK) or wl["rows"]
    s1 = min(s1, s2 // 2)
    dsp, _ = _ref_params(wl, cores, "cpu", args.quantized)
    ds2, t_ds = _ref_dataset(refapi, wl, s2, dsp, cores)
    threads = _calibrate_threads(refapi, ds2, wl, cores, "cpu", args.quantized)
    dsp, bp = _ref_params(wl, threads, "cpu", args.quantized)
    warm = 10 if wl.get("goss") else 1            # GOSS starts sampling after 1 / learning_rate iterations (goss.hpp:33)
    b2 = refapi.RefBooster(ds2, bp)
    t2 = _time_iters(b2, warm, 3)
    b2.free(); ds2.free()
    ds1, _ = _ref_dataset(refapi, wl, s1, dsp, cores)
    b1 = refapi.RefBooster(ds1, bp)
    t1 = _time_iters(b1, warm, 3)
    b1.free(); ds1.free()
    slope = max((t2 - t1) / (s2 - s1), 0.0)
    icpt = max(t1 - slope * s1, 0.0)
    est = icpt + slope * wl["rows"]
    sample = (f"ESTIMATE from two row samples of the workload ({s1} rows: {t1 * 1e3:.0f} ms/iter, {s2} rows: {t2 * 1e3:.0f} ms/iter, "
              f"{wl['cols']} cols, {wl['leaves']} leaves, {threads} threads): t = {icpt * 1e3:.0f} ms + {slope * 1e9:.1f} ns/row "
              f"evaluated at {wl['rows']} rows; the measured full-size run is `bench.py --impl reference`")
    return {"value": 1.0 / est, "unit": "iters/sec", "cores": threads, "kind": "reference", "sample": sample}


DUMP_SCORE_ROWS = 1 << 20      # 8 MB of float64 scores (+ their row ids) whatever the workload's row count


def dump_outputs(out_dir, tree, scores):
    """What B200Booster.update() hands back in the last timed step (the tree: every split field, the leaf arrays) and the
    training scores it leaves, as float64 .npy files.  Scores of more than DUMP_SCORE_ROWS rows are sampled at row ids
    fixed by a seed, so that runs with the same arguments write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    out = {f"tree_split_{k}": tree.splits[k] for k in tree.splits.dtype.names}
    out.update(tree_leaf_value=tree.leaf_value, tree_leaf_weight=tree.leaf_weight, tree_leaf_count=tree.leaf_count,
               tree_leaf_depth=tree.leaf_depth, tree_num_leaves=np.array([tree.num_leaves]))
    rows = np.arange(len(scores))
    if len(scores) > DUMP_SCORE_ROWS:
        rows = np.sort(np.random.default_rng(0).choice(len(scores), DUMP_SCORE_ROWS, replace=False))
    out.update(score_rows=rows, scores=scores[rows])
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference_cuda", "dropin", "dropin_device"])
    ap.add_argument("--workload", default=os.environ.get("BENCH_WORKLOAD", "C3"), choices=list(WORKLOADS))
    ap.add_argument("--rows", type=int, default=0, help="override rows (debug only; makes the number INVALID)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--quantized", type=int, default=0, metavar="Q",
                    help="NOT the headline: train with use_quantized_grad=true, num_grad_quant_bins=Q (both arms)")
    ap.add_argument("--no-replicate", action="store_true",
                    help="N>1: keep one copy of the partition columns across the box (the split's owner pushes go-left bits)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the tree of the last timed step and the training scores (a fixed "
                         "sample of rows) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of this repo's arm (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else max(args.warmup, 1)
    rank, world, local = dist_env()
    wl = dict(WORKLOADS[args.workload])
    if wl.get("goss"):
        args.warmup = max(args.warmup, 10)       # both arms: GOSS samples only after 1 / learning_rate = 10 iterations
    if args.rows:
        wl["rows"] = args.rows
    metric = METRIC if args.workload == "C3" else f"boosting iters/sec, {wl['rows']} x {wl['cols']} synthetic ({wl['kind']}), {wl['leaves']} leaves"
    kind_txt = {"dense": f"{wl['cols']} dense features, 255 bins",
                "efb4": f"{wl['cols']} sparse features (p=0.02, exclusive in blocks of 4 -> {wl['cols'] // 4} EFB-bundled columns, <= 253 bins)",
                "higgs": f"{wl['cols']} Higgs-shaped features (21 low-level + 7 derived), 255 bins"}[wl["kind"]]
    obj_txt = "L2 regression" if wl["objective"] == "regression" else "binary logloss"
    if wl.get("goss"):
        obj_txt += f", GOSS top_rate={wl['goss'][0]} other_rate={wl['goss'][1]}"
    config = {"workload": f"{args.workload}: {wl['rows']} rows x {kind_txt}, {wl['leaves']} leaves, "
                          f"{obj_txt}, min_data_in_leaf=20, lr=0.1" +
                          (f", use_quantized_grad num_grad_quant_bins={args.quantized} (NOT the BASELINE configuration)" if args.quantized else ""),
              "parallelism": ((f"row-shard x{world}" if wl["shard"] == "rows" else
                               f"feature-shard x{world}" + ("" if args.no_replicate else ", partition columns replicated on every GPU"))
                              if world > 1 else "single GPU"),
              "l2_flush": (f"inputs larger than L2 (bin matrix {wl['rows'] * wl_columns(wl) / 1e9:.2f} GB >> 126 MB)"
                           if wl["rows"] * wl_columns(wl) > 2e8 else "bin matrix smaller than L2: L2 flushed by the per-tree 8 B/row gradient pass only")}

    if args.impl in ("reference", "reference_cuda", "dropin", "dropin_device"):
        dev = "cpu" if args.impl == "reference" else "cuda"
        r = run_reference(args, wl, rank, world, dev, dropin={"dropin": "host", "dropin_device": "device"}.get(args.impl, False))
        if rank == 0:
            if "unavailable" in r:
                print(json.dumps({"impl": args.impl, "unavailable": r["unavailable"]}), flush=True)
                return
            if r["rows"] != wl["rows"]:       # never print a workload that was not the one trained on
                config["workload"] = config["workload"].replace(f"{wl['rows']} rows", f"{r['rows']} rows (SAMPLE of {wl['rows']})")
            line = {"metric": metric, "impl": args.impl, "value": r["value"], "unit": "iters/sec", "n_gpus": args.gpus,
                    "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                    "scaling": "strong", "vs_baseline": None,
                    "dtype": ("f64 histograms (fp32 grad/hess)" if dev == "cpu" else
                              "30-bit fixed-point (g,h) -> exact int32 shared-memory atomics -> int64 histograms" if args.impl.startswith("dropin") else
                              "fp32 shared-memory atomics -> f64 histograms (gpu_use_dp=false)"),
                    "data": "synthetic", "config": config,
                    "cpu_baseline": {"value": r["value"], "unit": "iters/sec", "cores": r["cores"], "kind": "reference",
                                     "sample": r["sample"]},
                    "e2e": {"value": r["value"], "unit": "iters/sec",
                            "h2d_bytes_per_step": (wl["rows"] * 4 + 4) if args.impl == "dropin" else 0,
                            "d2h_bytes_per_step": (wl["rows"] * (1 if wl["leaves"] <= 255 else 4) + 4096) if args.impl == "dropin" else 0},
                    "first_timed_tree": r["first_tree"]}
            print(json.dumps(line), flush=True)
        return

    # ------------------------------------------------------------------------------ this repo's arm
    import lightgbm_b200 as lgb
    from lightgbm_b200 import distributed as D
    rows, cols, leaves = wl["rows"], wl["cols"], wl["leaves"]
    dist = None
    if world > 1:
        # rank 0 prints ONE JSON line on stdout.  NCCL writes its version banner (NCCL_DEBUG=VERSION, which this image sets)
        # and its INFO lines to stdout when the communicator is created, and honours NCCL_DEBUG_FILE only above the VERSION
        # level: raise VERSION to WARN, point the log at stderr, and create the communicator (init + first collective)
        # with file descriptor 1 parked on stderr
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", rank=rank, world_size=world)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    host_threads = max(4, (os.cpu_count() or 8) // max(world, 1))
    ncols = wl_columns(wl)
    lc = LABEL_COLS[wl["kind"]]
    goss = wl.get("goss")
    const_hess = wl["objective"] == "regression" and not goss          # RegressionL2loss::IsConstantHessian, GOSS rescales
    cfg = lgb.Config(num_leaves=leaves, min_data_in_leaf=20, gpu_device_id=local, use_cuda_graph=True,
                     use_quantized_grad=args.quantized > 0, num_grad_quant_bins=max(args.quantized, 2), stochastic_rounding=True)
    if wl["shard"] == "rows" and world > 1:
        # row-shard (SURVEY.md §8e, C5): every rank holds its row slice x ALL columns and the labels of those rows
        r0, r1 = D.shard_rows(rows, world)[rank]
        a0 = r0 // GEN_CHUNK * GEN_CHUNK
        cols_arr = gen_columns(wl, threads=min(32, host_threads), row_lo=a0, row_hi=r1)[r0 - a0:]
        y = gen_label_wl(wl, cols_arr[:, :lc], row_lo=r0)
        lay = make_layout(lgb, wl, cols_arr)
        L = D.make_row_sharded_learner(lay, cfg, rank, world)
        my_cols, my_rows = ncols, r1 - r0
    else:
        # feature-shard (C2/C3/C4): every rank holds ALL rows x its column slice
        lo, hi = D.shard_columns(ncols, world)[rank]
        cols_arr = gen_columns(wl, lo, hi, threads=min(32, host_threads))
        label_cols = cols_arr[:, :lc] if lo == 0 and hi >= lc else gen_columns(wl, 0, lc, threads=min(32, host_threads))
        y = gen_label_wl(wl, label_cols)
        lay = make_layout(lgb, wl, cols_arr, lo)
        L = D.make_sharded_learner(lay, cfg, rank, world, replicate_columns=not args.no_replicate, is_constant_hessian=const_hess)
        my_cols, my_rows = hi - lo, rows
    bkw = dict(objective=wl["objective"])
    if goss:
        bkw.update(data_sample_strategy="goss", top_rate=goss[0], other_rate=goss[1])
    B = lgb.B200Booster(lay, y, cfg, learning_rate=0.1, device_resident=True, learner=L, **bkw)

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def barrier():
        if dist is not None:
            dist.barrier()

    # --- value: device-resident boosting iterations
    for _ in range(args.warmup):
        B.update()
    l0 = L.kernel_launches
    barrier()
    with ClockSampler(local) as clk:
        L.timer_start()
        t0 = time.time()
        first_tree = None
        for _ in range(args.steps):
            t = B.update()
            if first_tree is None:
                first_tree = t
        ms_total = L.timer_stop()
        barrier()
        wall = time.time() - t0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, t, B.scores())
    ms_total = max_over_ranks(ms_total)
    launches = L.kernel_launches - l0
    ms_per_step = ms_total / args.steps
    value = 1e3 / ms_per_step
    clocks = clk.summary()
    final_loss = B.l2() if wl["objective"] == "regression" else B.logloss()      # local rows in row-shard mode

    # --- roofline of the dominant kernel (k_hist), measured live with CUDA events around every launch
    L.set_profiling(True)
    L.hist_stats(reset=True)
    prof_steps = 3
    for _ in range(prof_steps):
        B.update()
    hist_ms, hist_rows, hist_launches = L.hist_stats()
    hist_root_rows = sum(int(t.leaf_count.sum()) for t in B.trees[-prof_steps:])      # bag sizes of the profiled trees
    by_kind = {k: v / prof_steps for k, v in L.profile_by_kind().items()}
    L.set_profiling(False)
    # algorithmic bytes: per histogrammed row C bin bytes + 8 (grad,hess) + 4 (row index, not for the root),
    # per launch the C*256*16 B of the int64 pool slot it fills (DESIGN.md §4)
    root_rows = hist_root_rows if goss else my_rows * prof_steps
    if wl["shard"] == "rows" and world > 1:       # split records carry GLOBAL counts; this rank built 1/world of those rows
        hist_rows /= world
        root_rows = root_rows / world if goss else root_rows
    alg_bytes = hist_rows * (my_cols + 8) + (hist_rows - root_rows) * 4 + hist_launches * my_cols * 256 * 16
    achieved = alg_bytes / (hist_ms * 1e-3) / 1e9
    peak, peak_kind = peak_hbm()
    tr = ncu_traffic(args.workload, world)
    roofline = {"bound": "hbm", "kernel": "k_hist_a (+ k_hist_reduce)" if not args.quantized else "k_hist_q", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "peak_kind": peak_kind,
                "traffic": tr["dram_bytes_per_launch"] if tr else None,
                # traffic: DRAM bytes per launch from the committed ncu capture (trees 4-5 of the same seeded run); the ratio is
                # taken against the algorithmic bytes of THOSE trees (later trees build fewer rows per launch); under ncu every
                # launch starts with a flushed L2, so k_hist_reduce's re-read of the dumped tables counts too
                "traffic_over_alg": (tr["dram_bytes_per_launch"] / tr.get("alg_bytes_per_launch_same_run", alg_bytes / max(hist_launches, 1))) if tr else None,
                "traffic_note": tr.get("note") if tr else None,
                "hist_share_of_step": (hist_ms / prof_steps) / ms_per_step,
                "alg_bytes_per_launch": alg_bytes / max(hist_launches, 1),
                "avg_launch_ms": hist_ms / max(hist_launches, 1), "rows_built_factor_k": hist_rows / root_rows,
                "ms_per_step_by_kernel": by_kind}

    # --- e2e: host buffers through the C-ABI, copies inside the timed region
    e2e = None
    if not args.no_e2e and not goss and not (wl["shard"] == "rows" and world > 1):
        if world > 1:
            # every rank owns a row slice of the HOST label / score: gradients of the slice H2D + one NVLink all-gather,
            # leaf ids of the slice D2H (lightgbm_b200/booster.py RowSlicedHostBooster)
            import torch
            from lightgbm_b200.booster import RowSlicedHostBooster
            H = RowSlicedHostBooster(L, y, 0.1, rank, world, dist, torch)
            h2d, d2h = H.per * 4, H.per
            note = ("every rank: L2 gradients of its N/world row slice on the host (pinned) -> H2D 4 B/row of the slice -> all-gather of the "
                    "full gradient vector over NVLink (NCCL) -> Train -> leaf ids of the slice D2H (1 B/row) -> host score += leaf value; "
                    "bytes are per rank")
        else:
            H = lgb.B200Booster(lay, y, cfg, learning_rate=0.1, device_resident=False, learner=L, pinned=True, objective=wl["objective"])
            h2d, d2h = rows * (4 if const_hess else 8) + 4, rows * (1 if leaves <= 255 else 4) + 4096
            note = ("host gradients (pinned, 4 B/row; the hessian is constant for L2 and only hessians[0] is read, as "
                    "in the reference) -> H2D inside Train; per-row leaf ids (1 B/row up to 255 leaves) D2H inside AddPredictionToScore; "
                    "host computes g = score - y and score += leaf_value[leaf_id]")
        for _ in range(args.warmup):
            H.update()
        barrier()
        for k in H.host_ms:
            H.host_ms[k] = 0.0
        t0 = time.time()
        for _ in range(args.steps):
            H.update()
        barrier()
        dt = max_over_ranks((time.time() - t0) / args.steps)
        e2e = {"value": 1.0 / dt, "unit": "iters/sec", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "ms_per_step": dt * 1e3, "host_ms_per_step": {k: v / args.steps for k, v in H.host_ms.items()}, "note": note}

    cpu = None
    if rank != 0:
        if dist is not None:
            dist.barrier(); dist.destroy_process_group()
        return
    if not args.no_cpu_baseline and world == 1:
        cpu = run_reference_fit(args, wl)

    line = {"metric": metric, "value": value, "unit": "iters/sec", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": ("int8 gradients -> packed int16:int16 histogram cells -> int64 pool, f64 gain scan" if args.quantized else
                      "30-bit fixed-point (g,h) per tree -> exact int32 hi/lo shared-memory atomics -> int64 histograms, f64 gain scan"), "data": "synthetic",
            "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline,
            "cpu_baseline": cpu, "wall_ms_per_step": wall * 1e3 / args.steps,
            ("final_train_l2" if wl["objective"] == "regression" else "final_train_logloss"): final_loss,
            "first_timed_tree": tree_signature(first_tree)}
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py — boosting iterations/sec of the LightGBM-on-Spark training hot path on N B200s.

Contract (driver): `python bench.py --gpus N --steps K --warmup W`; for N>1 it is launched under
torch.distributed.run (one rank per GPU).  A step = one boosting iteration (LGBM_BoosterUpdateOneIter
through the C ABI).  Default workload = BASELINE.json configs[2] (LightGBMClassifier binary, synthetic
100M x 512 dense, the config the metric is quoted on); `--config cfg2|cfg4|cfg5` selects the other GPU
configurations of BASELINE.json.  Rows are split evenly over the ranks (strong scaling), the per-split
histogram reduction is an NCCL int64 allreduce.  Rank 0 prints ONE JSON line.

Before the timed region every rank set runs (untimed, `--no-verify` skips it):
  * parity_check: 3 iterations on a 1M x 64 slice of the same generator on the SAME ranks, compared with the
    oracle's R-rank emulation (tree structure identical, values 1e-5) + equality of the model string across ranks;
  * bins_sample_check: a few thousand rows of the full-size dataset (incl. chunk boundaries) re-binned on the host;
  * hist_conservation_check: K4 over all local rows with integer gradients conserves (sum g, n) exactly per feature.

`--impl reference` times the CPU restatement of the reference path (the oracle; the real lightgbmlib
3.2.110 cannot be built or installed here — BASELINE.md §2) on a bounded row sample of the same workload.

`--dump-outputs DIR` writes, after the timed steps, what the last timed step computed as float64 .npy files (see
dump_outputs()).  The workload is synthesised from fixed seeds, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KIND_REGRESSION, KIND_BINARY, KIND_RANK, KIND_MULTI = 0, 1, 2, 3
CONFIG_ITERS = 100        # numIterations default of the estimator (LightGBMParams.scala:318-322): amortisation base for ingestion
DS_PARAMS = "max_bin=255 is_pre_partition=True bin_construct_sample_cnt=200000 num_threads=0"

# BASELINE.json configs[1..4] (configs[0] is the reference's CPU plumbing case: a parity test, not a bench line)
CONFIGS = {
    "cfg2": dict(rows=10_000_000, features=256, kind=KIND_REGRESSION, seed=2024, objective="regression", extra="", iters=200,
                 name="LightGBMRegressor, synthetic 10M x 256 dense f32, 255 bins, 200 iters (BASELINE.json configs[1])"),
    "cfg3": dict(rows=100_000_000, features=512, kind=KIND_BINARY, seed=2025, objective="binary", extra="is_unbalance=false", iters=100,
                 name="LightGBMClassifier binary, synthetic 100M x 512 dense f32, 255 bins, num_leaves=31, lr=0.1 (BASELINE.json configs[2], the config the metric is quoted on)"),
    "cfg4": dict(rows=20_000_000, features=136, kind=KIND_RANK, seed=4, objective="lambdarank",
                 extra="lambdarank_truncation_level=20 eval_at=1,2,3,4,5", iters=100,
                 name="LightGBMRanker lambdarank, synthetic 20M rows / ~200k query groups (50-150 docs) x 136 feats (BASELINE.json configs[3])"),
    "cfg5": dict(rows=50_000_000, features=1024, kind=KIND_MULTI, seed=5, objective="multiclass", extra="num_class=10", iters=100,
                 name="LightGBMClassifier multiclass(10), synthetic 50M x 1024 with 64 categorical cols of cardinality 10^3..10^5 (log-uniform ids; "
                      "bins per categorical feature up to thousands, uint16 columns) and 256 cols 70 % zeros (BASELINE.json configs[4]; on 1 GPU: its 1/8 row slice)"),
}


def booster_params(cfg, num_machines):
    return ("metric= boost_from_average=true is_pre_partition=True boosting_type=gbdt tree_learner=data_parallel top_k=20 "
            "num_iterations=%d learning_rate=0.1 num_leaves=31 max_bin=255 bagging_fraction=1.0 pos_bagging_fraction=1.0 "
            "neg_bagging_fraction=1.0 bagging_freq=0 bagging_seed=3 early_stopping_round=0 feature_fraction=1.0 max_depth=-1 "
            "min_sum_hessian_in_leaf=0.001 num_machines=%d verbosity=-1 lambda_l1=0.0 lambda_l2=0.0 metric= "
            "min_gain_to_split=0.0 max_delta_step=0.0 min_data_in_leaf=20 objective=%s num_threads=0 %s" % (cfg["iters"], num_machines, cfg["objective"], cfg["extra"]))


def categorical_columns(cfg, F):
    """kind 3 (cfg5): the generator makes the last F/16 columns categorical (64 of 1024)"""
    if cfg["kind"] != KIND_MULTI:
        return []
    ncat = max(F // 16, 1)
    return list(range(F - ncat, F))


def dataset_params(cfg, F):
    cats = categorical_columns(cfg, F)
    return DS_PARAMS + (" categorical_feature=" + ",".join(str(c) for c in cats) if cats else "")


def group_sizes(seed, total_rows):
    """deterministic query-group sizes 50..150 (mean 100) covering exactly total_rows rows"""
    rng = np.random.default_rng(seed)
    sizes = rng.integers(50, 151, size=total_rows // 100 + 1000).astype(np.int64)
    cs = np.cumsum(sizes)
    k = int(np.searchsorted(cs, total_rows, side="left"))
    sizes = sizes[:k + 1].copy()
    sizes[k] -= cs[k] - total_rows
    return sizes[sizes > 0].astype(np.int32)


def shard(cfg, rank, world, n_total):
    """(row_start, n_local, group sizes or None): contiguous row blocks; a ranker keeps whole query groups on one rank
    (LightGBMRanker.scala:93-108)."""
    if cfg["kind"] != KIND_RANK:
        n_local = n_total // world + (1 if rank < n_total % world else 0)
        return rank * (n_total // world) + min(rank, n_total % world), n_local, None
    sizes = group_sizes(cfg["seed"], n_total)
    ends = np.cumsum(sizes.astype(np.int64))
    cuts = [0]
    for r in range(1, world):
        cuts.append(int(np.searchsorted(ends, n_total * r / world, side="left")) + 1)
    cuts.append(len(sizes))
    g0, g1 = cuts[rank], cuts[rank + 1]
    row_start = int(ends[g0 - 1]) if g0 > 0 else 0
    return row_start, int(sizes[g0:g1].sum()), sizes[g0:g1]


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe's clocks line).  Sampled in-process through NVML every
    20 ms (an `nvidia-smi -lms` child needs ~0.5 s to produce its first line, longer than the timed region of a multi-GPU run); the device
    is addressed by the UUID of this rank's CUDA device.  Falls back to `nvidia-smi -lms 200` when NVML cannot be loaded."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []
        self.samples = []          # (sm_mhz, sm_max_mhz, reason bitmask)
        self.nvml = None
        self.handle = None
        self._stop = threading.Event()
        self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            handle = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                handle = None
            if handle is None:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                ids = [x for x in vis.split(",") if x.strip() != ""]
                phys = int(ids[index]) if ids and ids[index].strip().isdigit() else index
                handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nvml, self.handle = pynvml, handle
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        try:
            sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
            try:
                mask = int(n.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
            except Exception:
                mask = int(n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            self.samples.append((sm, self.max_mhz, mask))
        except Exception:
            pass

    def _loop(self):
        while not self._stop.is_set():
            self._sample_nvml()
            self._stop.wait(0.02)

    def start(self):
        if self.nvml is not None:
            self._sample_nvml()
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.nvml is not None:
            self._sample_nvml()          # one more while the last kernels of the region have just finished
            self._stop.set()
            if self.thread is not None:
                self.thread.join(timeout=1.0)
            n = self.nvml
            bits = {"hw_slowdown": n.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": n.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": n.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": n.nvmlClocksEventReasonSwPowerCap}
            sm = [x[0] for x in self.samples]
            reasons = sorted(nm for nm, bit in bits.items() if any(x[2] & bit for x in self.samples))
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.max_mhz if sm else None, "reasons": reasons,
                    "samples": len(sm), "source": "nvml, 20 ms period"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(self.NAMES, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi -lms 200"}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_cores():
    """threads the CPU arm may really use: min(affinity mask, cgroup CPU quota) — NOT OMP_NUM_THREADS, which torchrun forces to 1"""
    n = len(os.sched_getaffinity(0))
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, p = f.read().split()
            if q != "max":
                n = max(1, min(n, int(int(q) / int(p))))
    except Exception:
        pass
    return n


def host_bin(col, info, ub):
    """numpy restatement of BinMapper::ValueToBin (numerical) — the checker of bins_sample_check"""
    nb = info["num_bin"] - (1 if info["missing_type"] == 2 else 0)
    v = np.asarray(col, dtype=np.float64).copy()
    nan = np.isnan(v)
    v[nan] = 0.0
    b = np.searchsorted(ub[:nb - 1], v, side="left")
    if info["missing_type"] == 2:
        b[nan] = info["num_bin"] - 1
    return b


def build_dataset(capi, cfg, n_local, F, row_start, ingest, groups=None, chunk_bytes=1 << 30):
    """Synthesise this rank's row shard on the device in chunks and ingest it.
    ingest == 'host': every chunk is first staged in pinned HOST memory (untimed) and then pushed through
    LGBM_DatasetPushRows from the host pointer (H2D + binning timed by the library with CUDA events) —
    the streaming analogue of Spark rows arriving at the task.  ingest == 'device': pushed from HBM."""
    seed, kind = cfg["seed"], cfg["kind"]
    sample_rows = capi.sample_indices(n_local, 200000, 1)
    sample, _ = capi.synthetic_rows((sample_rows.astype(np.int64) + row_start).astype(np.int32), F, seed, kind)
    ds = capi.Dataset.from_sampled_columns(sample, n_local, dataset_params(cfg, F))
    chunk = min(n_local, max(1, chunk_bytes // (F * 4)))          # ~1 GiB of f32 per chunk
    dev_x = capi.DeviceBuffer(chunk * F * 4)
    dev_y = capi.DeviceBuffer(chunk * 4)
    label = np.empty(n_local, dtype=np.float32)
    pinned = capi.PinnedBuffer(chunk * F * 4) if ingest == "host" else None
    host_bytes = 0
    for off in range(0, n_local, chunk):
        rows = min(chunk, n_local - off)
        capi.synthetic_fill(dev_x.ptr, dev_y.ptr, row_start + off, rows, F, seed, kind)
        capi.memcpy(label[off:off + rows].ctypes.data, dev_y.ptr, rows * 4)
        if pinned is not None:
            capi.memcpy(pinned.ptr, dev_x.ptr, rows * F * 4)              # stage the chunk on the host (untimed)
            ds.push_rows(pinned.ptr, off, nrow=rows, ncol=F, dtype_code=capi.DTYPE_FLOAT32)
            host_bytes += rows * F * 4
        else:
            ds.push_rows(dev_x.ptr, off, nrow=rows, ncol=F, dtype_code=capi.DTYPE_FLOAT32)
    dev_x.free(); dev_y.free()
    if pinned is not None:
        pinned.free()
    ds.set_field("label", label)
    if groups is not None:
        ds.set_field("group", groups)
    return ds, label, host_bytes, chunk


def numpy_workload(cfg, rows, F):
    """same distribution as the device generator (csrc/c_api.cu syn_x / syn_label), drawn with numpy so that the reference arm
    touches none of the product's code"""
    rng = np.random.default_rng(cfg["seed"])
    U = rng.random((rows, F), dtype=np.float32)
    m = min(F, 16)
    s = (np.sin(6.2831853 * U[:, :m]) * (1.0 + 0.1 * np.arange(m, dtype=np.float32))).sum(axis=1)
    if F >= 2:
        s += 8.0 * (U[:, 0] - 0.5) * (U[:, 1] - 0.5)
    noise = rng.random(rows) + rng.random(rows) - 1.0
    kind = cfg["kind"]
    if kind == KIND_REGRESSION:
        y = (s + 0.2449 * noise).astype(np.float32)
    elif kind == KIND_RANK:
        y = np.clip(np.floor(2.0 + 0.6 * s + 1.5 * noise), 0, 4).astype(np.float32)
    elif kind == KIND_MULTI:
        y = None      # needs the first categorical column: set below
    else:
        y = (rng.random(rows) < 1.0 / (1.0 + np.exp(-s))).astype(np.float32)
    X = U.astype(np.float64)
    X *= (1.0 + (np.arange(F) % 7))
    X -= (np.arange(F) % 5)
    if kind == KIND_MULTI:
        ncat = max(F // 16, 1)
        for j in range(ncat):
            log10c = 3.0 + (2.0 * j / (ncat - 1) if ncat > 1 else 0.0)
            X[:, F - ncat + j] = np.floor(10.0 ** (U[:, F - ncat + j].astype(np.float64) * log10c)) - 1.0
        X[:, :F // 4][rng.random((rows, F // 4)) < 0.7] = 0.0
        shift = (X[:, F - ncat].astype(np.int64) % 3) - 1.0
        y = np.clip(np.floor(5.0 + 0.7 * s + 1.2 * shift + 1.5 * noise), 0, 9).astype(np.float32)
    return X, y


def cpu_reference_run(cfg, n_total, F, sample_rows, steps, warmup, use_gpu_generator=True):
    """The reference's CPU path restated (oracle, OpenMP over all host cores the container may use) on a bounded row sample of
    the same synthetic workload.  Returns (iters_per_sec_on_sample, extrapolated_iters_per_sec, info)."""
    from oracle import oracle as O
    cores = host_cores()
    O.lib().orc_set_num_threads(cores)          # explicit: OMP_NUM_THREADS=1 under torchrun must not throttle the reference arm
    used = int(O.lib().orc_num_threads())
    if used == 1 and len(os.sched_getaffinity(0)) > 1 and cores > 1:
        raise RuntimeError("reference arm would run on 1 thread on a %d-core box" % cores)
    groups = None
    if cfg["kind"] == KIND_RANK:
        sizes = group_sizes(cfg["seed"], n_total)
        k = int(np.searchsorted(np.cumsum(sizes.astype(np.int64)), sample_rows, side="right"))
        groups = sizes[:max(k, 1)]
        sample_rows = int(groups.sum())
    if use_gpu_generator:
        from mmlspark_b200 import capi
        X, y = capi.synthetic_rows(np.arange(sample_rows, dtype=np.int32), F, cfg["seed"], cfg["kind"])       # generator only; no product compute on this arm
    else:
        X, y = numpy_workload(cfg, sample_rows, F)
    ods = O.OracleDataset(X, dataset_params(cfg, F)).set_field("label", y)
    if groups is not None:
        ods.set_field("group", groups)
    ob = O.OracleBooster(ods, booster_params(cfg, 1))
    for _ in range(warmup):
        ob.update()
    t0 = time.perf_counter()
    for _ in range(steps):
        ob.update()
    dt = time.perf_counter() - t0
    hs, hc = ob.hist_stats()
    ips = steps / dt
    info = {"cores": used, "sample_rows": sample_rows, "hist_cells_per_s": hc / hs if hs > 0 else None,
            "hist_share": hs / (dt * (steps + warmup) / steps) if dt > 0 else None}
    return ips, ips * sample_rows / n_total, info


def k4_traffic(rows, feats, world):
    """roofline.traffic: DRAM bytes per K4 launch from the committed ncu --set full capture of this shape (profiles/), else null.
    (DRAM counters cannot be read without a profiler; the capture is refreshed whenever K4 changes.)"""
    for rnd in ("r02", "r01"):
        path = os.path.join(ROOT, "profiles", "%s_k4_dram_traffic_%dx%d.json" % (rnd, rows, feats))
        if world == 1 and os.path.exists(path):
            try:
                return float(json.load(open(path))["bytes_per_launch_avg"]), os.path.relpath(path, ROOT)
            except Exception:
                pass
    return None, None


# ---------------------------------------------------------------------------------------------- untimed verification legs
def verify_small_parity(capi, cfg, rank, world, dist):
    """3 iterations on 1M x 64 of the same generator, sharded over the SAME ranks, vs the oracle's R-rank emulation on rank 0.
    Returns (status string, model hash)."""
    n, F, iters = 1_000_000, 64, 3
    vcfg = dict(cfg, iters=iters)
    try:
        row_start, n_local, groups = shard(vcfg, rank, world, n)
        ds, label, _, _ = build_dataset(capi, vcfg, n_local, F, row_start, "device", groups, chunk_bytes=64 << 20)
        b = capi.Booster(ds, booster_params(vcfg, world))
        for _ in range(iters):
            b.update_one_iter()
        model = b.save_model_to_string()
        b.free(); ds.free()
    except Exception as e:      # noqa
        model = "ERROR " + repr(e)
    h = hashlib.sha256(model.split("\nparameters:")[0].encode()).hexdigest()[:16]
    hashes = [h]
    shards = [(0, n, None)]
    if dist is not None:
        hashes = [None] * world
        dist.all_gather_object(hashes, h)
        shards = [None] * world
        dist.all_gather_object(shards, shard(vcfg, rank, world, n)[:2])
    if rank != 0:
        return None, h
    if model.startswith("ERROR"):
        return "fail: " + model, h
    if len(set(hashes)) != 1:
        return "fail: model strings differ across ranks %s" % hashes, h
    try:
        from oracle import oracle as O
        from mmlspark_b200.modeltext import parse_model, compare_models
        O.lib().orc_set_num_threads(host_cores())
        X, y = capi.synthetic_rows(np.arange(n, dtype=np.int32), F, vcfg["seed"], vcfg["kind"])
        rank_rows = [s[1] for s in shards] if world > 1 else None
        ods = O.OracleDataset(X, dataset_params(vcfg, F), rank_rows=rank_rows).set_field("label", y)
        if vcfg["kind"] == KIND_RANK:
            ods.set_field("group", group_sizes(vcfg["seed"], n))
        ob = O.OracleBooster(ods, booster_params(vcfg, world))
        ob.train(iters)
        compare_models(parse_model(model), parse_model(ob.model_string()))
        return "ok", h
    except AssertionError as e:
        return "fail: " + str(e)[:300], h
    except Exception as e:      # noqa
        return "fail: " + repr(e)[:300], h


def verify_full_size(capi, cfg, ds, n_local, F, row_start, chunk):
    """size-independent properties of the dataset the timed region trains on; returns dict of 'ok' / 'fail: ...'"""
    out = {}
    try:
        rng = np.random.default_rng(11)
        edges = [r for k in range(1, 6) for r in (k * chunk - 1, k * chunk) if 0 <= r < n_local]
        rows = np.unique(np.concatenate([rng.integers(0, n_local, 3000), np.array([0, n_local - 1] + edges)])).astype(np.int32)
        Xs, _ = capi.synthetic_rows((rows.astype(np.int64) + row_start).astype(np.int32), F, cfg["seed"], cfg["kind"])
        got = ds.get_bins_rows(rows)
        bad = 0
        cats = set(categorical_columns(cfg, F))
        for f in range(0, F, max(1, F // 64)):              # 64 features spread over all tiles
            info = ds.feature_info(f)
            if info["is_trivial"] or f in cats:
                continue
            want = host_bin(Xs[:, f].astype(np.float32).astype(np.float64), info, ds.upper_bounds(f))
            bad += int((got[:, f] != want).sum())
        out["bins_sample_check"] = "ok" if bad == 0 else "fail: %d sampled cells differ from host binning" % bad
    except Exception as e:      # noqa
        out["bins_sample_check"] = "fail: " + repr(e)[:200]
    try:
        g = ((np.arange(n_local) % 7) - 3).astype(np.float32)
        h = np.ones(n_local, dtype=np.float32)
        H = ds.histogram(g, h)
        sg = float(g.astype(np.float64).sum())
        ok = True
        for f in range(F):
            info = ds.feature_info(f)
            if info["is_trivial"] or info["num_bin"] > 256:      # the kernel-level entry covers the uint8 tile features
                continue
            ok &= (float(H[f, :, 0].sum()) == sg) and (float(H[f, :, 1].sum()) == float(n_local))
        out["hist_conservation_check"] = "ok" if ok else "fail: a feature's bins do not sum to (sum g, n)"
    except Exception as e:      # noqa
        out["hist_conservation_check"] = "fail: " + repr(e)[:200]
    return out


DUMP_TREE_KEYS = ("num_leaves", "num_cat", "split_feature", "split_gain", "threshold", "decision_type", "left_child", "right_child",
                  "leaf_value", "leaf_weight", "leaf_count", "internal_value", "internal_weight", "internal_count", "cat_boundaries",
                  "cat_threshold")
DUMP_MAX_SCORES = 4 << 20         # float64 training scores kept in the dump: 32 MB


def dump_outputs(out_dir, bst, model_text):
    """What a caller of LGBM_BoosterUpdateOneIter has after the last timed step, as float64 arrays:
      tree_<key>.npy     the tree(s) that step added (one per class), read back through the model text; each key of the K trees
                         concatenated in class order (num_leaves and num_cat say where one tree ends); a key none of the trees
                         has values for (cat_* without categorical splits, split fields of single-leaf trees) is not written;
      train_score.npy    the raw training scores after that step, [K][m] for a fixed, seeded sample of m of this rank's rows
                         (all rows when they fit in DUMP_MAX_SCORES values)."""
    from mmlspark_b200.modeltext import parse_model
    os.makedirs(out_dir, exist_ok=True)
    model = parse_model(model_text)
    K = int(model["header"]["num_tree_per_iteration"])
    last = model["trees"][-K:]
    for key in DUMP_TREE_KEYS:
        arr = np.concatenate([np.atleast_1d(np.asarray(t.get(key, []), dtype=np.float64)) for t in last])
        if arr.size:
            np.save(os.path.join(out_dir, "tree_%s.npy" % key), arr)
    scores = bst.get_scores(0).reshape(K, -1)
    n = scores.shape[1]
    if n * K > DUMP_MAX_SCORES:
        rows = np.sort(np.random.default_rng(0).choice(n, size=DUMP_MAX_SCORES // K, replace=False))
        scores = scores[:, rows]
    np.save(os.path.join(out_dir, "train_score.npy"), np.ascontiguousarray(scores))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="cfg3", choices=sorted(CONFIGS))
    ap.add_argument("--rows", type=int, default=0, help="override the config's row count (debug)")
    ap.add_argument("--features", type=int, default=0)
    ap.add_argument("--ingest", default="host", choices=["host", "device"])
    ap.add_argument("--cpu-sample-rows", type=int, default=2_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's tree(s) and a sample of the training scores to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = dict(CONFIGS[args.config])
    N = args.rows or cfg["rows"]
    F = args.features or cfg["features"]
    if cfg["kind"] == KIND_MULTI and not args.rows:
        # 50M x 1024 is the 8-GPU configuration: one GPU runs its 1/8 row slice unless --rows says otherwise
        N = cfg["rows"] // 8 if world == 1 else cfg["rows"]
    config = {"workload": cfg["name"] if (N, F) == (cfg["rows"], cfg["features"]) else cfg["name"] + " [overridden to %dx%d]" % (N, F),
              "config": args.config, "rows": N, "features": F, "objective": cfg["objective"],
              "parallelism": "data_parallel x%d (rows sharded, NCCL int64 histogram allreduce)" % world,
              "l2_policy": "inputs (%.1f GB of bins per rank) are far larger than the 126 MB L2" % (N / world * F / 1e9)}

    if args.impl == "reference":
        if rank != 0:
            return
        ips_s, ips_x, info = cpu_reference_run(cfg, N, F, min(args.cpu_sample_rows, N), max(args.steps, 1), max(args.warmup, 1), use_gpu_generator=False)
        line = {"impl": "reference", "metric": "boosting_iters_per_sec", "value": ips_x, "unit": "iters/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": 1000.0 / ips_x, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64 histograms over u8 bins (fp32 gradients)", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": ips_x, "unit": "iters/s", "cores": info["cores"], "kind": "port",
                                 "sample": "restated CPU path (efficiency vs real lightgbmlib unverified): first %d rows of the same synthetic distribution, %d timed iterations at "
                                           "%.3f iters/s on the sample, scaled by rows (x%d/%d); histogram throughput %.3g cells/s" % (
                                               info["sample_rows"], args.steps, ips_s, info["sample_rows"], N, info["hist_cells_per_s"] or 0)},
                "e2e": {"value": ips_x, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    dist = None
    if world > 1:
        # torch first: its bundled libnccl.so.2 (2.28) must be the one the process binds; the engine's NCCL calls
        # (CommInitRank / AllReduce / AllGather) then resolve to the same library
        import torch  # noqa: F401
        import torch.distributed as dist_mod
    from mmlspark_b200 import capi
    capi.load()
    if world > 1:
        dist = dist_mod
        dist.init_process_group("gloo")          # host-side barrier / max-reduce only; training traffic is NCCL inside the library
    capi.set_device(local_rank)
    if world > 1:
        base = int(os.environ.get("MASTER_PORT", "29500")) + 512
        machines = ",".join("127.0.0.1:%d" % (base + r) for r in range(world))
        capi.network_init(machines, base + rank, 120, world)

    checks = {}
    if not args.no_verify:
        status, mh = verify_small_parity(capi, cfg, rank, world, dist)
        checks["parity_check"] = status
        checks["parity_check_what"] = "3 iterations on 1M x 64 of the same generator on the same %d rank(s) vs the oracle's %d-rank emulation; model hash %s on every rank" % (world, world, mh)

    row_start, n_local, groups = shard(cfg, rank, world, N)
    t_build = time.perf_counter()
    ds, label, host_bytes, chunk = build_dataset(capi, cfg, n_local, F, row_start, args.ingest, groups)
    ingest_ms = ds.ingest_ms()
    build_s = time.perf_counter() - t_build
    if not args.no_verify:
        full = verify_full_size(capi, cfg, ds, n_local, F, row_start, chunk)
        if dist is not None:
            allf = [None] * world
            dist.all_gather_object(allf, full)
            full = {k: ("ok" if all(a[k] == "ok" for a in allf) else next(a[k] for a in allf if a[k] != "ok")) for k in full}
        checks.update(full)
    bst = capi.Booster(ds, booster_params(cfg, world))
    bst.set_profile(True)

    def barrier():
        if dist is not None:
            dist.barrier()

    for _ in range(args.warmup):
        bst.update_one_iter()
    bst.get_timing(reset=True)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        bst.update_one_iter()           # returns after the iteration's tree was read back (device sync inside)
    wall = time.perf_counter() - wall0
    clocks = sampler.stop()
    barrier()
    tm = bst.get_timing()
    dev_ms = tm["total_ms"]
    model_text = bst.save_model_to_string().split("\nparameters:")[0]
    mhash = hashlib.sha256(model_text.encode()).hexdigest()[:16]
    leaves = [int(l.split("=")[1]) for l in model_text.split("\n") if l.startswith("num_leaves=")]
    # max over ranks
    if dist is not None:
        import torch
        t = torch.tensor([dev_ms, wall * 1000.0, ingest_ms, tm["hist_ms"]], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, ingest_ms_max, hist_ms = [float(x) for x in t]
        r = torch.tensor([float(tm["hist_rows"])], dtype=torch.float64)
        dist.all_reduce(r, op=dist.ReduceOp.SUM)
        hist_rows_all = float(r[0])
        hashes = [None] * world
        dist.all_gather_object(hashes, mhash)
    else:
        wall_ms, ingest_ms_max, hist_ms, hist_rows_all = wall * 1000.0, ingest_ms, tm["hist_ms"], float(tm["hist_rows"])
        hashes = [mhash]
    split_timing = os.environ.get("B200GBM_SPLIT_TIMING") is not None
    if rank != 0:
        if world > 1:
            capi.network_free()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, bst, model_text)
    checks["timed_model"] = {"trees": len(leaves), "min_leaves": min(leaves) if leaves else 0, "hash": mhash,
                             "identical_on_all_ranks": len(set(hashes)) == 1}
    steps = args.steps
    value = steps / (dev_ms / 1000.0)
    ms_per_step = dev_ms / steps
    # roofline of the dominant kernel (K4), per rank: algorithmic bytes / measured launch time
    launches = tm["hist_launches"]
    trees = steps
    rows_rank0 = float(tm["hist_rows"])
    nonroot_rows = max(rows_rank0 - trees * n_local, 0.0)
    algo_bytes = rows_rank0 * (F + 8.0) + nonroot_rows * 4.0 + launches * F * 255 * 16.0
    peak, peak_src = measured_peak()
    achieved = algo_bytes / (tm["hist_ms"] / 1000.0) / 1e9 if tm["hist_ms"] > 0 else None
    binfo = bst.get_info()
    minfo = bst.get_memory_info()
    traffic, traffic_src = k4_traffic(N, F, world)
    roofline = {"bound": "hbm", "kernel": "k4_hist_build_ws<%d>" % (3 if binfo["constant_hessian"] else 4), "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": (achieved / peak) if achieved else None,
                "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src, "launches": launches, "avg_launch_ms": tm["hist_ms"] / max(launches, 1),
                "cells_per_s": rows_rank0 * F / (tm["hist_ms"] / 1000.0) if tm["hist_ms"] > 0 else None,
                "k4_share_of_step": tm["hist_ms"] / dev_ms if dev_ms > 0 else None,
                "co_limit": "shared-memory ATOMS issue rate (profiles/r01_ubench_smem_scatter.json): %d native 32-bit atomics per cell" % (3 if binfo["constant_hessian"] else 4)}
    # e2e: per-iteration C-ABI wall time (tree read-back inside) + host ingestion amortised over the fit's iterations
    t_iter = wall_ms / steps
    amort = cfg["iters"]
    e2e_ms = t_iter + ingest_ms_max / amort
    tree_bytes = 31 * 80 + 256
    e2e = {"value": 1000.0 / e2e_ms, "unit": "iters/s", "h2d_bytes_per_step": int(host_bytes / amort), "d2h_bytes_per_step": tree_bytes,
           "ingest_ms": ingest_ms_max, "ingest_GBps_host_to_bins": host_bytes / 1e9 / (ingest_ms_max / 1000.0) if ingest_ms_max > 0 and host_bytes else None,
           "note": "UpdateOneIter through the C ABI incl. tree read-back, plus LGBM_DatasetPushRows ingestion from pinned host chunks "
                   "(H2D + binning) amortised over the %d iterations of the configured fit; ingest mode=%s. Deviations from the reference's feed, declared: "
                   "rows are handed over as f32 through the streaming API (the reference hands LGBM_DatasetCreateFromMat f64, DatasetAggregator.scala:335-343), "
                   "and the host-side row -> pinned-chunk staging (the Spark Row -> native array copy of a11) is outside the timed region" % (amort, args.ingest)}
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        ips_s, ips_x, info = cpu_reference_run(cfg, N, F, min(args.cpu_sample_rows, N), 3, 1)
        cpu = {"value": ips_x, "unit": "iters/s", "cores": info["cores"], "kind": "port",
               "sample": "restated CPU path (efficiency vs real lightgbmlib unverified): first %d rows of the same matrix, 3 timed iterations (%.3f iters/s on the sample), "
                         "scaled by rows; hist %.3g cells/s" % (info["sample_rows"], ips_s, info["hist_cells_per_s"] or 0)}
    line = {"metric": "boosting_iters_per_sec", "value": value, "unit": "iters/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int64 fixed-point histograms over u8 bins%s (fp32 gradients, fp64 split gains)" % (" + u16 bins of the wide categorical features" if cfg["kind"] == KIND_MULTI else ""),
            "data": "synthetic", "config": config,
            "hist_rows_x_feats_per_sec": hist_rows_all * F / (hist_ms / 1000.0) if hist_ms > 0 else None,
            "histogram_reduce": ("none (1 rank)" if world == 1 else
                                 {0: "ncclAllReduce int64", 1: "fused reduce-scatter+scan over NVLink peer memory (k_scan_dp)",
                                  2: "two-shot all-reduce kernel over NVLink peer memory (k_allreduce_p2p)"}[binfo["reduce_mode"]]),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": tm["launches"], "clocks": clocks,
            "dataset_build_s": build_s,
            "partition_column_copy_gb": round(minfo["partition_column_copy_bytes"] / 1e9, 2), "device_free_gb": round(minfo["device_free_bytes"] / 1e9, 1)}
    line.update(checks)
    print(json.dumps(line))
    if split_timing:
        bst.free()          # the per-operation breakdown of the TIMED booster (rank 0) goes to stderr when it is freed
    if world > 1:
        capi.network_free()


if __name__ == "__main__":
    main()

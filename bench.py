#!/usr/bin/env python
"""bench.py — flow-records/sec of fit+transform on the BASELINE.json workloads (default: configs[1], KDD99-full-shaped,
4,898,431 rows x 41 features, 5 classes, RandomForest 100 trees depth 16, maxBins 70, 75/25 split).

One "step" = one pass of the hot path over the whole record batch:
  StringIndexer.fit (category counts) -> randomSplit 75/25 (raw records) -> RandomForest.fit(train): findSplits sample +
  fused encode->bins straight from the records, bagging, level loop -> model.transform(test) -> confusion / macro-F1.
`value`   : records/s with the raw AoS records already resident in HBM (b200flow functional API).
`e2e`     : the same pass through the pyspark.ml-shaped shim (the call a user of the reference makes), starting from
            PINNED HOST records (H2D inside the timed region) and ending with predictions + metric back on the host.
`roofline`: dominant kernel (by CUDA-event time inside the timed steps); `frac` follows SURVEY.md 8(d)'s algorithmic bytes.
`cpu_baseline` (N=1): the MLlib-semantics oracle on the SAME batch, with `labels_equal` / `forest_equal` (bit parity at the
            benched size), plus scikit-learn's RandomForestClassifier on a bounded sample as secondary context (B2).
`--impl reference`: the CPU arm — the oracle ("port": Spark itself cannot run here, no JVM) on every host thread.
`--workload`: kdd_full (configs[1], default) | kdd10 (configs[0]) | kdd_script (kdd99.py:64 as written: 23 classes) |
            cicids_wed (configs[2]) | cicids_full (configs[3]) | cicids_script (cicids17.py:68 as written) | stream (configs[4]).
            The CICIDS workloads take the reference script's forest (20 trees, maxDepth 5, maxBins 78); `--trees 100 --depth 16`
            gives the configs[1]-sized forest on CICIDS-shaped rows (a stress case: 1.5 M nodes, see DESIGN.md).
`--scaling`: weak (rows per GPU fixed, default) | strong (the workload's global rows sharded over the ranks; every N prints
            `forest_hash`, equal for every N: integer histograms + global-row-keyed RNG).
`--dump-outputs DIR`: after the timed steps, the last timed step's results (predictions, probabilities, raw votes, confusion,
            macro-F1, thresholds and forest; the stream workload: predictions) as DIR/<name>.npy, float64, at most 64 MB in all
            (a seeded sample of rows when larger).  The inputs are seeded, so equal arguments give equal inputs on every run.
Launch: python bench.py --gpus N --steps K --warmup W   (N>1 under torchrun, one rank per GPU).
"""
import argparse
import hashlib
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "spark-network-traffic-classifier_b200")
for _p in (ROOT, PKG):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# name -> (schema, global rows, classes, trees, depth, maxBins, record dtype, reference site)
WORKLOADS = {
    "kdd_full": ("kdd", 4898431, 5, 100, 16, 70, "f32", "BASELINE configs[1]"),
    "kdd10": ("kdd", 494021, 2, 20, 5, 70, "f32", "BASELINE configs[0]; RandomForestClassifier(numTrees=20, maxBins=70) kdd99.py:64"),
    "kdd_script": ("kdd", 4898431, 23, 20, 5, 70, "f32", "kdd99.py:64 as written (23 attack labels)"),
    "cicids_wed": ("cicids", 692703, 6, 20, 5, 78, "f64", "BASELINE configs[2]; RandomForestClassifier(numTrees=20, maxBins=78) cicids17.py:68"),
    "cicids_full": ("cicids", 2830743, 15, 20, 5, 78, "f64", "BASELINE configs[3]; RandomForestClassifier(numTrees=20, maxBins=78) cicids17.py:68"),
    "cicids_script": ("cicids", 755774, 14, 20, 5, 78, "f64", "cicids17.py:68 as written (rows/classes left by the six filters)"),
    "stream": ("kdd", 1 << 26, 5, 100, 16, 70, "f32", "BASELINE configs[4]: rows per step (2^26-row chunk), 15 steps = 1.0e9 rows"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="kdd_full", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU (weak) / global rows (strong); 0 = the workload's")
    ap.add_argument("--trees", type=int, default=0)
    ap.add_argument("--depth", type=int, default=-1)
    ap.add_argument("--classes", type=int, default=0)
    ap.add_argument("--max-bins", type=int, default=0)
    ap.add_argument("--dtype", default="", choices=["", "f32", "f64"], help="record field type of the CICIDS workloads")
    ap.add_argument("--path", default="records", choices=["records", "dense"],
                    help="records: fused encode->bins from the raw records (product path); dense: materialised feature matrix")
    ap.add_argument("--cpu-rows", type=int, default=0, help="rows of the CPU arm's sample; 0 = auto")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sklearn", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float64)")
    a = ap.parse_args()
    kind, rows, classes, trees, depth, bins, dtype, site = WORKLOADS[a.workload]
    a.kind, a.site = kind, site
    a.rows = a.rows or rows
    a.classes = a.classes or classes
    a.trees = a.trees or trees
    a.depth = depth if a.depth < 0 else a.depth
    a.max_bins = a.max_bins or bins
    a.dtype = a.dtype or dtype
    return a


# ------------------------------------------------------------------------------------------------ workloads
class Workload:
    """the record schema, the synthetic generator and the encode plan of one BASELINE config."""

    def __init__(self, a):
        from b200flow import synth
        self.a, self.kind = a, a.kind
        if a.kind == "kdd":
            self.schema = synth.kdd_schema()
            self.cat_cols, self.label_col, self.F = list(synth.KDD_CATEGORICAL), "label", 41
        else:
            self.schema = synth.cicids_schema(78, a.dtype)
            self.cat_cols, self.label_col, self.F = [], "Label", 78
        self.row_bytes = self.schema.row_bytes

    def make(self, n, device, row_offset=0):
        from b200flow import synth
        if self.kind == "kdd":
            return synth.make_kdd(n, self.a.classes, seed=2019, device=device, row_offset=row_offset)
        return synth.make_cicids(n, self.a.classes, seed=2019, device=device, dtype=self.a.dtype, row_offset=row_offset)

    def count_cols(self):
        return self.cat_cols + [self.label_col]

    def plan(self, luts):
        """the reference scripts' feature vector: numeric columns in file order, then the indexed categorical ones
        (kdd99.py:39-46); CICIDS: all 78 numeric columns (cicids17.py:40-41)."""
        from b200flow import synth
        from b200flow.encode import EncodePlan
        plan = EncodePlan(self.schema)
        if self.kind == "kdd":
            for c in synth.KDD_COLUMNS:
                if c not in synth.KDD_CATEGORICAL and c != "label":
                    plan.add_numeric(c)
            for c in synth.KDD_CATEGORICAL:
                plan.add_index(c, luts[c])
        else:
            for f in self.schema.names[:-1]:
                plan.add_numeric(f)
        plan.set_label(self.label_col, luts[self.label_col])
        return plan

    def arity(self, ordered):
        return [0] * (self.F - len(self.cat_cols)) + [len(ordered[c]) for c in self.cat_cols]

    def describe(self, world, rows_local, global_rows):
        a = self.a
        shape = ("KDD99-shaped synthetic flows, 41 features (168-B AoS f32 records)" if self.kind == "kdd" else
                 "CICIDS2017-shaped synthetic flows, 78 features (%d-B AoS %s records)" % (self.row_bytes, a.dtype))
        return {"workload": "%s: %s: %d rows/GPU, %d-class, RandomForest numTrees=%d maxDepth=%d maxBins=%d, randomSplit 75/25, "
                            "fit+transform [%s]" % (a.workload, shape, rows_local, a.classes, a.trees, a.depth, a.max_bins, a.site),
                "name": a.workload, "rows_per_gpu": rows_local, "global_rows": global_rows, "features": self.F, "classes": a.classes,
                "num_trees": a.trees, "max_depth": a.depth, "max_bins": a.max_bins, "record_bytes": self.row_bytes,
                "path": a.path, "parallelism": "rows sharded over %d GPU(s), per-level histogram exchange (NCCL)" % world,
                "l2_policy": "inputs (%.0f MB records per GPU) larger than the 126 MB L2" % (rows_local * self.row_bytes / 1e6)}


def forest_hash(ex):
    """sha256 over the canonical forest export (tree, node id, split feature/kind/bin, left-set masks, class counts, gains)."""
    h = hashlib.sha256()
    for k in ("tree", "nid", "feat", "kind", "bin_thr", "is_leaf", "counts"):
        h.update(np.ascontiguousarray(np.asarray(ex[k]).astype(np.int64)).tobytes())
    h.update(np.ascontiguousarray(np.asarray(ex["mask"]).astype(np.uint64)).tobytes())
    internal = np.asarray(ex["is_leaf"]) == 0
    h.update(np.ascontiguousarray(np.asarray(ex["gain"], np.float64)[internal]).tobytes())
    return h.hexdigest()[:16]


DUMP_BYTES = 60 << 20          # all --dump-outputs files together, .npy headers included, stay under 64 MB


def forest_outputs(ex):
    """the canonical forest export as float64-exact arrays: the uint64 left-set masks are split into their 32-bit words."""
    return {"forest_" + k: (np.asarray(v, np.uint64).view(np.uint32) if k == "mask" else v) for k, v in ex.items()}


def dump_outputs(out_dir, outputs):
    """--dump-outputs: write each output of the last timed step as <out_dir>/<name>.npy in float64, so that two builds can be
    compared array for array.  When the arrays exceed DUMP_BYTES, every array over 1 MB keeps the same fraction of its rows,
    chosen by a generator seeded with its row count: arrays with one row per test record (prediction, probability,
    rawPrediction) keep the same records, and two runs of the same arguments keep the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: (v.detach().to(torch.float64).cpu().numpy() if torch.is_tensor(v) else np.asarray(v, np.float64))
              for k, v in outputs.items()}
    big = [k for k, v in arrays.items() if v.ndim and v.nbytes > (1 << 20)]
    big_bytes = sum(arrays[k].nbytes for k in big)
    room = DUMP_BYTES - sum(v.nbytes + 4096 for k, v in arrays.items() if k not in big) - 4096 * len(big)
    if big_bytes > room:
        rows = {}
        for k in big:
            n = arrays[k].shape[0]
            if n not in rows:
                rows[n] = np.sort(np.random.default_rng(n).choice(n, int(n * room / big_bytes), replace=False))
            arrays[k] = arrays[k][rows[n]]
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_pass(wl, rec_np, dicts, a, phases=None):
    """the oracle's (MLlib-semantics CPU restatement) version of one step on a host record batch.
    -> (macroF1, predictions, forest export)."""
    import oracle
    t0 = time.perf_counter()
    schema = wl.schema
    luts, ordered = {}, {}
    for c in wl.count_cols():
        cnt = oracle.category_counts(rec_np, schema.row_bytes, schema.offsets[c], len(dicts[c]))
        ordered[c], luts[c] = oracle.string_index_order(cnt, dicts[c])
    plan = wl.plan(luts)                                        # plan container only (host bookkeeping, no kernels)
    x, y, _ = oracle.encode(rec_np, schema.row_bytes, plan.slot_array(), plan.lut_array(), *plan.label)
    sid = oracle.random_split(2019, len(y), [0.75, 1.0])
    tr = sid == 0
    t1 = time.perf_counter()
    C = len(ordered[wl.label_col])
    fo, meta = oracle.fit_forest(x[tr], y[tr], C, wl.arity(ordered), num_trees=a.trees, max_bins=a.max_bins, max_depth=a.depth, seed=2019)
    t2 = time.perf_counter()
    tp, _ = oracle.bin_rows(x[~tr], meta["thresholds"], meta["n_thr"], meta["arity"], meta["max_bins"])
    _, _, pred = fo.predict(tp)
    cm = oracle.confusion(pred, y[~tr].astype(np.float64), C)
    f1 = oracle.metrics(cm)["macroF1"]
    t3 = time.perf_counter()
    if phases is not None:
        phases.update(encode_split_s=t1 - t0, fit_s=t2 - t1, transform_eval_s=t3 - t2)
    return f1, pred, fo.export()


def sklearn_pass(wl, rec_np, dicts, a, max_rows=400000):
    """secondary context (BASELINE.md B2): scikit-learn's RandomForestClassifier (a different algorithm: exact splits, no
    binning) on a bounded sample of the same arrays, every host core."""
    import oracle
    from sklearn.ensemble import RandomForestClassifier
    from sklearn.metrics import f1_score
    rec_np = rec_np[:max_rows]
    schema = wl.schema
    luts, ordered = {}, {}
    for c in wl.count_cols():
        cnt = oracle.category_counts(rec_np, schema.row_bytes, schema.offsets[c], len(dicts[c]))
        ordered[c], luts[c] = oracle.string_index_order(cnt, dicts[c])
    plan = wl.plan(luts)
    x, y, _ = oracle.encode(rec_np, schema.row_bytes, plan.slot_array(), plan.lut_array(), *plan.label)
    tr = oracle.random_split(2019, len(y), [0.75, 1.0]) == 0
    t0 = time.perf_counter()
    sk = RandomForestClassifier(n_estimators=a.trees, max_depth=a.depth, max_features="sqrt", n_jobs=-1, random_state=2019)
    sk.fit(x[tr], y[tr])
    pred = sk.predict(x[~tr])
    dt = time.perf_counter() - t0
    return {"value": len(y) / dt, "unit": "records/s", "rows": int(len(y)), "seconds": dt,
            "macro_f1": float(f1_score(y[~tr], pred, average="macro")),
            "what": "scikit-learn RandomForestClassifier(n_estimators=%d, max_depth=%d, n_jobs=-1) fit+predict, arrays pre-encoded "
                    "(exact CART, not MLlib's binned algorithm: context, not parity)" % (a.trees, a.depth)}


def cpu_stream_setup(wl, a, train_rows, train=None):
    """the oracle's resident forest for the stream workload: fitted like the GPU arm's.  `train` = (records, dicts) of the very
    batch the GPU arm trained on (the CUDA and CPU generators draw different streams for one seed)."""
    import oracle
    rec, dicts = train if train is not None else wl.make(train_rows, "cpu", row_offset=0)
    rec_np = rec.numpy()
    schema = wl.schema
    luts, ordered = {}, {}
    for c in wl.count_cols():
        cnt = oracle.category_counts(rec_np, schema.row_bytes, schema.offsets[c], len(dicts[c]))
        ordered[c], luts[c] = oracle.string_index_order(cnt, dicts[c])
    plan = wl.plan(luts)
    x, y, _ = oracle.encode(rec_np, schema.row_bytes, plan.slot_array(), plan.lut_array(), *plan.label)
    fo, meta = oracle.fit_forest(x, y, len(ordered[wl.label_col]), wl.arity(ordered), num_trees=a.trees, max_bins=a.max_bins,
                                 max_depth=a.depth, seed=2019)
    return plan, fo, meta


def cpu_stream_pass(wl, plan, fo, meta, rec_np):
    """one stream step on the CPU: encode -> bins -> predict with the resident forest.  -> predictions."""
    import oracle
    x, _, _ = oracle.encode(rec_np, wl.schema.row_bytes, plan.slot_array(), plan.lut_array(), *plan.label)
    tp, _ = oracle.bin_rows(x, meta["thresholds"], meta["n_thr"], meta["arity"], meta["max_bins"])
    return fo.predict(tp)[2]


def run_reference_stream(a, wl, threads):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    train_rows = min(a.rows, 4898431)
    plan, fo, meta = cpu_stream_setup(wl, a, train_rows)
    if a.cpu_rows <= 0:
        probe, _ = wl.make(200000, "cpu", row_offset=a.rows)
        t0 = time.perf_counter(); cpu_stream_pass(wl, plan, fo, meta, probe.numpy()); probe_s = time.perf_counter() - t0
        a.cpu_rows = int(max(50000, min(a.rows, 200000 / max(probe_s, 1e-3) * 240.0 / max(a.steps + a.warmup, 1))))
    rec, _ = wl.make(a.cpu_rows, "cpu", row_offset=a.rows)
    rec_np = rec.numpy()
    for _ in range(a.warmup):
        cpu_stream_pass(wl, plan, fo, meta, rec_np)
    t = []
    for _ in range(a.steps):
        t0 = time.perf_counter(); pred = cpu_stream_pass(wl, plan, fo, meta, rec_np); t.append(time.perf_counter() - t0)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"prediction": pred})
    ms = 1e3 * sum(t) / len(t)
    v = a.cpu_rows / (ms / 1e3)
    line = {"impl": "reference", "metric": "flow-records/sec encode+predict (stream)", "value": v, "unit": "records/s", "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "stream: KDD99-schema synthetic record stream, encode + predict with a resident RandomForest (%d trees, "
                                   "depth %d) [%s]" % (a.trees, a.depth, a.site), "name": "stream", "rows_per_gpu": a.rows,
                       "global_rows": a.rows * world, "sample_rows": a.cpu_rows, "features": 41, "classes": a.classes, "num_trees": a.trees,
                       "max_depth": a.depth, "max_bins": a.max_bins},
            "cpu_baseline": {"value": v, "unit": "records/s", "cores": threads, "kind": "port",
                             "sample": "%d-row chunk per step (same generator); oracle encode + bin + predict, forest fitted on %d rows"
                                       % (a.cpu_rows, train_rows)},
            "e2e": {"value": v, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle
    threads = oracle.set_num_threads()                           # torchrun exports OMP_NUM_THREADS=1: set the count explicitly
    wl = Workload(a)
    if a.workload == "stream":
        return run_reference_stream(a, wl, threads)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    full = a.rows
    if a.cpu_rows <= 0:                                          # calibrate on a small batch, then size the per-step sample
        probe_n = min(full, 300000)
        rec, dicts = wl.make(probe_n, "cpu")
        t0 = time.perf_counter(); cpu_pass(wl, rec.numpy(), dicts, a); probe_s = time.perf_counter() - t0
        budget_rows = probe_n / max(probe_s, 1e-3) * 240.0 / max(a.steps + a.warmup, 1)
        a.cpu_rows = int(max(20000, min(full, budget_rows)))
    a.cpu_rows = min(a.cpu_rows, full)
    rec, dicts = wl.make(a.cpu_rows, "cpu")
    rec_np = rec.numpy()
    for _ in range(a.warmup):
        cpu_pass(wl, rec_np, dicts, a)
    t, f1, ph = [], 0.0, {}
    for _ in range(a.steps):
        t0 = time.perf_counter(); f1, pred, ex = cpu_pass(wl, rec_np, dicts, a, ph); t.append(time.perf_counter() - t0)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"prediction": pred, "macro_f1": f1, **forest_outputs(ex)})
    ms = 1e3 * sum(t) / len(t)
    v = a.cpu_rows / (ms / 1e3)
    cfg = wl.describe(world, a.rows, a.rows * world if a.scaling == "weak" else a.rows)
    cfg["sample_rows"] = a.cpu_rows
    line = {"impl": "reference", "metric": "flow-records/sec fit+transform", "value": v, "unit": "records/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": a.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg, "macro_f1": f1,
            "phases_last_step_s": ph, "ms_min": 1e3 * min(t), "ms_max": 1e3 * max(t),
            "cpu_baseline": {"value": v, "unit": "records/s", "cores": threads, "kind": "port",
                             "sample": "%s (same generator/seed), full %d-tree depth-%d forest; oracle = C++/OpenMP restatement of "
                                       "MLlib (Spark needs a JVM: absent); thread count set explicitly (OMP_NUM_THREADS ignored)"
                                       % ("the whole %d-row batch" % full if a.cpu_rows >= full else
                                          "%d-row sample of the %d-row batch" % (a.cpu_rows, full), a.trees, a.depth)},
            "e2e": {"value": v, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arm
class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.05)
        except Exception as e:                                  # NVML missing: report that instead of dying
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def count_tables(wl, rec, dicts, grp):
    """R1 StringIndexer.fit, counting half: enqueue the category counts of every code column (one pass) -> device tensors."""
    from b200flow import dist as bdist, encode as enc
    cols = wl.count_cols()
    return [bdist.all_reduce_sum_(t, grp) for t in enc.category_counts_multi(rec, wl.schema, cols, [len(dicts[c]) for c in cols])]


def order_tables(wl, dicts, host_counts):
    """R1, ordering half (host, <= 70 entries per column): frequencyDesc ranks -> (luts, ordered)."""
    from b200flow import encode as enc
    luts, ordered = {}, {}
    for c, cnt in zip(wl.count_cols(), host_counts):
        ordered[c], luts[c] = enc.string_index_order(np.asarray(cnt), dicts[c])
    return luts, ordered


def fit_tables(wl, rec, dicts, grp):
    return order_tables(wl, dicts, [t.cpu().numpy() for t in count_tables(wl, rec, dicts, grp)])


def step_resident(wl, rec, dicts, a, grp, keep=None):
    """one pass with the records resident in HBM, functional API.  `keep` (dict) receives the model and the predictions."""
    from b200flow import dist as bdist, forest as fr, rows
    dev = rec.device
    n = rec.shape[0]
    counts = count_tables(wl, rec, dicts, grp)                                      # R1 (enqueued; read below)
    p = fr.ForestParams(num_trees=a.trees, max_depth=a.depth, max_bins=a.max_bins, seed=2019)
    off, _ = bdist.global_offset(n, dev, grp)
    sid = rows.random_split_ids(n, [0.75, 0.25], 2019, off, dev)                    # randomSplit (kdd99.py:52)
    if a.path == "records":
        # raw records only: 75/25 compaction; the category counts travel in the same device->host copy as the split sizes
        (([rtr], ntr), ([rte], nte)), host_counts = rows.split_many([rec], sid, 2, fetch=counts)
        luts, ordered = order_tables(wl, dicts, [h.numpy() for h in host_counts])
        plan, arity, C = wl.plan(luts), wl.arity(ordered), len(ordered[wl.label_col])
        toff, _ = bdist.global_offset(ntr, dev, grp)
        model = fr.fit_forest_records(rtr, plan, C, arity, p, row_offset=toff, group=grp)       # R2-R8, fused encode->bins
        raw, prob, pred, yte = model.predict_records(rte, plan, want_label=True)                # R9
    else:
        luts, ordered = order_tables(wl, dicts, [t.cpu().numpy() for t in counts])
        plan, arity, C = wl.plan(luts), wl.arity(ordered), len(ordered[wl.label_col])
        x, y, _ = plan.run(rec, torch.float32 if a.dtype == "f32" else torch.float64, want_valid=False)   # R2+R3 fused encode
        ((xtr, ytr), ntr), ((xte, yte), nte) = rows.split_many([x, y], sid, 2)
        del x, y
        toff, _ = bdist.global_offset(ntr, dev, grp)
        model = fr.fit_forest(xtr, ytr, C, arity, p, row_offset=toff, group=grp)
        raw, prob, pred = model.predict(xte)
    cm = bdist.all_reduce_sum_(fr.confusion_matrix(pred, yte.to(torch.float64), C), grp)   # R10
    f1 = fr.metrics_from_confusion(cm.cpu().numpy())["macroF1"]
    if keep is not None:
        keep.update(model=model, pred=pred, raw=raw, prob=prob, confusion=cm, macro_f1=f1)
    return f1, nte, model.train_stats, model.n_nodes


def step_e2e(wl, host_rec, dicts, a):
    """the same pass through the pyspark.ml-shaped shim, from pinned host records to host predictions."""
    from pyspark.ml import Pipeline
    from pyspark.ml.classification import RandomForestClassifier
    from pyspark.ml.evaluation import MulticlassClassificationEvaluator
    from pyspark.ml.feature import StringIndexer, VectorAssembler
    from pyspark.sql import DataFrame
    dataset = DataFrame.fromRecords(host_rec, wl.schema, dicts)                    # H2D of the raw records
    if wl.kind == "kdd":                                                           # kdd99.py:34-52
        cats = wl.cat_cols
        indexers = [StringIndexer(inputCol=c, outputCol=c + "_num") for c in cats]
        indexers.append(StringIndexer(inputCol="label", outputCol="label_num"))
        dataset = Pipeline(stages=indexers).fit(dataset).transform(dataset)
        numerical = [c for c in dataset.columns if c not in cats + ["label", "label_num"]]
        dataset = VectorAssembler(inputCols=numerical, outputCol="features").transform(dataset)
        label = "label_num"
    else:                                                                          # cicids17.py:40-54
        features = [f for f in dataset.columns if f not in ["Label"]]
        dataset = VectorAssembler(inputCols=features, outputCol="features").setHandleInvalid("skip").transform(dataset)
        dataset = StringIndexer(inputCol="Label", outputCol="Label_Idx").setHandleInvalid("skip").fit(dataset).transform(dataset)
        label = "Label_Idx"
    dataset = dataset.select(["features", label])
    train, test = dataset.randomSplit([0.75, 0.25], seed=2019)
    rf = RandomForestClassifier(labelCol=label, featuresCol="features", numTrees=a.trees, maxBins=a.max_bins, maxDepth=a.depth, seed=2019)
    pred = rf.fit(train).transform(test)
    ev = MulticlassClassificationEvaluator(labelCol=label, predictionCol="prediction", metricName="macroF1")
    f1 = ev.evaluate(pred)
    dev_pred = pred._cols["prediction"].data                                        # D2H of the step's result (pinned)
    host_pred = torch.empty(dev_pred.shape, dtype=dev_pred.dtype, pin_memory=True)
    host_pred.copy_(dev_pred, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return f1, host_pred


def timed(fn, steps, warmup, grp):
    import torch.distributed as dist
    out = None
    for _ in range(warmup):
        out = fn()
    if grp is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    if grp is not None:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if grp is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()) / steps, out


def load_counters():
    """per-kernel counters measured once with `ncu --set full` (profiles/): DRAM bytes per launch, LSU / issue utilisation."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


def main():
    a = parse()
    if a.impl == "reference":
        return run_reference(a)
    import torch.distributed as dist
    from b200flow import _lib, forest as fr
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    _lib.require_cuda()
    grp = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        grp = dist.group.WORLD
    dev = torch.device("cuda", local)
    wl = Workload(a)
    if a.workload == "stream":
        return run_stream(a, wl, dev, grp, world, rank, local)
    if a.scaling == "strong":                                   # the SAME global batch for every N, sharded by contiguous row blocks
        global_rows = a.rows
        rec, dicts = wl.make(global_rows, dev)
        lo, hi = (global_rows * rank) // world, (global_rows * (rank + 1)) // world
        rec = rec[lo:hi].clone()
        rows_local = hi - lo
    else:
        rows_local, global_rows = a.rows, a.rows * world
        rec, dicts = wl.make(rows_local, dev, row_offset=rank * rows_local)
    torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    # ---- value: records resident in HBM --------------------------------------------------------------
    for _ in range(a.warmup):
        step_resident(wl, rec, dicts, a, grp)
    fr.PROFILE = {}
    if sampler:
        sampler.start()
    k0 = _lib.launches
    keep = {}
    ms_step, (f1, nte, stats, n_nodes) = timed(lambda: step_resident(wl, rec, dicts, a, grp, keep), a.steps, 0, grp)
    launches = (_lib.launches - k0) // a.steps
    prof = fr.profile_totals()
    hist_entries = float(sum(float(t.item()) for t in fr.PROFILE.get("_hist_entries", [])))
    route_entries = float(sum(float(t.item()) for t in fr.PROFILE.get("_route_entries", [])))
    fr.PROFILE = None
    value = global_rows / (ms_step / 1e3)
    fhash = forest_hash(keep["model"].export())

    # ---- e2e: host records -> shim -> host predictions -----------------------------------------------
    e2e = None
    if not a.no_e2e:
        host_rec = rec.cpu().pin_memory()
        ms_e2e, (f1_e2e, host_pred) = timed(lambda: step_e2e(wl, host_rec, dicts, a), a.steps, min(a.warmup, 2), grp)
        e2e = {"value": global_rows / (ms_e2e / 1e3), "unit": "records/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": int(host_rec.numel()), "d2h_bytes_per_step": int(host_pred.numel() * 8 + 8),
               "macro_f1": f1_e2e, "macro_f1_equals_resident": bool(f1_e2e == f1),
               "api": "pyspark.ml shim: StringIndexer(s).fit/transform -> VectorAssembler -> randomSplit -> "
                      "RandomForestClassifier.fit -> transform -> MulticlassClassificationEvaluator"}
        del host_rec
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if a.dump_outputs:                                          # rank 0: its own test rows, and the global forest
        model = keep["model"]
        out = {"prediction": keep["pred"], "rawPrediction": keep["raw"], "probability": keep["prob"], "confusion": keep["confusion"],
               "macro_f1": keep["macro_f1"], "thresholds": model.thresholds, **forest_outputs(model.export())}
        if e2e is not None:
            out["e2e_prediction"] = host_pred
        dump_outputs(a.dump_outputs, out)

    # ---- roofline of the dominant kernel (CUDA events on the launching stream, inside the timed steps) -----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
    kern = {k: {"launches_per_step": v[0] // a.steps, "ms_per_step": v[1] / a.steps, "share_of_step": v[1] / a.steps / ms_step}
            for k, v in prof.items() if not k.startswith("_")}
    ntr_rows = stats.get("rows", rows_local - nte)                                  # local train rows
    F, T = wl.F, a.trees
    route_launches = max(kern.get("route_hist_level", {}).get("launches_per_step", 1), 1)
    # SURVEY.md 8(d) algorithmic bytes per step of each kernel
    alg = {
        "encode": rows_local * (wl.row_bytes + F * 4 + 4),
        "encode_bins": rows_local * (wl.row_bytes + F + 1),                         # "Encode -> bins": record in, bins + label out
        "bin_rows": rows_local * (4 * F + F + 1),
        "route_hist_level": route_launches * ntr_rows * (F + 1 + 5 * T),            # per level: F + 1 + T x (1 + 4) bytes per TRAINING ROW
        "hist_level": kern.get("hist_level", {}).get("launches_per_step", 0) * ntr_rows * (F + 1 + 5 * T),
        "predict": nte * (F + 8),                                                   # from bins: F in + 8 out per test row
    }
    for k in kern:
        if k in alg and kern[k]["ms_per_step"] > 0 and alg[k] > 0:
            kern[k]["algorithmic_bytes_per_step"] = alg[k]
            kern[k]["achieved_gbs"] = alg[k] / (kern[k]["ms_per_step"] * 1e-3) / 1e9
            kern[k]["frac_of_hbm_peak"] = kern[k]["achieved_gbs"] / peak
    if "route_hist_level" in kern:
        kern["route_hist_level"]["entries_per_step"] = route_entries / a.steps
        kern["route_hist_level"]["entries_per_s"] = route_entries / a.steps / (kern["route_hist_level"]["ms_per_step"] * 1e-3)
    dom = max(kern, key=lambda k: kern[k]["ms_per_step"])
    d = kern[dom]
    avg_ms = d["ms_per_step"] / max(d["launches_per_step"], 1)
    ctr = (load_counters().get(a.workload) or {}).get(dom) or {}       # counters exist for the workloads that were captured with ncu
    traffic = ctr.get("dram_bytes_per_launch")
    bound = {"route_hist_level": "lsu (shared-memory pipe: tile fills + tile reads + atomics), not hbm",
             "hist_level": "lsu / record gather", "encode_bins": "issue + shared-memory (binary search), not hbm",
             "predict": "l1 latency (divergent tree walk)", "encode": "hbm"}.get(dom, "hbm")
    if dom == "route_hist_level" and ctr.get("lsu_pct") is not None and ctr["lsu_pct"] < 60:
        bound = "gather latency (wide nodes: long-scoreboard stall, one record gather in flight per warp), not hbm"    # ncu: profiles/r02_route_hist_*_ncu.txt
    roofline = {"kernel": dom, "bound": bound, "achieved": d.get("achieved_gbs"), "peak": peak, "unit": "GB/s",
                "frac": d.get("frac_of_hbm_peak"), "traffic": traffic, "peak_source": peak_src,
                "dram_frac": (traffic / (avg_ms * 1e-3) / 1e9 / peak) if traffic else None,
                "lsu_pct": ctr.get("lsu_pct"), "issue_pct": ctr.get("issue_pct"), "counters_source": ctr.get("source"),
                "launches_per_step": d["launches_per_step"], "avg_launch_ms": avg_ms, "share_of_step": d["share_of_step"],
                "note": "achieved = SURVEY 8(d) algorithmic bytes (per level and TRAINING row: F + 1 + 5*T) / CUDA-event kernel time "
                        "inside the timed steps; after row de-duplication the kernel works on (unique record, tree) entries and is "
                        "bound by the SM's load/store pipe, so dram_frac (measured DRAM bytes per launch, ncu) is the HBM view"}

    # ---- CPU baseline + bit parity at the benched size -------------------------------------------------
    cpu = None
    if not a.no_cpu_baseline and world == 1:                     # rank 0 at N = 1 only (the tier contract)
        import oracle
        threads = oracle.set_num_threads()
        if a.cpu_rows <= 0:
            a.cpu_rows = rows_local                              # the whole batch the GPU arm processed
        same_batch = a.cpu_rows >= rows_local
        rec_c, dicts_c = (rec.cpu(), dicts) if same_batch else wl.make(a.cpu_rows, "cpu")
        ph = {}
        t0 = time.perf_counter(); f1_cpu, pred_cpu, ex_cpu = cpu_pass(wl, rec_c.numpy(), dicts_c, a, ph); dt = time.perf_counter() - t0
        cpu = {"value": rec_c.shape[0] / dt, "unit": "records/s", "cores": threads, "kind": "port",
               "sample": "%s, full %d-tree depth-%d forest, %.1f s; oracle = C++/OpenMP restatement of MLlib (Spark itself needs a "
                         "JVM: absent)" % ("the SAME %d-row batch the GPU arm processed" % rec_c.shape[0] if same_batch else
                                           "%d-row sample of the same workload (same generator)" % rec_c.shape[0], a.trees, a.depth, dt),
               "macro_f1": f1_cpu, "phases_s": ph}
        if same_batch:                                           # parity at the benched size, checkable from this line
            ex_gpu = keep["model"].export()
            cpu["macro_f1_equals_gpu"] = bool(f1_cpu == f1)
            cpu["labels_equal"] = bool(np.array_equal(keep["pred"].cpu().numpy(), pred_cpu))
            cpu["forest_equal"] = bool(forest_hash(ex_gpu) == forest_hash(ex_cpu) and len(ex_gpu["nid"]) == len(ex_cpu["nid"]))
            cpu["forest_hash_cpu"] = forest_hash(ex_cpu)
            cpu["test_rows_compared"] = int(len(pred_cpu))
        if not a.no_sklearn:
            try:
                cpu["sklearn"] = sklearn_pass(wl, rec_c.numpy(), dicts_c, a)
            except Exception as e:                               # secondary context only
                cpu["sklearn"] = {"unavailable": "%s: %s" % (type(e).__name__, e)}

    line = {"metric": "flow-records/sec fit+transform", "value": value, "unit": "records/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": a.scaling, "vs_baseline": None,
            "dtype": "u8 bins / uint32 histograms / f64 split scoring (%s records)" % a.dtype, "data": "synthetic",
            "config": wl.describe(world, rows_local, global_rows), "macro_f1": f1, "forest_nodes": n_nodes, "forest_hash": fhash,
            "train_levels": stats["levels"], "bagged_entries": stats["entries"],
            "train_rows": stats.get("rows"), "unique_binned_rows": stats.get("unique_rows"),
            "route_chunk": stats.get("route_chunk"), "route_passes": stats.get("route_passes"),
            "level_exchange_ms": kern.get("level_exchange", {}).get("ms_per_step"),   # collectives of the level loop (the sharded scoring of the reduce-scatter path runs inside this window)
            "clocks": sampler.summary() if sampler else None, "e2e": e2e, "gpu_launches": launches,
            "roofline": roofline, "kernels": kern, "cpu_baseline": cpu}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------ stream sweep (configs[4])
def run_stream(a, wl, dev, grp, world, rank, local):
    """BASELINE configs[4]: KDD99-schema record stream, encode + predict with a resident forest; a step = one chunk of
    `--rows` records per GPU (default 2^26; 15 steps = 1.0e9 rows per GPU-group).  The hot path per chunk is the fused
    encode->bins kernel, the de-duplication of the binned records, the batch predictor and the gather of the predictions back
    to the rows; no dense matrix, no collective (the stream shards by rows: comm-free, SURVEY.md 8e)."""
    import torch.distributed as dist
    from b200flow import _lib, forest as fr
    rows = a.rows
    train_rec, dicts = wl.make(min(rows, 4898431), dev, row_offset=0)            # the forest: fitted once, outside the timed region
    luts, ordered = fit_tables(wl, train_rec, dicts, None)
    plan = wl.plan(luts)
    p = fr.ForestParams(num_trees=a.trees, max_depth=a.depth, max_bins=a.max_bins, seed=2019)
    model = fr.fit_forest_records(train_rec, plan, len(ordered[wl.label_col]), wl.arity(ordered), p)
    train_host = (train_rec.cpu(), dicts) if (world == 1 and not a.no_cpu_baseline) else None
    del train_rec
    chunk, _ = wl.make(rows, dev, row_offset=(rank + 1) * rows)
    torch.cuda.synchronize()
    sampler = ClockSampler(local) if rank == 0 else None

    def step():
        raw, prob, pred, _ = model.predict_records(chunk, plan, want_raw=False, want_prob=False)
        return pred
    for _ in range(max(a.warmup, 1)):
        step()
    fr.PROFILE = {}
    if sampler:
        sampler.start()
    k0 = _lib.launches
    ms_step, pred = timed(step, a.steps, 0, grp)
    launches = (_lib.launches - k0) // a.steps
    prof = fr.profile_totals()
    fr.PROFILE = None
    # e2e: host chunks streamed in, double-buffered (copy stream), predictions streamed out
    e2e = None
    if not a.no_e2e:
        hrows = min(rows, 1 << 22)
        host = chunk[:hrows].cpu().pin_memory()
        bufs = [torch.empty_like(chunk[:hrows]) for _ in range(2)]
        hpred = torch.empty(hrows, dtype=torch.float64, pin_memory=True)
        copy_stream = torch.cuda.Stream(device=dev)
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        done = [torch.cuda.Event(), torch.cuda.Event()]
        state = {"i": 0}

        def issue(i):
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(done[i & 1])                             # the compute that last read this buffer has finished
                bufs[i & 1].copy_(host, non_blocking=True)
                ready[i & 1].record(copy_stream)
        for ev in done:
            ev.record()
        issue(0)

        def e2e_step():
            i = state["i"]; state["i"] += 1
            issue(i + 1)                                                        # next chunk's H2D overlaps this chunk's compute
            torch.cuda.current_stream().wait_event(ready[i & 1])
            _, _, pr, _ = model.predict_records(bufs[i & 1], plan, want_raw=False, want_prob=False)
            done[i & 1].record()
            hpred.copy_(pr, non_blocking=True)
            return pr
        ms_e2e, _ = timed(e2e_step, a.steps, 2, grp)
        torch.cuda.synchronize()
        e2e = {"value": hrows * world / (ms_e2e / 1e3), "unit": "records/s", "ms_per_step": ms_e2e, "rows_per_step": hrows,
               "h2d_bytes_per_step": int(host.numel()), "d2h_bytes_per_step": int(hrows * 8),
               "api": "ForestModel.predict_records on pinned host chunks, H2D of chunk i+1 overlapped with the compute of chunk i"}
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"prediction": pred})
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
    kern = {k: {"launches_per_step": v[0] // a.steps, "ms_per_step": v[1] / a.steps, "share_of_step": v[1] / a.steps / ms_step}
            for k, v in prof.items() if not k.startswith("_")}
    alg = {"encode_bins": rows * (wl.row_bytes + wl.F + 1), "predict": rows * (wl.F + 8)}
    for k in kern:
        if k in alg:
            kern[k]["achieved_gbs"] = alg[k] / (kern[k]["ms_per_step"] * 1e-3) / 1e9
            kern[k]["frac_of_hbm_peak"] = kern[k]["achieved_gbs"] / peak
    step_bytes = rows * (wl.row_bytes + 8)                                       # record in, prediction out
    achieved = step_bytes / (ms_step * 1e-3) / 1e9
    dom = max(kern, key=lambda k: kern[k]["ms_per_step"]) if kern else None
    line = {"metric": "flow-records/sec encode+predict (stream)", "value": rows * world / (ms_step / 1e3), "unit": "records/s",
            "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 1), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8 bins / f64 votes (f32 records)", "data": "synthetic",
            "config": {"workload": "stream: KDD99-schema synthetic record stream, %d rows per step and GPU (168-B records), "
                                   "encode + predict with a resident RandomForest (%d trees, depth %d, %d nodes) [%s]"
                                   % (rows, a.trees, a.depth, model.n_nodes, a.site),
                       "name": "stream", "rows_per_gpu": rows, "global_rows": rows * world, "rows_streamed_total": rows * world * a.steps,
                       "features": 41, "classes": a.classes, "num_trees": a.trees, "max_depth": a.depth, "max_bins": a.max_bins,
                       "parallelism": "row-sharded stream over %d GPU(s), no collective" % world,
                       "l2_policy": "inputs (%.0f MB per step) larger than the 126 MB L2" % (rows * wl.row_bytes / 1e6)},
            "clocks": sampler.summary() if sampler else None, "e2e": e2e, "gpu_launches": launches,
            "roofline": {"kernel": "step (encode_bins + dedup + predict + gather)", "bound": "hbm for the encode; the tree walk is latency-bound",
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                         "dominant_kernel": dom, "note": "achieved = (record bytes in + 8 B prediction out) x rows / step time, per GPU"},
            "kernels": kern, "cpu_baseline": None}
    if not a.no_cpu_baseline and world == 1:                    # the oracle on a bounded chunk, with bit parity of the predicted labels
        import oracle
        threads = oracle.set_num_threads()
        n_cpu = min(rows, a.cpu_rows if a.cpu_rows > 0 else 2000000)
        plan_c, fo, meta = cpu_stream_setup(wl, a, min(rows, 4898431), train_host)
        chunk_np = chunk[:n_cpu].cpu().numpy()
        t0 = time.perf_counter(); pred_cpu = cpu_stream_pass(wl, plan_c, fo, meta, chunk_np); dt = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": n_cpu / dt, "unit": "records/s", "cores": threads, "kind": "port",
                                "sample": "the first %d rows of the chunk the GPU arm processed, %.1f s; oracle encode + bin + predict with "
                                          "its own forest fitted on the same %d training rows" % (n_cpu, dt, min(rows, 4898431)),
                                "labels_equal": bool(np.array_equal(pred[:n_cpu].cpu().numpy(), pred_cpu)), "rows_compared": int(n_cpu)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

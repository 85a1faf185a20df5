#!/usr/bin/env python
"""bench.py -- rows/sec of the scoring hot path at batch = 65 536 x 23 features (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--model gbdt100d6|rf100d6] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

One "step" = one pass of the hot path over one 65 536-row batch of synthetic credit-default rows
(BASELINE configs[1]: 100-tree depth-6 GBDT in the reference's preprocessing; `--model rf100d6` times
the reference's own RandomForest shape instead).  One rank per GPU; rows are independent, so ranks share
nothing on the predict path (weak scaling, no collective); the only collective is the 576-byte NCCL
all-gather of the drift-monitor moments (config 5), done through the engine's C ABI.

Printed by rank 0: ONE JSON line.
  value      whole-job rows/s with inputs resident in HBM: K launches cycling over a pool of 32 distinct
             batches (201 MB > L2), CUDA events on the launching stream, max over ranks.
  e2e        the same metric through the C-ABI call b2f_predict() with HOST (pinned) buffers: H2D of the
             encoded rows and D2H of probabilities + labels inside the timed region, every step.
  roofline   algorithmic bytes (100 B/row: 92 B features in, 4 B probability + 4 B label out) / the average
             per-launch device time measured live in the timed region, against the measured HBM peak.
  cpu_baseline  the reference-style sklearn pipeline's predict_proba on this box's host cores (rank 0, N=1).

--impl reference times that CPU path alone (all host cores, process pool) and prints the same line shape.

--dump-outputs DIR  rank 0 writes what the last timed step of each timed path returned, as DIR/<name>.npy:
  value_proba1.npy, value_label.npy   float32 (65 536,): probability of class 1 and label of the value path's last launch
  e2e_predictions.npy                 float64 (65 536,): ``predictions`` of the plugin path's last B200Model.predict call
  Inputs and models are seeded, so two builds run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# rank 0's stdout carries exactly ONE JSON line.  Libraries (NCCL's "NCCL version ..." banner, torchrun notices) write
# to fd 1 directly, so fd 1 is pointed at stderr for the whole run and only the final line goes to the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(obj) -> None:
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())

BATCH = 65536
POOL = 32  # distinct device-resident batches: 32 * 6.29 MB = 201 MB > 126 MB L2
ALG_BYTES_PER_ROW = 100  # SURVEY.md section 8(d): 92 B in + 4 B proba + 4 B label
MOM_BYTES_PER_ROW = 92
METRIC = "rows/sec at batch=65536x23f"
MODELS = {
    "gbdt100d6": ("gbdt", dict(n_estimators=100, max_depth=6, random_state=0)),
    "rf100d6": ("rf", dict(n_estimators=100, max_depth=6, criterion="gini", random_state=0)),
    "gbdt500d8": ("gbdt", dict(n_estimators=500, max_depth=8, random_state=0)),
    "rf500d8": ("rf", dict(n_estimators=500, max_depth=8, criterion="entropy", random_state=0)),
}
N_TRAIN = 20000
# sklearn's GBDT fit is single-threaded: 500 x depth-8 on 20 000 rows takes minutes, so that model (config 3, latency sweep)
# is fitted on fewer synthetic rows -- its trees are as deep and as many, which is what the sweep measures
N_TRAIN_BY_MODEL = {"gbdt500d8": 4000}
TRAIN_SEED = 20239
DATA_SEED = 20240


def workload_label(model: str) -> str:
    """The same string in both arms' ``config.workload`` (the driver compares them)."""
    return f"cfg2: {model} in the reference preprocessing, batch {BATCH} x 23 features per GPU"


# ----------------------------------------------------------------------------- distributed plumbing
class Dist:
    def __init__(self, want_gpus: int, use_cuda: bool, solo: bool = False):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = 1 if solo else int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.torch = None
        self.use_cuda = use_cuda
        if self.world > 1:
            import torch
            import torch.distributed as dist

            self.torch = torch
            if use_cuda:
                torch.cuda.set_device(self.local_rank)
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            else:
                dist.init_process_group("gloo")
            self.dist = dist
        if want_gpus != self.world and self.rank == 0 and self.world > 1:
            print(f"[bench] note: --gpus {want_gpus} but WORLD_SIZE={self.world}; using WORLD_SIZE", file=sys.stderr)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
            if self.use_cuda:
                self.torch.cuda.synchronize()

    def max(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda" if self.use_cuda else "cpu")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum(self, x: float) -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda" if self.use_cuda else "cpu")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def bcast_bytes(self, b: bytes | None) -> bytes:
        if self.world == 1:
            return b
        obj = [b]
        self.dist.broadcast_object_list(obj, src=0)
        return obj[0]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


# ----------------------------------------------------------------------------- workload
def get_pipeline(name: str, dist: Dist):
    """Fitted sklearn pipeline for the named model (rank 0 fits, cached on local disk for the other
    ranks and for the other arm run on the same box)."""
    import joblib
    import sklearn

    from databricks_kubernetes_mlops_poc_b200 import training

    kind, params = MODELS[name]
    # per user: on a shared host another user's directory of the same name is neither writable nor to be unpickled
    cache_dir = os.environ.get("B2F_BENCH_CACHE", os.path.join(tempfile.gettempdir(), f"b2f_bench_cache_{os.getuid()}"))
    os.makedirs(cache_dir, exist_ok=True)
    n_train = N_TRAIN_BY_MODEL.get(name, N_TRAIN)
    path = os.path.join(cache_dir, f"{name}_n{n_train}_s{TRAIN_SEED}_sk{sklearn.__version__}.joblib")
    base = training.load_base_frame()
    if dist.rank == 0 and not os.path.exists(path):
        t0 = time.time()
        pipe = training.fit_synthetic(kind, base, n_train, TRAIN_SEED, **params)
        joblib.dump(pipe, path + ".tmp")
        os.replace(path + ".tmp", path)
        print(f"[bench] fitted {name} on {n_train} synthetic rows in {time.time() - t0:.1f}s", file=sys.stderr)
    dist.barrier()
    return joblib.load(path), base


def make_batches(base, enc, n_batches: int, seed: int):
    """-> (vocabs, codes, nums, rows uint32 (n_batches*BATCH, 24))"""
    from databricks_kubernetes_mlops_poc_b200 import training

    vocabs, codes, nums = training.synth_arrays(base, n_batches * BATCH, seed)
    return vocabs, codes, nums, enc.encode_arrays(codes, nums)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.samples = []  # (t, sm, max, power, [reasons])
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

        def pump():
            for line in self.proc.stdout:
                f = [x.strip() for x in line.split(",")]
                try:
                    if int(f[0]) != self.idx:
                        continue
                    reasons = [n for n, v in zip(names, f[4:8]) if v == "Active"]
                    self.samples.append((time.time(), float(f[1]), float(f[2]), float(f[3]), reasons))
                except (ValueError, IndexError):
                    continue

        self.thread = threading.Thread(target=pump, daemon=True)
        self.thread.start()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, t0: float, t1: float) -> dict:
        win = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
        if not win:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = sorted({r for s in win for r in s[4]})
        return {"sm_mhz": statistics.median(s[1] for s in win), "sm_max_mhz": max(s[2] for s in win),
                "power_w_max": max(s[3] for s in win), "reasons": reasons, "samples": len(win)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(model_name: str):
    """dram bytes per launch from the committed ncu capture, if one exists for this model."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            v = json.load(open(p)).get(model_name, {})
            return v.get("dram_bytes_per_launch") if isinstance(v, dict) else None
        except Exception:
            return None
    return None


# ----------------------------------------------------------------------------- CPU baseline
_POOL_STATE = {}


def _pool_predict(i):
    pipe, frames = _POOL_STATE["pipe"], _POOL_STATE["frames"]
    return pipe.predict_proba(frames[i])[:, 1]


def cpu_reference_rate(pipe, df, repeats: int, procs: int):
    """rows/s of pipeline.predict_proba over df split across `procs` forked worker processes
    (sklearn's GBDT predict holds the GIL; its RandomForest threads itself with n_jobs=-1)."""
    import multiprocessing as mp

    n = len(df)
    if procs <= 1:
        times = []
        for _ in range(repeats + 1):
            t0 = time.perf_counter()
            pipe.predict_proba(df)
            times.append(time.perf_counter() - t0)
        times = times[1:]
        return n / min(times), n / statistics.median(times), times
    idx = np.array_split(np.arange(n), procs)
    _POOL_STATE["pipe"] = pipe
    _POOL_STATE["frames"] = [df.iloc[i] for i in idx]
    ctx = mp.get_context("fork")
    with ctx.Pool(procs) as pool:
        pool.map(_pool_predict, range(procs))  # warm-up
        times = []
        for _ in range(repeats):
            t0 = time.perf_counter()
            pool.map(_pool_predict, range(procs))
            times.append(time.perf_counter() - t0)
    return n / min(times), n / statistics.median(times), times


def cpu_port_rate(pipe, codes, nums, repeats: int):
    """rows/s of the OpenMP C restatement (oracle/c/forest_walk.c) on all cores."""
    from oracle import treewalk as tw

    dump = tw.dump_pipeline(pipe)
    tw.predict_c(dump, codes[:1024], nums[:1024])
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        tw.predict_c(dump, codes, nums)
        times.append(time.perf_counter() - t0)
    return len(codes) / min(times)


def cpu_bandwidth() -> float:
    """CPUs the container may burn (cgroup CFS quota / period), 0.0 when unlimited.  The B200 boxes give a 128-CPU host a quota
    of 16: more busy workers than that (forked sklearn processes, polling encoder threads) get the whole cgroup throttled."""
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return 0.0 if q == "max" else float(q) / float(per)
    except (OSError, ValueError):
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return q / per if q > 0 and per > 0 else 0.0
    except (OSError, ValueError):
        return 0.0


def reference_procs(kind: str) -> int:
    """Worker processes of the reference arm: RF threads itself (n_jobs=-1, as the reference sets it); a GBDT is single-threaded
    in sklearn, so the batch is split over forked processes -- as many as the host has CPUs, at most 64, at most the quota."""
    if kind == "rf":
        return 1
    cores = os.cpu_count() or 1
    bw = cpu_bandwidth()
    return max(1, min(cores, 64, int(bw) if bw >= 1.0 else cores))


# ----------------------------------------------------------------------------- arms
def run_reference(args, dist: Dist):
    """--impl reference: the reference-style CPU path (sklearn Pipeline.predict_proba, the library the
    reference itself calls at 02-register-model.ipynb:335-337) on this box's host cores, rank 0 only.
    Each step scores a bounded sample of the cfg2 batch, sized so K steps end within ~2 minutes."""
    import sklearn

    from databricks_kubernetes_mlops_poc_b200 import training
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES

    pipe, base = get_pipeline(args.model, dist)
    kind = MODELS[args.model][0]
    cores = os.cpu_count() or 1
    vocabs, codes, nums = training.synth_arrays(base, BATCH, DATA_SEED)
    df = training.arrays_to_frame(vocabs, codes, nums)[ALL_FEATURES]
    procs = reference_procs(kind)
    K = max(args.steps, 1)
    _, _, t_probe = cpu_reference_rate(pipe, df, 1, procs)
    rows = BATCH
    if K * t_probe[0] > 120.0:
        rows = max(2048, int(BATCH * 120.0 / (K * t_probe[0])))
    best, med, times = cpu_reference_rate(pipe, df.iloc[:rows], K, procs)
    med_t = statistics.median(times)  # median, not mean: one descheduled worker process must not move the number 3x
    value = rows / med_t
    how = "n_jobs=-1 threads" if procs == 1 else f"{procs} forked processes (pool created once), rows split evenly"
    sample = (f"{len(times)} steps x {rows} rows of the {BATCH}-row cfg2 batch (a DataFrame of 9 string + 14 float columns) through sklearn "
              f"{sklearn.__version__} Pipeline.predict_proba ({how}); median step time")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": len(times),
        "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * med_t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32cmp+f64acc", "data": "synthetic",
        "config": {"workload": workload_label(args.model), "batch": BATCH, "forest": args.model, "rows_per_step": rows},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": cores if procs == 1 else procs, "kind": "reference", "sample": sample,
                         "host_cores": cores, "cpu_quota": cpu_bandwidth(), "best": best, "mean": rows / statistics.mean(times)},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "api": "sklearn Pipeline.predict_proba(DataFrame) -> ndarray (what the reference's CustomModel.predict calls, 02-register-model.ipynb:335-337)"},
        "gpu_launches": 0,
    }
    emit(line)


def host_thread_share(dist: Dist) -> int:
    """Encoder threads for this rank.  One rank: the library's default (the GPU's NUMA node, capped by the container's CPU
    bandwidth -- `b2f_host_threads_default`).  Under torchrun the ranks share the host: a rank takes the physical cores of its
    GPU's NUMA node divided by the ranks whose GPUs sit on that node, plus two, and never more than its share of the CPU
    quota.  (Measured on the 8-GPU box, 2 x 32 cores, quota 96: 8 ranks x 10 threads 548 M rows/s, x 7: 489 M, x 13: 502 M;
    4 ranks -- all four GPUs on node 0 -- x 10: 368 M, x 14: 306 M, x 22: 256 M.)"""
    env = os.environ.get("B200_HOST_THREADS")
    if env:
        return int(env)
    if dist.world == 1:
        return 0  # the library's default
    import ctypes

    from databricks_kubernetes_mlops_poc_b200 import _cabi

    lib = _cabi.load_library()
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(dist.world)))
    ncpu = ctypes.c_int(0)
    my_node = lib.b2f_device_numa_node(dist.local_rank, ctypes.byref(ncpu))
    if my_node >= 0 and ncpu.value > 0:
        on_my_node = sum(1 for r in range(local_world) if lib.b2f_device_numa_node(r, None) == my_node)
        share = (ncpu.value // 2) // max(1, on_my_node) + 2  # two hyper-threads per core on the B200 hosts
    else:
        share = (os.cpu_count() or 2) // 2 // max(1, local_world) + 2
    limit = float(lib.b2f_host_cpu_limit())
    if limit > 0:
        share = min(share, (int(limit) - 2 * local_world) // local_world)
    return max(1, min(32, share))


def run_b200(args, dist: Dist):
    from databricks_kubernetes_mlops_poc_b200 import _cabi, flatten, training
    from databricks_kubernetes_mlops_poc_b200._cabi import SCORED_DTYPE
    from databricks_kubernetes_mlops_poc_b200.engine import ForestEngine
    from databricks_kubernetes_mlops_poc_b200.model import B200Model
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES

    K, W = args.steps, max(args.warmup, 3)
    # one process per GPU: live on the GPU's socket (the DataFrame the encoder threads read, the Python heap the response lists
    # are built in and the pinned staging then share a NUMA node; on the 8-GPU box ranks 4-7 serve GPUs of node 1)
    bound_cpus = 0
    lib0 = _cabi.load_library()
    if os.environ.get("B200_BIND_CALLER", "1") != "0" and (dist.world > 1 or lib0.b2f_device_count() == 1):
        # (not when ONE process drives several GPUs -- the config-4 stream leg binds a thread per GPU to that GPU's node itself)
        bound_cpus = int(lib0.b2f_bind_caller_near(dist.local_rank))
    pipe, base = get_pipeline(args.model, dist)
    flat = flatten.flatten_pipeline(pipe)
    model = B200Model(flat, devices=[dist.local_rank], host_threads=host_thread_share(dist))  # the plugin object (classifier only)
    eng, enc = model.engine, model.encoder
    info0 = eng.info()

    # ---- inputs: POOL distinct batches per rank (rank-seeded), resident in HBM and in pinned host memory
    vocabs, codes, nums, rows24 = make_batches(base, enc, POOL, DATA_SEED + 1000 * dist.rank)
    if args.rows == "ranked" and info0["rank_ok"]:
        fmt, rows, fmt_name = _cabi.ROWS_RANKED, enc.rank_rows(rows24), "ranked"  # 32-byte rows: ranks among the forest's split values
    elif args.rows in ("ranked", "packed64") and info0["packed_ok"]:
        fmt, rows, fmt_name = _cabi.ROWS_PACKED64, enc.pack_rows(rows24), "packed64"
    else:
        fmt, rows, fmt_name = _cabi.ROWS_WORDS24, rows24, "words24"
    row_bytes = rows.shape[1] * 4
    n_pool = POOL * BATCH
    d_rows = eng.device_alloc(rows.nbytes)
    d_proba = eng.device_alloc(n_pool * 4)
    d_label = eng.device_alloc(n_pool * 4)
    eng.h2d(d_rows, rows)
    h_rows = eng.pinned("bench_rows", rows.nbytes).view(np.uint32, rows.shape)
    h_rows[:] = rows
    h_out = eng.pinned("bench_out", n_pool * 8).view(SCORED_DTYPE, (n_pool,))  # {float32 proba1, int32 label} per row

    sampler = ClockSampler(dist.local_rank)
    sampler.start()
    t_load0 = time.time()

    # ---- value: device-resident, K back-to-back launches, ONE CUDA-event pair around the region on the launching stream
    #      (no events between launches: consecutive launches of the rank kernel overlap head and tail through programmatic
    #      dependent launch, which an event record in between would serialise)
    eng.predict_stream_timed(d_rows, BATCH, POOL, d_proba, False, d_label, W, fmt=fmt, per_launch=False)  # warm-up
    dist.barrier()
    l0 = eng.info()["launches"]
    _, ms_total = eng.predict_stream_timed(d_rows, BATCH, POOL, d_proba, False, d_label, K, fmt=fmt, per_launch=False)
    launches_value = eng.info()["launches"] - l0
    outputs = {}
    if args.dump_outputs and dist.rank == 0:  # launch i scores pool batch i % POOL into its own slot of d_proba / d_label
        last = (K - 1) % POOL
        outputs["value_proba1"] = np.empty(BATCH, dtype=np.float32)
        eng.d2h(outputs["value_proba1"], d_proba + last * BATCH * 4)
        label = np.empty(BATCH, dtype=np.int32)
        eng.d2h(label, d_label + last * BATCH * 4)
        outputs["value_label"] = label.astype(np.float32)
    dist.barrier()
    ms_total_max = dist.max(ms_total)
    value = dist.world * BATCH * K / (ms_total_max * 1e-3)
    inf1 = eng.info()
    kernel_used = ("k_forest_predict_rank (thread per row, integer rank compares, 4-byte nodes)" if inf1["launches_rank"] > 0 else
                   "k_forest_predict_tile (thread per row)" if inf1["launches_tile"] > 0 else "k_forest_predict (warp per row)")
    # the same launches one at a time, each bracketed by its own event pair (no overlap between launches): the isolated launch time
    iso_ms, _ = eng.predict_stream_timed(d_rows, BATCH, POOL, d_proba, False, d_label, min(K, 100), fmt=fmt, per_launch=True)

    # ---- parity spot check inside the bench (GPU vs sklearn on 2 048 rows of this rank's batch 0), EVERY rank
    got = np.empty(n_pool, dtype=np.float32)
    eng.d2h(got, d_proba)
    got_lab = np.empty(n_pool, dtype=np.int32)
    eng.d2h(got_lab, d_label)
    sel = np.arange(0, BATCH, BATCH // 2048)[:2048]
    df_sel = training.arrays_to_frame(vocabs, codes[sel], nums[sel])[ALL_FEATURES]
    want = pipe.predict_proba(df_sel)[:, 1]
    parity = dist.max(float(np.abs(got[sel].astype(np.float64) - want).max()))
    labels_equal = dist.max(0.0 if bool((got_lab[sel] == pipe.predict(df_sel)).all()) else 1.0) == 0.0

    # ---- e2e at the C ABI: pre-encoded rows in pinned host memory, H2D + kernel + D2H every step, wall clock around synchronous calls
    for i in range(W):
        b = i % POOL
        eng.predict_pairs(h_rows[b * BATCH:(b + 1) * BATCH], out=h_out[b * BATCH:(b + 1) * BATCH])
    dist.barrier()
    lat = []
    l0 = eng.info()["launches"]
    t0 = time.perf_counter()
    for i in range(K):
        b = i % POOL
        t1 = time.perf_counter()
        eng.predict_pairs(h_rows[b * BATCH:(b + 1) * BATCH], out=h_out[b * BATCH:(b + 1) * BATCH])
        lat.append(time.perf_counter() - t1)
    cabi_s = time.perf_counter() - t0
    launches_cabi = eng.info()["launches"] - l0
    dist.barrier()
    k_chk = min(K, POOL) * BATCH
    cabi_parity = float(np.abs(h_out["proba1"][:k_chk].astype(np.float64) - got[:k_chk]).max())  # host-buffer path == device path
    cabi_value = dist.world * BATCH * K / dist.max(cabi_s)
    ring = []
    for i in range(W):
        b = i % POOL
        eng.wait(eng.predict_pairs_async(h_rows[b * BATCH:(b + 1) * BATCH], h_out[b * BATCH:(b + 1) * BATCH]))
    dist.barrier()
    t0 = time.perf_counter()
    for i in range(K):
        b = i % POOL
        if len(ring) >= 2:
            eng.wait(ring.pop(0))
        ring.append(eng.predict_pairs_async(h_rows[b * BATCH:(b + 1) * BATCH], h_out[b * BATCH:(b + 1) * BATCH]))
    for t in ring:
        eng.wait(t)
    pipe_s = time.perf_counter() - t0
    dist.barrier()
    pipe_value = dist.world * BATCH * K / dist.max(pipe_s)

    # ---- e2e at the PLUGIN interface (the headline): B200Model.predict(DataFrame) -> dict, the call the reference makes at
    #      app/main.py:72, on the same 65 536-row DataFrame of 9 string + 14 float columns the reference arm scores (rank 0;
    #      other ranks: their own seed).  Inside every step: column buffers -> encode (host threads) -> H2D -> kernel -> D2H ->
    #      Python lists.
    if dist.rank == 0:
        pv, pc, pn = training.synth_arrays(base, BATCH, DATA_SEED)
    else:
        pv, pc, pn = vocabs, codes[:BATCH], nums[:BATCH]
    df0 = training.arrays_to_frame(pv, pc, pn)[ALL_FEATURES]
    plugin_warmup = max(W, 10)  # a warm service: encoder threads polling, staging allocated, three generations of response floats
    for _ in range(plugin_warmup):
        out0 = model.predict(df0)
    want0 = pipe.predict_proba(df0.iloc[sel])[:, 1]
    plugin_parity = dist.max(float(np.abs(np.asarray(out0["predictions"])[sel] - want0).max()))
    # collector hygiene of a long-lived service: everything allocated so far (the fitted sklearn pipeline, the synthetic frames)
    # moves to the permanent generation, so a generational collection inside the timed loops only looks at the loop's own objects
    import gc

    gc.collect()
    gc.freeze()
    dist.barrier()
    plat, stages = [], []
    l0 = eng.info()["launches"]
    t0 = time.perf_counter()
    for _ in range(K):
        t1 = time.perf_counter()
        out0 = model.predict(df0)
        plat.append(time.perf_counter() - t1)
        stages.append(model.last_timing)
    plugin_s = time.perf_counter() - t0
    launches_plugin = eng.info()["launches"] - l0
    if args.dump_outputs and dist.rank == 0:
        outputs["e2e_predictions"] = np.asarray(out0["predictions"], dtype=np.float64)
    dist.barrier()
    plugin_value = dist.world * BATCH * K / dist.max(plugin_s)
    st = [s for s in stages if s]
    breakdown = None
    if st:
        breakdown = {"columns_ms": 1e3 * statistics.median(s["columns_s"] for s in st),
                     "first_chunk_ms": 1e3 * statistics.median(s["first_chunk_s"] for s in st),
                     "chunks_and_lists_ms": 1e3 * statistics.median(s["chunks_and_lists_s"] for s in st),
                     "chunks": st[0]["chunks"], "host_threads": st[0]["threads"], "row_format": st[0]["row_format"]}
        a = np.random.default_rng(0).random(BATCH)
        tl = []
        for _ in range(5):
            t1 = time.perf_counter()
            a.tolist()
            tl.append(time.perf_counter() - t1)
        breakdown["tolist_65536_float64_alone_ms"] = 1e3 * min(tl)

    # ---- PCIe probe: one batch, pinned host -> device, synchronous copy (the C-ABI e2e floor is set by this)
    tt = []
    for _ in range(10):
        t1 = time.perf_counter()
        eng.h2d(d_rows, h_rows[:BATCH])
        tt.append(time.perf_counter() - t1)
    h2d_gbs = BATCH * row_bytes / min(tt) / 1e9

    # ---- sustained phase (>= 1.5 s of back-to-back launches) so the clock sampler sees the kernel under load
    t_sus0 = time.time()
    sus_steps, sus_ms = 0, 0.0
    while time.time() - t_sus0 < args.sustain:
        _, tot = eng.predict_stream_timed(d_rows, BATCH, POOL, d_proba, False, d_label, 2000, fmt=fmt, per_launch=False)
        sus_steps += 2000
        sus_ms += tot
    t_load1 = time.time()
    sustained = BATCH * sus_steps / (sus_ms * 1e-3) if sus_steps else None

    # ---- config 5: drift-monitor moments over 1M rows per job (K2), merged across ranks with NCCL
    mom = None
    if not args.no_moments:
        n_mom = min(1_000_000 // dist.world, n_pool)
        d_rows24 = d_rows
        if fmt != _cabi.ROWS_WORDS24:  # the moments kernel reads the 96-byte layout
            d_rows24 = eng.device_alloc(rows24.nbytes)
            eng.h2d(d_rows24, rows24)
        ms_m, local = eng.moments_device_timed(d_rows24, n_mom, 20, False)
        if dist.world > 1:
            uid = dist.bcast_bytes(ForestEngine.comm_unique_id() if dist.rank == 0 else None)
            eng.comm_init_rank(dist.world, dist.rank, uid)
            eng.moments_allgather(local)  # warm-up (communicator setup)
            dist.barrier()
            t0 = time.perf_counter()
            merged = eng.moments_allgather(local)
            t_gather = time.perf_counter() - t0
        else:
            merged, t_gather = local, 0.0
        # kernel-only roofline on the whole pool (201 MB, larger than L2) and on a >= 1 GiB input (SURVEY 8d)
        ms_big, _ = eng.moments_device_timed(d_rows24, n_pool, 10, False)
        if d_rows24 != d_rows:
            eng.device_free(d_rows24)
        peak, _ = measured_peak_gbs()
        mom = {
            "rows_total": n_mom * dist.world, "kernel_ms_per_rank": float(np.median(ms_m)),
            "nccl_allgather_merge_ms": 1e3 * t_gather,
            "kernel_gbs_201MB": MOM_BYTES_PER_ROW * n_pool / (float(np.median(ms_big)) * 1e-3) / 1e9,
            "kernel_frac_of_hbm_peak_201MB": MOM_BYTES_PER_ROW * n_pool / (float(np.median(ms_big)) * 1e-3) / 1e9 / peak,
            "count0": float(merged[9, 0]),
        }
        if dist.rank == 0 and dist.world == 1 and not args.no_gib:
            n_gib = 11_200_000  # x 96 B = 1.075 GB of 96-byte rows (1.03 GB algorithmic at 92 B/row)
            d_gib = eng.device_alloc(n_gib * 96)
            reps = (n_gib + rows24.shape[0] - 1) // rows24.shape[0]
            for r in range(reps):
                cnt = min(rows24.shape[0], n_gib - r * rows24.shape[0])
                eng.h2d(d_gib + r * rows24.shape[0] * 96, rows24[:cnt])
            ms_gib, _ = eng.moments_device_timed(d_gib, n_gib, 10, False)
            eng.device_free(d_gib)
            mom["kernel_gbs_1GiB"] = MOM_BYTES_PER_ROW * n_gib / (float(np.median(ms_gib)) * 1e-3) / 1e9
            mom["kernel_frac_of_hbm_peak_1GiB"] = mom["kernel_gbs_1GiB"] / peak
            mom["rows_1GiB"] = n_gib

    sampler.stop()
    clocks = sampler.summary(t_load0, t_load1)

    # ---- K4 (SURVEY a8): the reference's outlier detector as a second forest over the same rows (rank 0, N=1)
    outl = None
    if dist.rank == 0 and dist.world == 1 and not args.no_outliers:
        pk = enc.pack_rows(rows24) if info0["packed_ok"] else rows24
        d_pk = eng.device_alloc(pk.nbytes)
        eng.h2d(d_pk, pk)
        h_pk = eng.pinned("bench_rows_pk", pk.nbytes).view(np.uint32, pk.shape)
        h_pk[:] = pk
        outl = outlier_section(eng, enc, base, flat, d_pk, d_proba, d_label, h_pk, nums, K, W, bool(info0["packed_ok"]))
        eng.device_free(d_pk)

    # ---- cpu baseline (rank 0, N=1 only): bounded sample = the same 65 536-row batch the plugin e2e scores
    cpu = None
    if dist.rank == 0 and dist.world == 1 and not args.no_cpu:
        import sklearn

        kind = MODELS[args.model][0]
        cores = os.cpu_count() or 1
        procs = reference_procs(kind)
        best, med, times = cpu_reference_rate(pipe, df0, 5, procs)
        one_best, _, _ = cpu_reference_rate(pipe, df0.iloc[:16384], 2, 1) if procs > 1 else (best, None, None)
        port = cpu_port_rate(pipe, pc, pn, 5)
        cpu = {
            "value": med, "unit": "rows/s", "cores": cores if procs == 1 else procs, "kind": "reference",
            "sample": (f"5 x the {BATCH}-row cfg2 DataFrame through sklearn {sklearn.__version__} Pipeline.predict_proba, "
                       f"{'n_jobs=-1 threads' if procs == 1 else str(procs) + ' forked processes'}; median"),
            "best": best, "single_process": one_best,
            "port_openmp_rows_per_s": port, "host_cores": cores, "cpu_quota": cpu_bandwidth(),
        }

    avg_launch_ms = ms_total_max / K  # the kernel is the only work of the timed region: region time / launches
    achieved = ALG_BYTES_PER_ROW * BATCH / (avg_launch_ms * 1e-3) / 1e9
    peak, peak_src = measured_peak_gbs()
    line = {
        "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": dist.world, "steps": K, "warmup": W,
        "ms_per_step": ms_total_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16 ranks + f64acc" if fmt == _cabi.ROWS_RANKED else "f32cmp+f64acc", "data": "synthetic",
        "config": {
            "workload": workload_label(args.model),
            "forest": args.model, "trees": info0["n_trees"], "depth": info0["max_depth"], "nodes": flat.total_nodes, "batch": BATCH,
            "parallelism": f"dp{dist.world} (rows sharded, forest replicated, no collective)",
            "l2": f"inputs rotate over {POOL} distinct batches ({POOL * BATCH * row_bytes / 1e6:.0f} MB of rows + {POOL * BATCH * 8 / 1e6:.0f} MB of results > 126 MB L2)",
            "walk": info0["walk"], "row_format": f"{fmt_name}: {row_bytes}-byte encoded rows",
            "kernel": kernel_used,
        },
        "e2e": {"value": plugin_value, "unit": "rows/s", "h2d_bytes_per_step": BATCH * {2: info0["rank_row_bytes"], 1: 64, 0: 96}[(breakdown or {}).get("row_format", 1)],
                "d2h_bytes_per_step": BATCH * 8, "ms_per_step": 1e3 * dist.max(plugin_s) / K,
                "p50_ms": 1e3 * float(np.percentile(plat, 50)), "p99_ms": 1e3 * float(np.percentile(plat, 99)),
                "slowest_steps_ms": [round(1e3 * v, 3) for v in sorted(plat)[-5:]], "sum_of_steps_ms": 1e3 * float(np.sum(plat)),
                "api": "B200Model.predict(DataFrame of 9 string + 14 float64 columns) -> {'predictions': list[float], 'outliers': list, "
                       "'feature_drift_batch': dict}: the plugin call of reference app/main.py:72 (classifier only, like the reference arm)",
                "breakdown": breakdown, "parity_max_abs_dp_vs_sklearn_2048rows": plugin_parity, "gpu_launches": int(launches_plugin),
                "warmup_calls": plugin_warmup, "process_bound_to_gpu_node_cpus": bound_cpus},
        "e2e_c_abi": {"value": cabi_value, "unit": "rows/s", "h2d_bytes_per_step": BATCH * row_bytes, "d2h_bytes_per_step": BATCH * 8,
                      "ms_per_step": 1e3 * dist.max(cabi_s) / K, "p50_ms": 1e3 * float(np.percentile(lat, 50)), "p99_ms": 1e3 * float(np.percentile(lat, 99)),
                      "api": f"b2f_predict_pairs(pre-encoded {row_bytes}-byte rows in pinned host memory) -> {{float32 proba, int32 label}} per row",
                      "parity_max_abs_dp_vs_device_path": cabi_parity, "gpu_launches": int(launches_cabi),
                      "pipelined_2_in_flight": {"value": pipe_value, "unit": "rows/s", "api": "b2f_predict_async_ex + b2f_wait, two batches in flight"},
                      "pcie_h2d_gbs_one_batch": h2d_gbs},
        "gpu_launches": int(launches_value),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": ncu_traffic(args.model), "peak_source": peak_src, "kernel": kernel_used,
                     "alg_bytes_per_launch": ALG_BYTES_PER_ROW * BATCH, "avg_launch_ms": avg_launch_ms,
                     "how": "timed region / launches (back-to-back launches overlap head and tail: programmatic dependent launch)",
                     "isolated_launch_ms": float(np.mean(iso_ms)), "isolated_launch_min_ms": float(np.min(iso_ms)),
                     "actual_bytes_per_launch": BATCH * (row_bytes + 8)},
        "clocks": clocks,
        "sustained_rows_per_s": sustained,
        "parity_max_abs_dp_vs_sklearn_2048rows_all_ranks": parity, "parity_labels_equal_all_ranks": labels_equal,
    }
    if dist.rank == 0 and dist.world == 1 and not args.no_sweep:  # single-process runs only (the sweep fits / loads its own models)
        line["latency_sweep"] = {m: latency_sweep(args, dist, m, full=args.sweep) for m in (["rf500d8", "gbdt500d8"] if not args.sweep_model else [args.sweep_model])}
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if mom is not None:
        line["cfg5_moments"] = mom
    if outl is not None:
        line["outlier_forest"] = outl
    if dist.rank == 0 and dist.world == 1 and not args.no_drift:
        line["drift_detector"] = drift_section(base, flat, dist.local_rank)
    for d in (d_rows, d_proba, d_label):
        eng.device_free(d)
    model.close()
    if dist.rank == 0 and dist.world == 1 and not args.no_stream:
        from databricks_kubernetes_mlops_poc_b200.engine import device_count

        if device_count() > 1:  # config 4 inside the default single-process run when the box shows several GPUs
            line["cfg4_stream"] = stream_leg(args, pipe, base, flat, rows_total=args.stream_rows, sustain=1.0)
    if outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
        print(f"[bench] wrote {', '.join(f'{n}.npy' for n in outputs)} to {args.dump_outputs}", file=sys.stderr)
    if dist.rank == 0:
        emit(line)


def outlier_section(eng, enc, base, flat, d_rows, d_proba, d_label, h_rows, nums, K, W, packed):
    """IsolationForest(100) fitted as the reference fits it (02-register-model.ipynb:232-233, on the curated table's 14
    numerics): kernel-only rate of the isolation-forest walk on the resident pool, the end-to-end rate of
    b2f_predict_full (classifier + outlier forest on ONE H2D copy of the rows, 24-byte records back), sklearn's own
    decision_function on the host beside it, and a flag / score parity spot check."""
    from sklearn.ensemble import IsolationForest

    from databricks_kubernetes_mlops_poc_b200 import flatten
    from databricks_kubernetes_mlops_poc_b200._cabi import SCORED_FULL_DTYPE
    from databricks_kubernetes_mlops_poc_b200.engine import ForestEngine

    thr = 0.0  # the reference's 0.95 can never fire (score <= 0.5); 0.0 exercises both outcomes
    iso = IsolationForest(n_estimators=100, random_state=0).fit(base[list(flat.num_features)].to_numpy())
    blob = flatten.flatten_isolation_forest(iso, len(flat.cat_features), len(flat.num_features), threshold=thr)
    alone = ForestEngine(blob, eng.device)
    alone.predict_stream_timed(d_rows, BATCH, POOL, d_proba, False, d_label, W, packed=packed)
    ms_each, ms_total = alone.predict_stream_timed(d_rows, BATCH, POOL, d_proba, False, d_label, K, packed=packed)
    got_s = np.empty(BATCH, dtype=np.float32)
    got_f = np.empty(BATCH, dtype=np.int32)
    alone.d2h(got_s, d_proba)
    alone.d2h(got_f, d_label)
    info = alone.info()
    alone.close()
    x = nums[:BATCH].astype(np.float64)
    # parity sample: complete rows only -- the reference's detector refuses NaN (sklearn 1.1.1), the installed sklearn
    # routes it by a per-node random flag, the kernel sends it to the second child (flatten_isolation_forest)
    sel = np.nonzero(~np.isnan(x).any(axis=1))[0][:2048]
    t0 = time.perf_counter()
    iso.decision_function(x[:16384])
    cpu_s = time.perf_counter() - t0
    want_sel = -iso.decision_function(x[sel])

    eng.attach_outlier_forest(blob)
    h_full = eng.pinned("bench_full", BATCH * POOL * 24).view(SCORED_FULL_DTYPE, (BATCH * POOL,))
    for i in range(W):
        b = i % POOL
        eng.predict_full(h_rows[b * BATCH:(b + 1) * BATCH], out=h_full[b * BATCH:(b + 1) * BATCH])
    t0 = time.perf_counter()
    for i in range(K):
        b = i % POOL
        eng.predict_full(h_rows[b * BATCH:(b + 1) * BATCH], out=h_full[b * BATCH:(b + 1) * BATCH])
    full_s = time.perf_counter() - t0
    return {
        "detector": "IsolationForest(n_estimators=100, max_samples=256) on the 14 numerics, score = -decision_function, flag = score > 0.0",
        "trees": info["n_trees"], "max_depth": info["max_depth"], "walk": info["walk"],
        "kernel_rows_per_s": BATCH * K / (ms_total * 1e-3), "kernel_avg_launch_ms": float(np.mean(ms_each)),
        "e2e_full_rows_per_s": BATCH * K / full_s, "e2e_full_ms_per_step": 1e3 * full_s / K,
        "e2e_api": "b2f_predict_full(host pinned rows) -> {f64 proba, i32 label, i32 is_outlier, f32 score} per row",
        "d2h_bytes_per_step": BATCH * 24,
        "cpu_sklearn_rows_per_s": 16384 / cpu_s, "cpu_sample": "IsolationForest.decision_function on 16384 rows, sklearn default threading",
        "parity_max_abs_dscore_2048_complete_rows": float(np.abs(got_s[sel].astype(np.float64) - want_sel).max()),
        "parity_flags_equal_2048_complete_rows": bool((got_f[sel] == (want_sel > thr)).all()),
        "parity_full_vs_alone_flags_equal": bool((h_full["is_outlier"][:BATCH] == got_f).all()),
    }


def drift_section(base, flat, device):
    """K3 (SURVEY a7): per-request drift scores against the 30 000-row reference table -- chi-squared on the 9
    categoricals, exact two-sample K-S on the 14 numerics -- on the GPU, with the scipy path the reference runs
    (restated in oracle/drift.py) timed on this box's host beside it for request-sized batches."""
    from databricks_kubernetes_mlops_poc_b200.drift import TabularDrift
    from oracle import drift as od

    feats = flat.all_features
    ref = base[feats]
    det = TabularDrift(ref, flat.cat_features, device=device)
    rng = np.random.default_rng(DATA_SEED + 7)
    rows = []
    for n in (1, 16, 128, 1000, 65536):  # closed form; row scan in shared memory (2..448 rows); sweep
        batch = ref.iloc[rng.integers(0, len(ref), n)].reset_index(drop=True)
        got = det.p_values(batch)  # warm-up + parity sample
        dev, wall = [], []
        for _ in range(10 if n < 65536 else 3):
            t0 = time.perf_counter()
            det.statistics(batch)
            wall.append(time.perf_counter() - t0)
            dev.append(det.last_device_ms)
        row = {"batch": n, "device_ms": float(np.median(dev)), "call_ms": 1e3 * float(np.median(wall))}
        if n <= 1000:
            t0 = time.perf_counter()
            want = od.tabular_drift_p_values(ref, batch, flat.cat_features)
            row["cpu_scipy_ms"] = 1e3 * (time.perf_counter() - t0)
            row["parity_max_abs_dp"] = float(np.abs(got.astype(np.float64) - want.astype(np.float64)).max())
        rows.append(row)
    launches = det.launches
    det.close()
    return {"reference_rows": len(ref), "features": "9 categorical (chi-squared) + 14 numeric (exact two-sample K-S)",
            "api": "b2f_drift_score (H2D of the batch columns + k_drift_count + k_drift_finish + D2H of 23 p-values)",
            "gpu_launches": int(launches), "by_batch": rows}


def latency_sweep(args, dist: Dist, name: str, full: bool = False):
    """BASELINE config 3: batch in {1, 16, 256, 4096, 65536}, 500-tree depth-8 model; p50 / p99 of the C-ABI
    call (pinned host buffers, H2D + kernel + D2H inside) and of the plugin call model.predict(DataFrame) -> dict.
    The default run takes a compact form of it (fewer calls per size); ``--sweep`` the 1000-call form and, for the
    RandomForest, the whole CustomModel.predict (outlier forest + drift detector attached)."""
    from databricks_kubernetes_mlops_poc_b200 import flatten, training
    from databricks_kubernetes_mlops_poc_b200._cabi import SCORED_DTYPE
    from databricks_kubernetes_mlops_poc_b200.model import B200Model
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES

    pipe, base = get_pipeline(name, dist)
    model = B200Model(flatten.flatten_pipeline(pipe), devices=[dist.local_rank], host_threads=host_thread_share(dist))
    eng, enc = model.engine, model.encoder
    n_max = 65536
    vocabs, codes, nums = training.synth_arrays(base, n_max, DATA_SEED + 1)
    from databricks_kubernetes_mlops_poc_b200.engine import STREAMED_RANK_MIN_ROWS

    pk64 = eng.pinned("sweep_rows", n_max * 64).view(np.uint32, (n_max, 16))
    enc.encode_arrays_packed(codes, nums, out=pk64)
    inf0 = eng.info()
    rk = None
    if inf0["rank_ok"]:  # ranked 32-byte rows: every size when the rank layout is resident, the large sizes when it streams
        words = enc.ranked_row_words
        rk = eng.pinned("sweep_rows_rk", n_max * words * 4).view(np.uint32, (n_max, words))
        enc.rank_rows(enc.encode_arrays(codes, nums), out=rk)
    rank_from = (STREAMED_RANK_MIN_ROWS if inf0["rank_stream"] else 0) if rk is not None else n_max + 1
    out = eng.pinned("sweep_out", n_max * 8).view(SCORED_DTYPE, (n_max,))
    df_all = training.arrays_to_frame(vocabs, codes, nums)[ALL_FEATURES]
    # parity of the plugin call at every sweep size against the library (float64 outputs)
    want_all = pipe.predict_proba(df_all.iloc[:4096])[:, 1]
    res = {}
    parity = 0.0
    for n in (1, 16, 256, 4096, 65536):
        calls = (1000 if n <= 4096 else 200) if full else (200 if n <= 4096 else 50)
        pk = rk if n >= rank_from else pk64
        for _ in range(20):
            eng.predict_pairs(pk[:n], out=out[:n])
        ts = np.empty(calls)
        for i in range(calls):
            t0 = time.perf_counter()
            eng.predict_pairs(pk[:n], out=out[:n])
            ts[i] = time.perf_counter() - t0
        df = df_all.iloc[:n]
        pcalls = (200 if n <= 4096 else 20) if full else (50 if n <= 4096 else 20)
        for _ in range(3):
            got = model.predict(df)
        m = min(n, 4096)
        parity = max(parity, float(np.abs(np.asarray(got["predictions"])[:m] - want_all[:m]).max()))
        tp = np.empty(pcalls)
        for i in range(pcalls):
            t0 = time.perf_counter()
            model.predict(df)
            tp[i] = time.perf_counter() - t0
        res[str(n)] = {"c_abi_p50_us": 1e6 * float(np.percentile(ts, 50)), "c_abi_p99_us": 1e6 * float(np.percentile(ts, 99)),
                       "predict_p50_us": 1e6 * float(np.percentile(tp, 50)), "predict_p99_us": 1e6 * float(np.percentile(tp, 99)),
                       "calls": calls, "predict_calls": pcalls}
    info = eng.info()
    model.close()
    if full and MODELS[name][0] == "rf":
        # the whole CustomModel.predict replacement: classifier + outlier forest (one pass) + drift detector, all on the GPU
        from sklearn.ensemble import IsolationForest

        iso = IsolationForest(n_estimators=100, random_state=0).fit(base[list(model.numeric_features)].to_numpy())
        fullm = B200Model.from_pipeline(pipe, reference_frame=base, outlier=iso, outlier_threshold=0.95, devices=[dist.local_rank])
        # the reference's outlier detector refuses NaN numerics (sklearn 1.1.1 -> HTTP 500), so this leg scores complete rows
        df_complete = df_all.iloc[:4096].copy()
        for col in model.numeric_features:
            df_complete[col] = df_complete[col].fillna(float(base[col].median()))
        for n in (1, 16, 256, 4096):
            df = df_complete.iloc[:n]
            for _ in range(3):
                fullm.predict(df)
            tp = np.empty(100)
            for i in range(100):
                t0 = time.perf_counter()
                fullm.predict(df)
                tp[i] = time.perf_counter() - t0
            res[str(n)]["predict_full_p50_us"] = 1e6 * float(np.percentile(tp, 50))
            res[str(n)]["predict_full_p99_us"] = 1e6 * float(np.percentile(tp, 99))
        fullm.close()
    return {"model": name, "walk": info["walk"], "tile_resident": info["tile_resident"], "rank_ok": info["rank_ok"], "rank_stream": info["rank_stream"],
            "row_bytes_by_batch": {str(n): int((rk if n >= rank_from else pk64).shape[1] * 4) for n in (1, 16, 256, 4096, 65536)},
            "split_max_rows": info["split_max_rows"],
            "parity_max_abs_dp_vs_sklearn": parity,
            "api": "C ABI: b2f_predict_pairs on pinned pre-encoded rows; plugin: B200Model.predict(DataFrame) -> dict, classifier only "
                   "(predict_*)" + ("; predict_full_*: with the outlier forest + drift detector attached (the whole CustomModel.predict)" if full else ""),
            "batches": res}


def run_cfg1(args):
    """BASELINE config 1: the reference's own CPU path on 1 000 rows of the reference's curated.csv (frozen copy
    under tests/golden), single process, n_jobs=-1 as the reference sets it; classifier alone and the whole
    CustomModel.predict restatement (classifier + drift + outliers).  No GPU involved."""
    import sklearn

    from oracle import datasets
    from oracle import reference_pipeline as rp
    from oracle.custom_model import ReferenceCustomModel

    cur = datasets.load_curated()
    df = cur[rp.FEATURES].iloc[:1000]
    out = {"rows": 1000, "cores": os.cpu_count(), "sklearn": sklearn.__version__, "models": {}}
    for name, params in rp.PINNED_RF.items():
        pipe = rp.fit_reference_pipeline(cur, params)
        ts = []
        for _ in range(6):
            t0 = time.perf_counter()
            pipe.predict_proba(df)
            ts.append(time.perf_counter() - t0)
        ts = ts[1:]
        entry = {"classifier_best_ms": 1e3 * min(ts), "classifier_median_ms": 1e3 * statistics.median(ts),
                 "classifier_rows_per_s": 1000 / min(ts)}
        if name == "rf100d6":
            cm = ReferenceCustomModel(pipe, cur)
            tt = []
            for _ in range(3):
                t0 = time.perf_counter()
                cm.predict(None, df)
                tt.append(time.perf_counter() - t0)
            entry["custom_model_predict_best_ms"] = 1e3 * min(tt)
        out["models"][name] = entry
    emit({"metric": "reference CPU predict() on 1k curated rows (config 1)", "impl": "reference", "unit": "ms", **out})


def stream_leg(args, pipe, base, flat, rows_total: int, sustain: float, ngpu: int = 0):
    """BASELINE config 4: ONE process deals a synthetic stream in 65 536-row batches round-robin over all GPUs of the box
    (forest replicated, rows independent, no inter-GPU traffic) through b2f_predict_stream (one host thread per GPU inside the C
    call, two batches in flight per GPU, pinned buffers placed on each GPU's NUMA node by slices)."""
    from databricks_kubernetes_mlops_poc_b200 import training
    from databricks_kubernetes_mlops_poc_b200.encode import RowEncoder
    from databricks_kubernetes_mlops_poc_b200.engine import EngineGroup, device_count
    from databricks_kubernetes_mlops_poc_b200.sharding import round_robin_batches

    enc = RowEncoder(flat)
    ngpu = min(ngpu, device_count()) if ngpu > 0 else device_count()
    group = EngineGroup(flat, devices=list(range(ngpu)))
    engines = group.engines
    total = rows_total
    vocabs, codes, nums = training.synth_arrays(base, total, DATA_SEED + 7)
    ranked = bool(engines[0].info()["rank_ok"])
    rows24 = enc.encode_arrays(codes, nums)
    enc_rows = enc.rank_rows(rows24) if ranked else enc.pack_rows(rows24)
    words = enc_rows.shape[1]
    # one pinned buffer each, striped by batch over the NUMA nodes of the GPUs the batches go to
    host = group.pinned_striped(np.uint32, (total, words), BATCH)
    host[:] = enc_rows
    proba = group.pinned_striped(np.float32, (total,), BATCH)
    label = group.pinned_striped(np.int32, (total,), BATCH)
    plan = list(round_robin_batches(total, BATCH, ngpu))
    rows_gpu = [sum(hi - lo for g, lo, hi in plan if g == d) for d in range(ngpu)]

    group.predict_stream(host, BATCH, proba, label)  # warm-up pass (allocations, first touch)
    sampler = ClockSampler(0)
    sampler.start()
    t0w = time.time()
    t0 = time.perf_counter()
    passes = 0
    while passes < 3 or time.perf_counter() - t0 < sustain:
        group.predict_stream(host, BATCH, proba, label)  # ONE C call: a host thread per GPU deals its batches
        passes += 1
    dt = (time.perf_counter() - t0) / passes
    t1w = time.time()
    sampler.stop()
    # parity spot check on the last pass: 1 024 rows against sklearn
    sel = np.arange(0, min(total, BATCH), 64)[:1024]
    df = training.arrays_to_frame(vocabs, codes[sel], nums[sel])
    want = pipe.predict_proba(df)[:, 1]
    err = float(np.abs(proba[sel].astype(np.float64) - want).max())
    launches = sum(e.info()["launches"] for e in engines)
    group.close()
    return {
        "metric": "rows/sec, synthetic stream dealt round-robin over the GPUs of one box by ONE process (config 4)", "unit": "rows/s",
        "value": total / dt, "n_gpus": ngpu, "rows": total, "batch": BATCH, "seconds": dt, "per_gpu_rows_per_s": [r / dt for r in rows_gpu],
        "higher_is_better": True, "scaling": "strong", "data": "synthetic", "dtype": "u16 ranks + f64acc" if ranked else "f32cmp+f64acc",
        "config": {"workload": f"cfg4: {args.model}, {total} rows in {len(plan)} batches of {BATCH}, one process, b2f_predict_stream (one host thread per "
                               f"GPU inside the C call, 2 batches in flight per GPU, pinned buffers), {words * 4}-byte rows",
                   "forest": args.model, "parallelism": f"round-robin over {ngpu} GPUs, forest replicated, no collective"},
        "e2e": {"value": total / dt, "unit": "rows/s", "h2d_bytes_per_step": BATCH * words * 4, "d2h_bytes_per_step": BATCH * 8},
        "gpu_launches": int(launches // (passes + 1)), "clocks": sampler.summary(t0w, t1w), "parity_max_abs_dp_vs_sklearn_1024rows": err,
        "roofline_frac_of_n_gpu_hbm": (total / dt) * ALG_BYTES_PER_ROW / 1e9 / (measured_peak_gbs()[0] * ngpu),
        "passes": passes,
    }


def run_stream(args):
    """--stream: config 4 on its own (10 M rows by default)."""
    from databricks_kubernetes_mlops_poc_b200 import flatten

    solo = Dist(1, use_cuda=False, solo=True)
    pipe, base = get_pipeline(args.model, solo)
    emit(stream_leg(args, pipe, base, flatten.flatten_pipeline(pipe), args.stream_rows, args.sustain, args.stream_gpus))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="gbdt100d6", choices=sorted(MODELS))
    ap.add_argument("--sustain", type=float, default=1.5, help="seconds of back-to-back launches for the clock record")
    ap.add_argument("--rows", default="ranked", choices=["ranked", "packed64", "words24"], help="encoded row layout fed to the engine")
    ap.add_argument("--sweep", action="store_true", help="config-3 latency sweep in its long form (1000 calls per size, whole CustomModel.predict leg)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the config-3 latency sweep")
    ap.add_argument("--sweep-model", default=None, choices=sorted(MODELS), help="sweep this model only (default: rf500d8 and gbdt500d8)")
    ap.add_argument("--no-stream", action="store_true", help="skip the config-4 stream leg (single-process runs on a multi-GPU box)")
    ap.add_argument("--no-gib", action="store_true", help="skip the >= 1 GiB run of the moments kernel")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-moments", action="store_true")
    ap.add_argument("--no-outliers", action="store_true", help="skip the K4 outlier-forest section")
    ap.add_argument("--no-drift", action="store_true", help="skip the K3 drift-detector section")
    ap.add_argument("--cfg1", action="store_true", help="config 1: the reference CPU path on 1k curated rows (no GPU)")
    ap.add_argument("--stream", action="store_true", help="config 4: one process, 10M-row stream round-robin over all GPUs")
    ap.add_argument("--stream-rows", type=int, default=10_000_000)
    ap.add_argument("--quick", action="store_true", help="only the timed value / e2e legs (no sweep, stream, cpu baseline, outliers, drift)")
    ap.add_argument("--stream-gpus", type=int, default=0, help="GPUs used by --stream (0 = all visible)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (rank 0; see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.quick:
        args.no_sweep = args.no_stream = args.no_cpu = args.no_outliers = args.no_drift = args.no_gib = True

    if args.cfg1:
        run_cfg1(args)
        return
    if args.stream:
        run_stream(args)
        return
    if args.impl == "reference":
        # under torchrun only rank 0 works; the other ranks exit 0 without joining anything
        if int(os.environ.get("RANK", "0")) == 0:
            run_reference(args, Dist(args.gpus, use_cuda=False, solo=True))
        return
    dist = Dist(args.gpus, use_cuda=True)
    try:
        run_b200(args, dist)
    finally:
        dist.close()


if __name__ == "__main__":
    main()

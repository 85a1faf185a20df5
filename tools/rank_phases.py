"""Where the time of a back-to-back step of k_forest_predict_rank goes, phase by phase.

Builds a copy of the engine with B2F_RANK_TRACE (thread 0 of every CTA records its SM and %globaltimer at entry, forest
landed, griddepcontrol.wait returned, rows staged, walk done, exit) into a temporary directory, then runs the loop of
bench.py's `value`: GBDT 100 x d6, ranked rows, a pool of 32 batches of 65 536 rows, back-to-back launches without events in
between.  Per CTA it takes the time of each phase, and per SM the gap between a CTA's exit and the walk start of the next
launch's CTA on the same SM; it writes median / p10 / p90 of each (microseconds) under --label in the --out JSON file.

usage: python tools/rank_phases.py --label parent|result [--out profiles/r03_rank_phases.json] [--steps 200] [--warmup 10]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CSRC = os.path.join(ROOT, "databricks_kubernetes_mlops_poc_b200", "csrc")
WORDS = 8  # B2F_RANK_TRACE_WORDS
SMID, ENTRY, FOREST, WAIT, STAGED, WALKED, EXIT = range(7)  # forest_predict_rank.cuh RT_*


def build_traced(tmp: str) -> str:
    so = os.path.join(tmp, "libb200forest.so")
    t0 = time.time()
    subprocess.check_call(["make", "-s", "-C", CSRC, so, f"OUT={so}", f"HOSTOBJ={os.path.join(tmp, 'host_simd.o')}",
                           "B2F_DEFINES=-DB2F_RANK_TRACE"], stdout=subprocess.DEVNULL)
    print(f"[rank_phases] traced build in {time.time() - t0:.0f}s", file=sys.stderr)
    return so


def stats(x) -> dict:
    x = np.asarray(x, dtype=np.float64)
    return {"median_us": float(np.median(x)), "p10_us": float(np.percentile(x, 10)), "p90_us": float(np.percentile(x, 90)), "n": int(x.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--label", required=True)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_rank_phases.json"))
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    args = ap.parse_args()

    import ctypes as C

    import bench
    from databricks_kubernetes_mlops_poc_b200 import _cabi, flatten
    from databricks_kubernetes_mlops_poc_b200.encode import RowEncoder

    tmp = tempfile.mkdtemp(prefix="b2f_rank_trace_")
    _cabi.LIB_PATH = build_traced(tmp)
    from databricks_kubernetes_mlops_poc_b200.engine import ForestEngine

    lib = _cabi.load_library()
    lib.b2f_rank_trace_read.restype = C.c_int64
    lib.b2f_rank_trace_read.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]

    d = bench.Dist(1, use_cuda=False, solo=True)
    pipe, base = bench.get_pipeline("gbdt100d6", d)
    flat = flatten.flatten_pipeline(pipe)
    enc = RowEncoder(flat)
    _, _, _, rows24 = bench.make_batches(base, enc, bench.POOL, bench.DATA_SEED)
    rows = enc.rank_rows(rows24)
    B, P = bench.BATCH, bench.POOL
    eng = ForestEngine(flat, 0)
    d_rows = eng.device_alloc(rows.nbytes)
    d_p = eng.device_alloc(P * B * 4)
    d_l = eng.device_alloc(P * B * 4)
    eng.h2d(d_rows, rows)
    eng.predict_stream_timed(d_rows, B, P, d_p, False, d_l, args.warmup, fmt=_cabi.ROWS_RANKED, per_launch=False)
    _, ms_total = eng.predict_stream_timed(d_rows, B, P, d_p, False, d_l, args.steps, fmt=_cabi.ROWS_RANKED, per_launch=False)

    slots, ctas = C.c_int32(0), C.c_int32(0)
    n_sm = eng.info()["sm_count"]
    buf = np.zeros(256 * n_sm * WORDS, dtype=np.uint64)
    launches = lib.b2f_rank_trace_read(eng._h, buf.ctypes.data, C.byref(slots), C.byref(ctas))
    if launches < 0:
        raise RuntimeError("b2f_rank_trace_read failed")
    steps = min(args.steps, slots.value)
    ring = buf.reshape(slots.value, ctas.value, WORDS)
    recs = np.stack([ring[i % slots.value] for i in range(launches - steps, launches)])  # (steps, ctas, WORDS)
    grid = min(ctas.value, (B + 31) // 32)
    recs = recs[:, :grid].astype(np.int64)
    t = recs[..., :EXIT + 1].astype(np.float64) / 1e3  # ns -> us
    ph = {
        "entry_to_wait_returned": t[..., WAIT] - t[..., ENTRY],
        "entry_to_rows_staged": t[..., STAGED] - t[..., ENTRY],
        "rows_staged_to_forest_landed": t[..., FOREST] - t[..., STAGED],
        "walk": t[..., WALKED] - t[..., FOREST],
        "walk_done_to_exit": t[..., EXIT] - t[..., WALKED],
        "cta_entry_to_exit": t[..., EXIT] - t[..., ENTRY],
    }
    # the next launch's CTA on the same SM: exit of launch i -> walk start (forest landed, rows staged) of launch i + 1
    gaps, overlap = [], []
    for i in range(steps - 1):
        nxt = {int(s): k for k, s in enumerate(recs[i + 1, :, SMID])}
        for k in range(grid):
            j = nxt.get(int(recs[i, k, SMID]))
            if j is not None:
                gaps.append(t[i + 1, j, FOREST] - t[i, k, EXIT])
                overlap.append(t[i, k, EXIT] - t[i + 1, j, ENTRY])
    starts = t[:, :, ENTRY].min(axis=1)
    stamps = np.sort(np.unique(recs[..., ENTRY:EXIT + 1]))
    res = {
        "workload": f"GBDT 100 x d6, ranked rows, {P} x {B} rows pool, {args.steps} back-to-back launches after {args.warmup}",
        "us_per_step_cuda_events": ms_total * 1e3 / args.steps,
        "us_per_step_first_entry_to_first_entry": stats(np.diff(starts)),
        "ctas_per_launch": grid,
        "globaltimer_resolution_ns": int(np.diff(stamps)[np.diff(stamps) > 0].min()) if stamps.size > 1 else None,
        "phases": {k: stats(v) for k, v in ph.items()},
        "exit_to_next_launch_walk_start_same_sm": stats(gaps),
        "next_launch_entry_before_exit_same_sm": stats(overlap),
    }
    eng.close()
    out = {}
    if os.path.exists(args.out):
        with open(args.out) as f:
            out = json.load(f)
    out[args.label] = res
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({args.label: res}, indent=1))


if __name__ == "__main__":
    main()

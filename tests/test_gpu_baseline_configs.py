"""GPU parity on BASELINE.json's OWN models and sizes (the bench's models, fitted by the bench's own recipe):
configs[1]  GBDT 100 x depth 6 at the full 65 536-row synthetic batch -- every kernel, every row format, float64 <= 1e-12 and
            labels exact on the WHOLE batch (not a sample);
configs[2]  GBDT 500 x depth 8 and RF 500 x depth 8 at the latency-sweep sizes {1, 16, 256, 4096, 65536}."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOL64 = 1e-12
TOL32 = 2e-7


@pytest.fixture(scope="module")
def bench_mod():
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench

    return bench


def _model(bench_mod, name):
    pipe, base = bench_mod.get_pipeline(name, bench_mod.Dist(1, use_cuda=False, solo=True))
    return pipe, base


def _synthetic(bench_mod, base, n, seed):
    from databricks_kubernetes_mlops_poc_b200 import training
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES

    vocabs, codes, nums = training.synth_arrays(base, n, seed)
    return codes, nums, training.arrays_to_frame(vocabs, codes, nums)[ALL_FEATURES]


def _engine_with(flat, **env):
    from databricks_kubernetes_mlops_poc_b200.engine import ForestEngine

    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        return ForestEngine(flat, 0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def test_cfg2_gbdt100d6_full_batch_every_kernel_and_format(bench_mod):
    from databricks_kubernetes_mlops_poc_b200 import flatten
    from databricks_kubernetes_mlops_poc_b200.encode import RowEncoder

    pipe, base = _model(bench_mod, "gbdt100d6")
    codes, nums, df = _synthetic(bench_mod, base, bench_mod.BATCH, bench_mod.DATA_SEED)
    want_p = pipe.predict_proba(df)[:, 1]
    want_l = pipe.predict(df)
    flat = flatten.flatten_pipeline(pipe)
    enc = RowEncoder(flat)
    rows24 = enc.encode_arrays(codes, nums)
    formats = {"words24": rows24, "packed64": enc.pack_rows(rows24), "ranked": enc.rank_rows(rows24)}
    assert np.array_equal(enc.encode_frame_ranked(df), formats["ranked"])  # DataFrame -> ranked rows == arrays -> ranked rows
    seen = set()
    for kernel in ("warp", "tile", "split", "auto"):
        eng = _engine_with(flat, **({"B2F_KERNEL": kernel} if kernel != "auto" else {}))
        try:
            for name, rows in formats.items():
                i0 = eng.info()
                n = 4096 if kernel == "split" else len(rows)  # the latency kernel launches one CTA per two rows
                p64, l64 = eng.predict_rows(rows[:n], np.float64)
                assert np.abs(p64 - want_p[:n]).max() <= TOL64, (kernel, name)
                assert (l64 == want_l[:n]).all(), (kernel, name)
                p32, l32 = eng.predict_rows(rows[:n], np.float32)
                assert np.abs(p32.astype(np.float64) - want_p[:n]).max() <= TOL32 and (l32 == want_l[:n]).all(), (kernel, name)
                i1 = eng.info()
                for k in ("launches_rank", "launches_tile", "launches_split"):
                    if i1[k] > i0[k]:
                        seen.add(k)
                if i1["launches"] - i0["launches"] > (i1["launches_rank"] - i0["launches_rank"]) + (i1["launches_tile"] - i0["launches_tile"]) + (
                        i1["launches_split"] - i0["launches_split"]):
                    seen.add("launches_warp")
        finally:
            eng.close()
    assert seen == {"launches_rank", "launches_tile", "launches_split", "launches_warp"}, seen


@pytest.mark.parametrize("name", ["rf500d8", "gbdt500d8"])
def test_cfg3_500d8_at_the_sweep_sizes(bench_mod, name):
    from databricks_kubernetes_mlops_poc_b200 import flatten
    from databricks_kubernetes_mlops_poc_b200.encode import RowEncoder
    from databricks_kubernetes_mlops_poc_b200.engine import ForestEngine
    from databricks_kubernetes_mlops_poc_b200.model import B200Model

    pipe, base = _model(bench_mod, name)
    codes, nums, df = _synthetic(bench_mod, base, 65536, bench_mod.DATA_SEED + 1)
    want_p = pipe.predict_proba(df)[:, 1]
    want_l = pipe.predict(df)
    flat = flatten.flatten_pipeline(pipe)
    enc = RowEncoder(flat)
    rows24 = enc.encode_arrays(codes, nums)
    pk = enc.pack_rows(rows24)
    eng = ForestEngine(flat, 0)
    try:
        info = eng.info()
        assert info["rank_ok"] and info["rank_stream"], "500 x depth-8: the rank layout (1.5 MB) streams through shared memory"
        rk = enc.rank_rows(rows24)
        for n in (1, 16, 256, 4096, 65536):
            for rows in (rows24, pk, rk):
                p, l = eng.predict_rows(rows[:n], np.float64)
                assert np.abs(p - want_p[:n]).max() <= TOL64 and (l == want_l[:n]).all(), (name, n, rows.shape[1])
    finally:
        eng.close()
    model = B200Model(flat, devices=[0])
    try:
        for n in (1, 16, 256, 4096, 65536):
            out = model.predict(df.iloc[:n])
            assert np.abs(np.asarray(out["predictions"]) - want_p[:n]).max() <= TOL64, (name, n)
    finally:
        model.close()


def test_bench_dumps_the_last_timed_step(bench_mod, tmp_path):
    """`bench.py --steps K --dump-outputs DIR`: K timed launches, and the dumped arrays are what the last of them (pool batch
    (K - 1) % POOL) and the plugin path's last call returned -- each equal to sklearn on its own rows."""
    from databricks_kubernetes_mlops_poc_b200 import training
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES

    K = 35  # the last launch scores pool batch 2, not batch 0
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--quick", "--no-moments", "--steps", str(K), "--warmup", "3",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=1800)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == K and line["gpu_launches"] == K
    assert sorted(os.listdir(tmp_path)) == ["e2e_predictions.npy", "value_label.npy", "value_proba1.npy"]
    proba, label, e2e = (np.load(tmp_path / f"{n}.npy") for n in ("value_proba1", "value_label", "e2e_predictions"))
    assert proba.dtype == label.dtype == np.float32 and e2e.dtype == np.float64
    assert proba.shape == label.shape == e2e.shape == (bench_mod.BATCH,)

    pipe, base = _model(bench_mod, "gbdt100d6")
    last = (K - 1) % bench_mod.POOL
    vocabs, codes, nums = training.synth_arrays(base, bench_mod.POOL * bench_mod.BATCH, bench_mod.DATA_SEED)
    rows = slice(last * bench_mod.BATCH, (last + 1) * bench_mod.BATCH)
    df = training.arrays_to_frame(vocabs, codes[rows], nums[rows])[ALL_FEATURES]
    assert np.abs(proba.astype(np.float64) - pipe.predict_proba(df)[:, 1]).max() <= TOL32
    assert (label == pipe.predict(df)).all()
    _, _, df0 = _synthetic(bench_mod, base, bench_mod.BATCH, bench_mod.DATA_SEED)
    assert np.abs(e2e - pipe.predict_proba(df0)[:, 1]).max() <= TOL64

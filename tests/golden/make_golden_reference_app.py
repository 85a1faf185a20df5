#!/usr/bin/env python
"""Record what the reference's unmodified ``app/main.py`` does on the project's ``mlflow`` shim into ``reference_app.json``.

The reference app is imported as it is, with ``databricks_kubernetes_mlops_poc_b200/shim`` ahead on the path, so its
``mlflow.pyfunc.load_model`` call lands in ``databricks_kubernetes_mlops_poc_b200.load_model``.  That is replaced by
``StubModel``, whose outputs are a fixed function of the rows it is given.  For every body of ``request_bodies`` the
file keeps the HTTP status and, for a 200, the response, the frame the app handed to ``predict`` and its two JSON log
records; and it keeps the path the app asked ``load_model`` for.  ``tests/test_server_cpu.py`` sends the same bodies to
the project's own app, built around the same stub, and compares.

Usage:  python tests/golden/make_golden_reference_app.py <checkout of the reference repository>
"""

from __future__ import annotations

import contextlib
import importlib
import json
import logging
import os
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
GOLDEN = os.path.join(HERE, "reference_app.json")
SHIM = os.path.join(ROOT, "databricks_kubernetes_mlops_poc_b200", "shim")
CURATED_ROWS = 80  # a body of this many curated rows is larger than ingest.NATIVE_MIN_BYTES: the native parser's path


def request_bodies(curated) -> list[tuple[str, bytes]]:
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES, sample_request

    return [
        ("sample_request", json.dumps(sample_request()).encode()),
        ("partial_rows", b'[{"credit_limit": 1250.0}, {}, {"sex": "female", "credit_limit": 333}]'),
        ("defaults_only", b"[{}]"),
        ("coercions", b'[{"age": "41", "credit_limit": 5100, "unknown_key": 1}, {"age": true, "education": ""}]'),
        ("numbers", b'[{"bill_amount_1": 1e3, "bill_amount_2": -1.5E-3, "payment_amount_6": -0.0, "credit_limit": 0.30000000000000004}]'),
        ("wrong_type", b'[{"sex": 3}]'),
        ("not_a_list", b'{"sex": "male"}'),
        ("empty_list", b"[]"),
        ("curated_rows", json.dumps(curated[ALL_FEATURES].iloc[:CURATED_ROWS].to_dict(orient="records")).encode()),
    ]


def frame_record(df) -> dict:
    return {"columns": [str(c) for c in df.columns], "dtypes": [str(t) for t in df.dtypes],
            "values": {str(c): df[c].tolist() for c in df.columns}}


class StubModel:
    """Stands in for the GPU model behind both plugin shapes: ``predict(DataFrame) -> dict`` (what the reference app calls,
    its ``CustomModel.predict``) and ``score(DataFrame) -> (proba, flags)`` with ``drift.score`` (what the project's app
    calls).  P = (credit_limit mod 1000) / 1000, outlier = credit_limit > 5000, drift score i = (i + rows) / 1000."""

    def __init__(self):
        self.inputs = []
        self.drift = self._Drift()

    class _Drift:
        def score(self, df):
            return [0.001 * (i + len(df)) for i in range(len(df.columns))]

    def score(self, df):
        self.inputs.append(frame_record(df))
        x = df["credit_limit"].to_numpy(dtype=np.float64)
        return (x % 1000) / 1000.0, (x > 5000).astype(np.int32)

    def predict(self, df):
        if len(df.columns) == 0:
            raise KeyError("no columns")  # the reference's CustomModel indexes the feature columns
        proba, flags = self.score(df)
        return {"predictions": proba.tolist(), "outliers": flags.tolist(),
                "feature_drift_batch": dict(zip(df.columns, self.drift.score(df)))}


@contextlib.contextmanager
def captured_log_records():
    """The JSON log records (``InferenceData`` / ``ModelOutput``) the app writes through the root logger."""
    records = []

    class Sink(logging.Handler):
        def emit(self, record):
            msg = record.getMessage()
            if msg.startswith("{"):
                records.append(json.loads(msg))

    root, sink = logging.getLogger(), Sink(logging.INFO)
    level = root.level
    root.addHandler(sink)
    root.setLevel(logging.INFO)
    try:
        yield records
    finally:
        root.removeHandler(sink)
        root.setLevel(level)


def replay(client, bodies, model: StubModel, records: list) -> list[dict]:
    """POST each body in turn; -> one dict per body: status, and for a 200 the response, the model's input frame and the
    log records (request id left out: it is random)."""
    out = []
    for name, body in bodies:
        model.inputs.clear()
        n0 = len(records)
        r = client.post("/predict", content=body, headers={"content-type": "application/json"})
        case = {"name": name, "status": r.status_code}
        if r.status_code == 200:
            deadline = time.monotonic() + 10.0
            while len(records) < n0 + 2 and time.monotonic() < deadline:  # the log records may be written off the request path
                time.sleep(0.01)
            logged = records[n0:n0 + 2]
            assert len(model.inputs) == 1 and len({rec.pop("request_id") for rec in logged}) == 1, name
            case.update(response=r.json(), model_input=model.inputs[0], logged={rec["type"]: rec for rec in logged})
        out.append(case)
    return out


def main() -> None:
    reference = sys.argv[1]
    sys.path.insert(0, ROOT)
    import databricks_kubernetes_mlops_poc_b200 as pkg
    from fastapi.testclient import TestClient

    from oracle import datasets

    for var in ("MODEL_DIRECTORY", "SERVICE_NAME"):
        os.environ.pop(var, None)
    sys.path[:0] = [os.path.join(reference, "app"), SHIM]  # the shim first: `import mlflow` must find it
    model, load_calls = StubModel(), []
    pkg.load_model = lambda path, **kw: (load_calls.append(path), model)[1]
    main_mod = importlib.import_module("main")
    assert main_mod.__file__.startswith(os.path.join(reference, "app"))
    assert sys.modules["mlflow"].__file__.startswith(SHIM)
    with captured_log_records() as records, TestClient(main_mod.app, raise_server_exceptions=False) as client:
        cases = replay(client, request_bodies(datasets.load_curated()), model, records)
    with open(GOLDEN, "w") as f:  # one case per line
        f.write('{"what": %s,\n "load_model_calls": %s,\n "cases": [\n  %s\n ]}\n' % (
            json.dumps(__doc__.split("\n\n")[0]), json.dumps(load_calls), ",\n  ".join(json.dumps(c) for c in cases)))
    print(GOLDEN, os.path.getsize(GOLDEN), [(c["name"], c["status"]) for c in cases])


if __name__ == "__main__":
    main()

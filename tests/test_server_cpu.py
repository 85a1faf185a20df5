"""HTTP surface with a stub scorer (CPU): status codes, schema, logging, cross-request batching.
Mirrors the behaviours probed on the unmodified reference app (SURVEY.md section 4)."""

import asyncio
import json
import logging

import numpy as np
import pytest
from fastapi.testclient import TestClient


class StubModel:
    """Deterministic scorer standing in for the GPU model: P = (credit_limit mod 1000) / 1000."""

    drift = None

    def __init__(self, fail=False):
        self.calls, self.fail = [], fail
        self.replicas = [self]

    def predict_proba1(self, df):
        if self.fail:
            raise RuntimeError("b2f_predict failed (rc=-2): CUDA error")
        self.calls.append(len(df))
        return (df["credit_limit"].to_numpy() % 1000) / 1000.0


def _client(model):
    from databricks_kubernetes_mlops_poc_b200.server import create_app

    return TestClient(create_app(model=model), raise_server_exceptions=False)


def test_predict_contract(caplog):
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES, sample_request

    m = StubModel()
    with caplog.at_level(logging.INFO), _client(m) as c:
        r = c.post("/predict", json=sample_request())  # the reference CI smoke test body
        assert r.status_code == 200
        body = r.json()
        assert set(body) == {"predictions", "outliers", "feature_drift_batch"}
        assert body["predictions"] == [0.0] and body["outliers"] == [0.0]  # int flags serialised as floats
        assert list(body["feature_drift_batch"]) == ALL_FEATURES
        r = c.post("/predict", json=[{"credit_limit": 1250.0}, {}, {"sex": "female", "credit_limit": 333}])
        assert r.status_code == 200 and r.json()["predictions"] == [0.25, 0.0, 0.333]
        assert c.post("/predict", json=[{}]).status_code == 200  # defaults make {} a valid row
        assert c.post("/predict", json=[{"sex": 3}]).status_code == 422
        assert c.post("/predict", json={"sex": "male"}).status_code == 422
        assert c.post("/predict", json=[]).status_code == 500  # as the reference (empty DataFrame)
        assert c.get("/").status_code == 200  # Swagger UI at the root
    import time

    time.sleep(0.2)  # log lines are produced off the request path
    recs = [json.loads(r.getMessage()) for r in caplog.records if r.getMessage().startswith("{")]
    kinds = [r["type"] for r in recs]
    assert "InferenceData" in kinds and "ModelOutput" in kinds
    inf = next(r for r in recs if r["type"] == "InferenceData")
    assert inf["service_name"] == "credit-default-api" and len(inf["request_id"]) == 32
    assert json.loads(inf["data"])[0]["sex"] == "male"  # data is a JSON *string* of records, as in the reference
    out = next(r for r in recs if r["type"] == "ModelOutput" and r["request_id"] == inf["request_id"])
    assert set(out["data"]) == {"predictions", "outliers", "feature_drift_batch"}


def test_outlier_flags_pass_through():
    """A replica with ``score`` (classifier + outlier forest in one pass) feeds the response's ``outliers``."""

    class Scoring(StubModel):
        def score(self, df):
            x = df["credit_limit"].to_numpy()
            return (x % 1000) / 1000.0, (x > 5000).astype(np.int32)

    with _client(Scoring()) as c:
        r = c.post("/predict", json=[{"credit_limit": 1250.0}, {"credit_limit": 9100.0}, {}])
        assert r.status_code == 200
        assert r.json()["predictions"] == [0.25, 0.1, 0.0] and r.json()["outliers"] == [0.0, 1.0, 1.0]  # {} = the schema defaults (credit_limit 18000)


def test_engine_failure_is_http_500():
    with _client(StubModel(fail=True)) as c:
        assert c.post("/predict", json=[{}]).status_code == 500


def test_concurrent_requests_share_batches():
    import pandas as pd

    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES, DEFAULTS
    from databricks_kubernetes_mlops_poc_b200.server import MicroBatcher

    m = StubModel()
    mb = MicroBatcher([m], max_rows=4096, window_us=20000)

    async def main():
        frames = [pd.DataFrame([{**DEFAULTS, "credit_limit": float(1000 * i + j)} for j in range(3)])[ALL_FEATURES] for i in range(40)]
        outs = await asyncio.gather(*[mb.score(f) for f in frames])
        for i, o in enumerate(outs):
            assert np.allclose(o[0], [0.0, 0.001, 0.002]) and o[1] is None
        return len(outs)

    try:
        assert asyncio.run(main()) == 40
    finally:
        mb.close()
    assert sum(m.calls) == 120 and len(m.calls) < 40  # requests were merged into fewer engine calls


def test_service_and_shim_match_the_recorded_reference_app(monkeypatch, curated):
    """SURVEY 8f rank 4: the reference's own app/main.py, run unmodified on the mlflow shim, was recorded into
    tests/golden/reference_app.json (make_golden_reference_app.py) with a stub scorer behind `load_model`.  The shim
    must serve the `load_model` call that app made, and the project's app, given the same stub and the same request
    bodies, must answer with the same statuses and responses, hand the model the same frames and log the same records."""
    import importlib.util
    import json
    import os
    import sys

    import databricks_kubernetes_mlops_poc_b200 as pkg
    from databricks_kubernetes_mlops_poc_b200.ingest import NATIVE_MIN_BYTES
    from databricks_kubernetes_mlops_poc_b200.server import create_app

    golden_dir = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    spec = importlib.util.spec_from_file_location("make_golden_reference_app", os.path.join(golden_dir, "make_golden_reference_app.py"))
    rec = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(rec)
    with open(rec.GOLDEN) as f:
        golden = json.load(f)
    bodies = rec.request_bodies(curated)
    assert [name for name, _ in bodies] == [c["name"] for c in golden["cases"]]
    assert len(bodies[-1][1]) > NATIVE_MIN_BYTES  # one body takes the native parser

    model, load_calls = rec.StubModel(), []
    monkeypatch.setattr(pkg, "load_model", lambda path, **kw: (load_calls.append(path), model)[1])
    for var in ("MODEL_DIRECTORY", "SERVICE_NAME"):
        monkeypatch.delenv(var, raising=False)

    monkeypatch.syspath_prepend(rec.SHIM)
    for name in [m for m in sys.modules if m == "mlflow" or m.startswith("mlflow.")]:
        monkeypatch.delitem(sys.modules, name)
    try:
        import mlflow

        assert mlflow.__file__.startswith(rec.SHIM)
        for path in golden["load_model_calls"]:
            assert mlflow.pyfunc.load_model(path) is model
        assert load_calls == golden["load_model_calls"]
    finally:
        for name in [m for m in sys.modules if m == "mlflow" or m.startswith("mlflow.")]:
            sys.modules.pop(name, None)

    load_calls.clear()
    with rec.captured_log_records() as records, TestClient(create_app(), raise_server_exceptions=False) as c:
        got = rec.replay(c, bodies, model, records)
    assert load_calls == golden["load_model_calls"]  # lifespan loads from the same default path
    for g, want in zip(got, golden["cases"]):
        assert g["status"] == want["status"], g["name"]
        if "response" in g:  # the reference's response model renders the 0 / 1 outlier flags as 0.0 / 1.0, the project as 0 / 1
            g["response"]["outliers"] = [float(v) for v in g["response"]["outliers"]]
        # everything else exactly, keys in order (json.dumps tells -0.0 from 0.0 and 1 from 1.0)
        assert json.dumps(g) == json.dumps(want), g["name"]


def test_one_pass_request_parsing_equals_the_model_validation():
    """parse_request (pydantic-core over the raw bytes into dict rows) accepts, rejects and coerces exactly like
    FastAPI's `data: list[LoanApplicant]` (json.loads + one model per row), and the docs keep the request schema."""
    from fastapi.exceptions import RequestValidationError
    from pydantic import TypeAdapter, ValidationError

    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES, DEFAULTS, LoanApplicant
    from databricks_kubernetes_mlops_poc_b200.server import create_app, parse_request, rows_to_frame

    model_rows = TypeAdapter(list[LoanApplicant])
    good = [
        b"[]", b"[{}]", b'[{"sex": "female", "age": 41}]', b'[{"age": "41", "credit_limit": 5, "unknown_key": 1}]',
        b'[{"bill_amount_1": 1e3, "education": ""}, {"payment_amount_6": -0.0}]', b'[{"age": true}]',
    ]
    for raw in good:
        want = model_rows.validate_json(raw)
        got = parse_request(raw)
        assert len(got) == len(want)
        if want:
            a, b = rows_to_frame(got), rows_to_frame(want)
            assert list(a.columns) == ALL_FEATURES and a.equals(b)
    assert rows_to_frame(parse_request(b"[{}]")).iloc[0].to_dict() == DEFAULTS
    bad = [b"", b"{", b'{"sex": "male"}', b'[{"sex": 3}]', b'[{"age": "old"}]', b"[1]", b'[{"age": null}]', b'[{"sex": null}]', b"null"]
    for raw in bad:
        with pytest.raises(ValidationError):
            model_rows.validate_json(raw)
        with pytest.raises(RequestValidationError) as ei:
            parse_request(raw)
        assert all(err["loc"][0] == "body" for err in ei.value.errors())
    with _client(StubModel()) as c:
        for raw in bad:
            r = c.post("/predict", content=raw, headers={"content-type": "application/json"})
            assert r.status_code == 422 and "detail" in r.json()
        spec = c.get("/openapi.json").json()
        body = spec["paths"]["/predict"]["post"]["requestBody"]["content"]["application/json"]["schema"]
        assert body["type"] == "array" and list(body["items"]["properties"]) == ALL_FEATURES
        assert body["items"]["properties"]["age"]["default"] == 18000.0


def _frames_identical(a, b):
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES, CATEGORICAL_FEATURES

    assert list(a.columns) == list(b.columns) == ALL_FEATURES and len(a) == len(b)
    for name in ALL_FEATURES:
        if name in CATEGORICAL_FEATURES:
            assert a[name].tolist() == b[name].tolist(), name
        else:  # bit patterns, so that -0.0 / 0.0 and the last ulp count
            assert (a[name].to_numpy(np.float64).view(np.uint64) == b[name].to_numpy(np.float64).view(np.uint64)).all(), name


def test_native_request_parser_equals_the_general_validator():
    """ingest.NativeRequestParser (csrc/json_rows.h): for every body the fast path accepts the columns are identical to
    the pydantic path's; everything else is declined (-> general validator -> same coercions / 422 as before)."""
    from fastapi.exceptions import RequestValidationError

    from databricks_kubernetes_mlops_poc_b200.ingest import NativeRequestParser, parse_rows, rows_to_frame
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES, DEFAULTS, sample_request

    p = NativeRequestParser(min_bytes=0)  # the service only takes this path for large bodies; here every body does
    accepted = [
        b"[]", b" [ ] ", b"[{}]", b"[{},{}]", json.dumps(sample_request()).encode(), json.dumps(sample_request(), indent=2).encode(),
        b'[{"sex": "female", "age": 41}]', b'[{"age":41.5,"sex":"","education":"a b/c:d,e"}]',
        b'[{"bill_amount_1": 1e3, "bill_amount_2": -1.5E-3, "bill_amount_3": 0, "bill_amount_4": -0, "bill_amount_5": -0.0, "bill_amount_6": 0.1}]',
        b'[{"credit_limit": 123456789012345, "age": 1.7976931348623157e308, "payment_amount_1": 5e-324, "payment_amount_2": 2.2250738585072011e-308}]',
        b'[{"credit_limit": 0.30000000000000004, "age": 9007199254740993.0, "payment_amount_3": 1.0000000000000002}]',
        b'\n[\t{"sex"\r:\n"male" ,"age" : 1 }\n, {"age":2}]\n',
    ]
    for raw in accepted:
        got = p.columns(raw)
        assert got is not None, raw
        rows = parse_rows(raw)
        assert got[0] == len(rows)
        if rows:
            _frames_identical(p.frame(raw), rows_to_frame(rows))
    assert p.frame(b"[{}]").iloc[0].to_dict() == DEFAULTS and len(p.frame(b"[]")) == 0
    declined = [
        b"", b"[", b"{", b'{"sex": "male"}', b"[1]", b"null", b'[{"sex": 3}]', b'[{"age": "41"}]', b'[{"age": "old"}]', b'[{"age": null}]',
        b'[{"age": true}]', b'[{"unknown_key": 1}]', b'[{"age": 1, "age": 2}]', b'[{"sex": "a\\"b"}]', b'[{"sex": "caf\xc3\xa9"}]',
        b'[{"sex": "x\\u0041"}]', b'[{"age": 01}]', b'[{"age": 1.}]', b'[{"age": .5}]', b'[{"age": +1}]', b'[{"age": 1e999}]', b'[{"age": NaN}]',
        b'[{"age": Infinity}]', b'[{"age": 1234567890123456}]', b'[{"age": 1},]', b'[{"age": 1,}]', b'[{"age": 1}] x', b'[{"age" 1}]', b"[{]",
        b'[{"sex": "a\tb"}]', b'[{"": 1}]', b"[[]]",
    ]
    for raw in declined:
        assert p.columns(raw) is None, raw
        try:  # ... and frame() then behaves exactly like the general path
            want = parse_rows(raw)
        except RequestValidationError:
            with pytest.raises(RequestValidationError):
                p.frame(raw)
        else:
            _frames_identical(p.frame(raw), rows_to_frame(want))
    assert p.fast > 0 and p.general > 0
    p.close()


def test_native_request_parser_on_generated_bodies():
    """Property test: random bodies built from the schema (random subsets of keys, random spacing, numbers printed in
    several styles) -- whenever the fast path accepts, its columns equal the general validator's bit for bit."""
    from hypothesis import given, settings
    from hypothesis import strategies as st

    from databricks_kubernetes_mlops_poc_b200.ingest import NativeRequestParser, parse_rows, rows_to_frame
    from databricks_kubernetes_mlops_poc_b200.schema import CATEGORICAL_FEATURES, NUMERIC_FEATURES

    p = NativeRequestParser(min_bytes=0)
    ws = st.sampled_from(["", " ", "\n", "\t ", "  "])
    number = st.one_of(
        st.floats(allow_nan=False, allow_infinity=False).map(repr),
        st.integers(-10**14, 10**14).map(str),
        st.floats(-1e6, 1e6, allow_nan=False).map(lambda v: f"{v:.3f}"),
        st.floats(allow_nan=False, allow_infinity=False).map(lambda v: f"{v:e}"),
        st.sampled_from(["0", "-0", "0.0", "-0.0", "1E2", "1e+2", "1e-2", "5e-324", "1.7976931348623157e308"]),
    )
    text = st.text(alphabet=st.characters(min_codepoint=32, max_codepoint=126, exclude_characters='"\\'), max_size=12)

    @st.composite
    def body(draw):
        rows = []
        for _ in range(draw(st.integers(0, 4))):
            keys = draw(st.lists(st.sampled_from(CATEGORICAL_FEATURES + NUMERIC_FEATURES), unique=True, max_size=23))
            pairs = []
            for k in keys:
                v = '"' + draw(text) + '"' if k in CATEGORICAL_FEATURES else draw(number)
                pairs.append(f'{draw(ws)}"{k}"{draw(ws)}:{draw(ws)}{v}{draw(ws)}')
            rows.append("{" + ",".join(pairs) + (draw(ws) if not pairs else "") + "}")
        return (draw(ws) + "[" + draw(ws) + (draw(ws) + "," + draw(ws)).join(rows) + draw(ws) + "]" + draw(ws)).encode()

    accepted = [0]

    @settings(max_examples=300, deadline=None)
    @given(body())
    def check(raw):
        rows = parse_rows(raw)  # generated bodies are valid requests
        got = p.columns(raw)
        if got is not None:
            accepted[0] += 1
            assert got[0] == len(rows)
            if rows:
                _frames_identical(p.frame(raw), rows_to_frame(rows))

    check()
    assert accepted[0] > 100
    p.close()


def test_native_request_frames_encode_like_general_frames(curated, rf100d6):
    """Bytes -> native parser -> DataFrame -> row encoder gives the same encoded rows as the pydantic path (1 000-row
    body: large enough for the service to take the native parser and the native row encoder)."""
    from databricks_kubernetes_mlops_poc_b200 import flatten
    from databricks_kubernetes_mlops_poc_b200.encode import RowEncoder
    from databricks_kubernetes_mlops_poc_b200.ingest import NATIVE_MIN_BYTES, NativeRequestParser, parse_rows, rows_to_frame
    from databricks_kubernetes_mlops_poc_b200.schema import ALL_FEATURES

    raw = json.dumps(curated[ALL_FEATURES].iloc[:1000].to_dict(orient="records")).encode()
    assert len(raw) > NATIVE_MIN_BYTES
    p = NativeRequestParser()
    a = p.frame(raw)
    assert p.fast == 1 and p.general == 0
    b = rows_to_frame(parse_rows(raw))
    _frames_identical(a, b)
    enc = RowEncoder(flatten.flatten_pipeline(rf100d6))
    assert (enc.encode_frame_packed(a) == enc.encode_frame_packed(b)).all()
    assert (enc.encode_frame(a) == enc.encode_frame(curated[ALL_FEATURES].iloc[:1000])).all()
    small = json.dumps(curated[ALL_FEATURES].iloc[:3].to_dict(orient="records")).encode()
    p.frame(small)
    assert p.general == 1  # small bodies stay on the general path
    p.close()

"""Frozen copies of the reference's data fixtures (TEST INFRASTRUCTURE).

``tests/golden/curated.npz`` / ``inference.npz`` are lossless dictionary-encoded
copies of the reference's ``databricks/data/curated.csv`` (30 000 labelled rows)
and ``databricks/data/inference.csv`` (80 rows, different column order), written
by ``tests/golden/make_golden.py``, so that the tests need nothing outside the
repository.  Every numeric value in those files has at most two decimals; it is
stored as int32 hundredths (``nums_cents``), and ``cents / 100.0`` gives back the
float64 the CSV parser produced, bit for bit.
"""

from __future__ import annotations

import os

import numpy as np
import pandas as pd

from .reference_pipeline import CATEGORICAL_FEATURES, NUMERIC_FEATURES, TARGET

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _thaw(z, with_target: bool) -> pd.DataFrame:
    cols = {}
    for j, name in enumerate(CATEGORICAL_FEATURES):
        cols[name] = z[f"vocab_{j}"][z[f"codes_{j}"].astype(np.int64)].astype(object)
    nums = z["nums_cents"] / 100.0
    for j, name in enumerate(NUMERIC_FEATURES):
        cols[name] = nums[:, j]
    df = pd.DataFrame(cols)
    for name in CATEGORICAL_FEATURES:
        df[name] = df[name].astype(str)
    if with_target:
        df[TARGET] = z["target"].astype(np.int64)
    return df


def load_curated() -> pd.DataFrame:
    """30 000 rows, columns = 9 categorical + 14 numeric + target, CSV row order."""
    with np.load(os.path.join(GOLDEN_DIR, "curated.npz")) as z:
        return _thaw(z, True)


def load_inference() -> pd.DataFrame:
    """80 unlabelled rows in the inference.csv column order (credit_limit first)."""
    with np.load(os.path.join(GOLDEN_DIR, "inference.npz")) as z:
        df = _thaw(z, False)
        return df[[str(c) for c in z["column_order"]]]


def load_expected(name: str) -> dict:
    with np.load(os.path.join(GOLDEN_DIR, f"expected_{name}.npz")) as z:
        return {k: z[k] for k in z.files}

"""Model-artefact tooling: builds the sklearn pipelines the engine is fed with, and the synthetic
workloads BASELINE.json's configs name.  Offline / harness code -- nothing here runs per request.

* ``make_pipeline``: the reference's pipeline shape (``databricks/src/01-train-model.ipynb:195-231``:
  constant-impute + one-hot for the 9 categoricals, median-impute for the 14 numerics, then the
  classifier).  ``kind="rf"`` is the reference's RandomForestClassifier; ``kind="gbdt"`` puts sklearn's
  GradientBoostingClassifier behind the same preprocessing for BASELINE configs 2-4 (the reference has
  no GBDT; SURVEY.md section 0 row 2).
* ``synth_frame`` / ``synth_arrays``: seeded synthetic request batches in the credit-default schema
  (SURVEY.md section 8d, cfg 2): category codes uniform over the training vocabularies with 1 % unknown,
  numerics bootstrap-resampled from the training columns with 0.5 % NaN.
"""

from __future__ import annotations

import numpy as np
import pandas as pd

from .schema import CATEGORICAL_FEATURES, NUMERIC_FEATURES


def make_pipeline(kind: str, **params):
    from sklearn.compose import ColumnTransformer
    from sklearn.ensemble import GradientBoostingClassifier, RandomForestClassifier
    from sklearn.impute import SimpleImputer
    from sklearn.pipeline import Pipeline
    from sklearn.preprocessing import OneHotEncoder

    cat = Pipeline([("imputer", SimpleImputer(strategy="constant", fill_value="missing")), ("ohe", OneHotEncoder(handle_unknown="ignore"))])
    num = Pipeline([("imputer", SimpleImputer(strategy="median"))])
    pre = ColumnTransformer([("categorical", cat, CATEGORICAL_FEATURES), ("numeric", num, NUMERIC_FEATURES)])
    if kind == "rf":
        clf = RandomForestClassifier(**params, n_jobs=-1)
    elif kind == "gbdt":
        clf = GradientBoostingClassifier(**params)
    else:
        raise ValueError(kind)
    return Pipeline([("preprocessor", pre), ("classifier", clf)])


def synth_arrays(base: pd.DataFrame, n: int, seed: int, unknown_frac: float = 0.01, nan_frac: float = 0.005):
    """-> (vocab list, codes int32 (n, 9) with -1 = unknown, nums float64 (n, 14) with NaN = missing)."""
    rng = np.random.default_rng(seed)
    vocabs = [np.unique(base[c].astype(str).to_numpy()) for c in CATEGORICAL_FEATURES]
    codes = np.empty((n, len(vocabs)), dtype=np.int32)
    for j, v in enumerate(vocabs):
        codes[:, j] = rng.integers(0, len(v), size=n)
    codes[rng.random(codes.shape) < unknown_frac] = -1
    nums = np.empty((n, len(NUMERIC_FEATURES)), dtype=np.float64)
    for k, c in enumerate(NUMERIC_FEATURES):
        col = base[c].to_numpy(dtype=np.float64)
        nums[:, k] = col[rng.integers(0, len(col), size=n)]
    nums[rng.random(nums.shape) < nan_frac] = np.nan
    return vocabs, codes, nums


def arrays_to_frame(vocabs, codes: np.ndarray, nums: np.ndarray) -> pd.DataFrame:
    """Decode (codes, nums) into the string/float DataFrame a request would carry
    (unknown code -> the out-of-vocabulary string "__unseen__")."""
    cols = {}
    for j, name in enumerate(CATEGORICAL_FEATURES):
        ext = np.concatenate([np.asarray(vocabs[j], dtype=object), np.array(["__unseen__"], dtype=object)])
        cols[name] = ext[np.where(codes[:, j] < 0, len(vocabs[j]), codes[:, j])]
    for k, name in enumerate(NUMERIC_FEATURES):
        cols[name] = nums[:, k]
    return pd.DataFrame(cols)


def synth_frame(base: pd.DataFrame, n: int, seed: int, **kw) -> pd.DataFrame:
    v, c, x = synth_arrays(base, n, seed, **kw)
    return arrays_to_frame(v, c, x)


def synth_labels(codes: np.ndarray, nums: np.ndarray, seed: int) -> np.ndarray:
    """A fixed, mildly non-linear rule + noise so synthetic GBDT / RF fits grow real trees."""
    rng = np.random.default_rng(seed)
    x = np.nan_to_num(nums, nan=0.0)
    z = (
        0.35 * (codes[:, 3] % 4)
        + 0.25 * (codes[:, 4] % 3)
        - 0.00004 * x[:, 0]
        + 0.00003 * (x[:, 2] - x[:, 8])
        + 0.4 * ((codes[:, 1] == 2) & (x[:, 1] > 40))
        - 0.8
    )
    p = 1.0 / (1.0 + np.exp(-z))
    return (rng.random(len(p)) < p).astype(np.int64)


def fit_synthetic(kind: str, base: pd.DataFrame, n_train: int, seed: int, **params):
    """Fit ``kind`` on n_train seeded synthetic rows; returns the fitted pipeline."""
    vocabs, codes, nums = synth_arrays(base, n_train, seed)
    # training rows carry no unknowns for the categorical vocabulary to be complete
    codes = np.where(codes < 0, 0, codes)
    df = arrays_to_frame(vocabs, codes, nums)
    y = synth_labels(codes, nums, seed + 1)
    pipe = make_pipeline(kind, **params)
    pipe.fit(df[CATEGORICAL_FEATURES + NUMERIC_FEATURES], y)
    return pipe


def load_base_frame(path: str | None = None) -> pd.DataFrame:
    """The 30 000-row credit-default table (frozen copy of the reference's
    ``databricks/data/curated.csv`` under ``tests/golden/curated.npz``) that synthetic workloads are
    bootstrap-resampled from.  Data fixture only -- no oracle code involved."""
    import os

    if path is None:
        path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden", "curated.npz")
    with np.load(path) as z:
        cols = {}
        for j, name in enumerate(CATEGORICAL_FEATURES):
            cols[name] = z[f"vocab_{j}"][z[f"codes_{j}"].astype(np.int64)].astype(object)
        nums = z["nums_cents"] / 100.0  # stored as int32 hundredths; exact for the table's two-decimal values
        for k, name in enumerate(NUMERIC_FEATURES):
            cols[name] = nums[:, k]
        df = pd.DataFrame(cols)
        for name in CATEGORICAL_FEATURES:
            df[name] = df[name].astype(str)
        df["default_payment_next_month"] = z["target"].astype(np.int64)
    return df

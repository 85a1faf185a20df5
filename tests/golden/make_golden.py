#!/usr/bin/env python
"""Generate the golden fixtures under tests/golden/ (run in the authoring container only).

The reference (``/root/reference``) does not exist on the GPU box, and it ships no
golden vectors of its own (SURVEY.md section 4).  This script

1. reads the reference's own data fixtures
   (``databricks/data/curated.csv`` -- 30 000 labelled rows, ``databricks/data/inference.csv``
   -- 80 unlabelled rows in a different column order) and freezes them, losslessly
   dictionary-encoded, into ``curated.npz`` / ``inference.npz``;
2. re-fits the reference pipeline definition (``oracle.reference_pipeline``; reference
   ``databricks/src/01-train-model.ipynb:195-231`` + split ``:260-264``) for the two pinned
   models and freezes the REAL library outputs (``predict_proba[:, 1]`` and ``predict``) on
   all 30 000 + 80 rows into ``expected_<model>.npz`` together with the sklearn version;
3. checks the numpy and C restatements against the library before writing anything.

Usage:  python tests/golden/make_golden.py [--reference /root/reference]
"""

from __future__ import annotations

import argparse
import os
import sys

import numpy as np
import pandas as pd
import sklearn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import datasets, reference_pipeline as rp, treewalk as tw  # noqa: E402


def freeze_frame(df: pd.DataFrame, with_target: bool) -> dict:
    out = {}
    for j, name in enumerate(rp.CATEGORICAL_FEATURES):
        vocab, codes = np.unique(df[name].astype(str).to_numpy(), return_inverse=True)
        out[f"vocab_{j}"] = vocab.astype("U")
        out[f"codes_{j}"] = codes.astype(np.int8)
    # the CSV's numerics carry at most two decimals: int32 hundredths store them exactly in half the bytes of float64
    nums = df[rp.NUMERIC_FEATURES].to_numpy(dtype=np.float64)
    out["nums_cents"] = np.round(nums * 100.0).astype(np.int32)
    assert (out["nums_cents"] / 100.0 == nums).all() and not (np.signbit(nums) & (nums == 0)).any()
    if with_target:
        out["target"] = df[rp.TARGET].to_numpy(dtype=np.int8)
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reference", default="/root/reference")
    args = ap.parse_args()

    cur_csv = pd.read_csv(os.path.join(args.reference, "databricks/data/curated.csv"))
    inf_csv = pd.read_csv(os.path.join(args.reference, "databricks/data/inference.csv"))
    assert not cur_csv[rp.FEATURES].isna().any().any()

    np.savez_compressed(os.path.join(HERE, "curated.npz"), **freeze_frame(cur_csv, True))
    inf_frozen = freeze_frame(inf_csv, False)
    inf_frozen["column_order"] = np.array(list(inf_csv.columns), dtype="U")
    np.savez_compressed(os.path.join(HERE, "inference.npz"), **inf_frozen)

    # round trip: the frozen frames must reproduce the CSV frames exactly
    cur = datasets.load_curated()
    inf = datasets.load_inference()
    for name in rp.CATEGORICAL_FEATURES:
        assert (cur[name].to_numpy() == cur_csv[name].astype(str).to_numpy()).all()
        assert (inf[name].to_numpy() == inf_csv[name].astype(str).to_numpy()).all()
    for name in rp.NUMERIC_FEATURES:
        assert (cur[name].to_numpy() == cur_csv[name].to_numpy(dtype=np.float64)).all()
        assert (inf[name].to_numpy() == inf_csv[name].to_numpy(dtype=np.float64)).all()
    assert list(inf.columns) == list(inf_csv.columns)

    for name, params in rp.PINNED_RF.items():
        pipe_csv = rp.fit_reference_pipeline(cur_csv, params)  # straight from the reference CSV
        pipe = rp.fit_reference_pipeline(cur, params)  # from the frozen copy
        p_csv, l_csv = rp.oracle_predict(pipe_csv, cur_csv)
        p, l = rp.oracle_predict(pipe, cur)
        # RF summation order is thread-dependent at the 1e-16 level; labels must agree exactly
        assert np.abs(p - p_csv).max() < 1e-14 and (l == l_csv).all(), name
        pi, li = rp.oracle_predict(pipe, inf)
        # restatements vs the library
        dump = tw.dump_pipeline(pipe)
        pn, ln = tw.predict_numpy(dump, cur)
        codes, nums = tw.encode_frame(dump, cur)
        pc, lc = tw.predict_c(dump, codes, nums)
        assert np.abs(pn - p).max() < 1e-14 and (ln == l).all()
        assert np.abs(pc - p).max() < 1e-14 and (lc == l).all()
        margin = float(np.abs(p - 0.5).min())
        assert margin > 1e-9, "a pinned-model row sits on the label knife edge"
        clf = pipe.named_steps["classifier"]
        np.savez_compressed(
            os.path.join(HERE, f"expected_{name}.npz"),
            sklearn_version=np.array(sklearn.__version__),
            params=np.array(repr(params)),
            proba1=p,
            label=l.astype(np.int8),
            inf_proba1=pi,
            inf_label=li.astype(np.int8),
            total_nodes=np.array(sum(e.tree_.node_count for e in clf.estimators_)),
            min_margin=np.array(margin),
        )
        print(f"{name}: nodes={sum(e.tree_.node_count for e in clf.estimators_)} "
              f"min|p-0.5|={margin:.3e} restatement max err numpy={np.abs(pn - p).max():.2e} C={np.abs(pc - p).max():.2e}")
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == "__main__":
    main()

"""Back-to-back rank launches with programmatic dependent launch: the kernel reads its rows before it waits for the previous
launch, so a launch whose rows are what the previous rank launch on the stream writes must still see the finished values."""

import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _engine(pipe):
    from databricks_kubernetes_mlops_poc_b200 import flatten
    from databricks_kubernetes_mlops_poc_b200.encode import RowEncoder
    from databricks_kubernetes_mlops_poc_b200.engine import ForestEngine

    flat = flatten.flatten_pipeline(pipe)
    return ForestEngine(flat, 0), RowEncoder(flat)


def test_rows_written_by_the_previous_launch(curated, rf100d6):
    from databricks_kubernetes_mlops_poc_b200._cabi import ROWS_RANKED

    eng, enc = _engine(rf100d6)
    try:
        rk = enc.rank_rows(enc.encode_frame(curated))
        n1 = rk.shape[0]
        n2 = n1 * 8 // (rk.shape[1] * 4)  # the first launch's float64 probabilities, read as ranked rows
        d_rows = eng.device_alloc(rk.nbytes)
        d_p1 = eng.device_alloc(n1 * 8)
        d_l1 = eng.device_alloc(n1 * 4)
        d_p2 = eng.device_alloc(n2 * 8)
        d_l2 = eng.device_alloc(n2 * 4)
        eng.h2d(d_rows, rk)
        stale = np.full(n1, 0.75, dtype=np.float64)  # what the second launch would see if it read its rows too early

        def pair(sync_between: bool):
            eng.h2d(d_p1, stale)
            eng.sync()
            eng.predict_device(d_rows, n1, d_p1, True, d_l1, fmt=ROWS_RANKED)
            if sync_between:
                eng.sync()
            eng.predict_device(d_p1, n2, d_p2, True, d_l2, fmt=ROWS_RANKED)
            pdl = eng.info()["rank_last_pdl"]
            eng.sync()
            p1, p2 = np.empty(n1), np.empty(n2)
            l2 = np.empty(n2, dtype=np.int32)
            eng.d2h(p1, d_p1)
            eng.d2h(p2, d_p2)
            eng.d2h(l2, d_l2)
            return p1, p2, l2, pdl

        q1, q2, m2, pdl_q = pair(False)
        s1, s2, k2, _ = pair(True)
        assert pdl_q == 0, "rows that overlap the previous rank launch's outputs must not go out with programmatic serialization"
        assert np.array_equal(q1, s1)
        assert np.array_equal(q2, s2) and np.array_equal(m2, k2)
        # and the second launch did read the first one's results, not the stale fill
        eng.h2d(d_p1, stale)
        eng.predict_device(d_p1, n2, d_p2, True, d_l2, fmt=ROWS_RANKED)
        eng.sync()
        from_stale = np.empty(n2)
        eng.d2h(from_stale, d_p2)
        assert not np.array_equal(from_stale, s2)
        for p in (d_rows, d_p1, d_l1, d_p2, d_l2):
            eng.device_free(p)
    finally:
        eng.close()


@pytest.mark.skipif(os.environ.get("B2F_NO_PDL") is not None, reason="B2F_NO_PDL turns programmatic dependent launch off")
def test_separate_buffers_keep_programmatic_launch(curated, rf100d6):
    from databricks_kubernetes_mlops_poc_b200._cabi import ROWS_RANKED

    eng, enc = _engine(rf100d6)
    try:
        rk = enc.rank_rows(enc.encode_frame(curated))
        n = rk.shape[0]
        d_rows = eng.device_alloc(2 * rk.nbytes)
        d_p = eng.device_alloc(2 * n * 4)
        d_l = eng.device_alloc(2 * n * 4)
        eng.h2d(d_rows, np.concatenate([rk, rk]))
        eng.predict_device(d_rows, n, d_p, False, d_l, fmt=ROWS_RANKED)
        eng.predict_device(d_rows + rk.nbytes, n, d_p + n * 4, False, d_l + n * 4, fmt=ROWS_RANKED)
        assert eng.info()["rank_last_pdl"] == 1
        # the same rows again, into the same outputs: rows never overlap outputs, so programmatic launch stays on
        eng.predict_device(d_rows, n, d_p, False, d_l, fmt=ROWS_RANKED)
        assert eng.info()["rank_last_pdl"] == 1
        # rows inside the previous launch's label buffer: serialised
        eng.predict_device(d_l, n // rk.shape[1], d_p + n * 4, False, d_l + n * 4, fmt=ROWS_RANKED)
        assert eng.info()["rank_last_pdl"] == 0
        eng.sync()
        p = np.empty(2 * n, dtype=np.float32)
        eng.d2h(p, d_p)
        assert np.isfinite(p[:n]).all()
        for q in (d_rows, d_p, d_l):
            eng.device_free(q)
    finally:
        eng.close()


@pytest.mark.skipif(os.environ.get("B2F_NO_PDL") is not None, reason="B2F_NO_PDL turns programmatic dependent launch off")
def test_rows_written_two_launches_back(curated, rf100d6):
    """Launches with the attribute chain (each triggers its dependents at entry), so with small grids launch C can run while
    A has not stored yet: C reading A's probabilities must go out without the attribute even though B between them is unrelated."""
    from databricks_kubernetes_mlops_poc_b200._cabi import ROWS_RANKED

    eng, enc = _engine(rf100d6)
    try:
        rk = enc.rank_rows(enc.encode_frame(curated))[:1024]  # 32 tiles: a third of the SMs per launch
        n = rk.shape[0]
        n3 = n * 8 // (rk.shape[1] * 4)
        d_rows = eng.device_alloc(2 * rk.nbytes)
        d_pa, d_la = eng.device_alloc(n * 8), eng.device_alloc(n * 4)
        d_pb, d_lb = eng.device_alloc(n * 8), eng.device_alloc(n * 4)
        d_pc, d_lc = eng.device_alloc(n3 * 8), eng.device_alloc(n3 * 4)
        eng.h2d(d_rows, np.concatenate([rk, rk]))

        def chain(sync_between: bool):
            eng.h2d(d_pa, np.full(n, 0.75))
            eng.sync()
            eng.predict_device(d_rows, n, d_pa, True, d_la, fmt=ROWS_RANKED)
            eng.predict_device(d_rows + rk.nbytes, n, d_pb, True, d_lb, fmt=ROWS_RANKED)
            pdl_b = eng.info()["rank_last_pdl"]
            if sync_between:
                eng.sync()
            eng.predict_device(d_pa, n3, d_pc, True, d_lc, fmt=ROWS_RANKED)
            pdl_c = eng.info()["rank_last_pdl"]
            eng.sync()
            pc, lc = np.empty(n3), np.empty(n3, dtype=np.int32)
            eng.d2h(pc, d_pc)
            eng.d2h(lc, d_lc)
            return pc, lc, pdl_b, pdl_c

        pc, lc, pdl_b, pdl_c = chain(False)
        assert pdl_b == 1, "B's rows are not written by A: B keeps programmatic launch"
        assert pdl_c == 0, "C reads what A (two launches back, same chain) writes"
        sc, sl, _, _ = chain(True)
        assert np.array_equal(pc, sc) and np.array_equal(lc, sl)
        for p in (d_rows, d_pa, d_la, d_pb, d_lb, d_pc, d_lc):
            eng.device_free(p)
    finally:
        eng.close()


@pytest.mark.skipif(os.environ.get("B2F_NO_PDL") is not None, reason="B2F_NO_PDL turns programmatic dependent launch off")
def test_long_chain_remembers_every_launch(curated, rf100d6):
    """Separate buffers keep programmatic launch however long the chain; rows written ten launches back still serialise."""
    from databricks_kubernetes_mlops_poc_b200._cabi import ROWS_RANKED

    eng, enc = _engine(rf100d6)
    try:
        rk = enc.rank_rows(enc.encode_frame(curated))[:256]
        n, k = rk.shape[0], 12
        d_rows = eng.device_alloc(rk.nbytes)
        d_p, d_l = eng.device_alloc(k * n * 4), eng.device_alloc(k * n * 4)
        eng.h2d(d_rows, rk)
        seen = []
        for i in range(k - 1):
            eng.predict_device(d_rows, n, d_p + i * n * 4, False, d_l + i * n * 4, fmt=ROWS_RANKED)
            seen.append(eng.info()["rank_last_pdl"])
        assert seen[1:] == [1] * (k - 2)
        eng.predict_device(d_l, n // rk.shape[1], d_p + (k - 1) * n * 4, False, d_l + (k - 1) * n * 4, fmt=ROWS_RANKED)
        assert eng.info()["rank_last_pdl"] == 0  # rows = the labels of the first launch of the chain
        eng.sync()
        for p in (d_rows, d_p, d_l):
            eng.device_free(p)
    finally:
        eng.close()

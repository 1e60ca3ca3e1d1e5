"""slm_cv_score_stats against numpy: max, percentage sum and median of |r| over row ranges and row lists, with and
without intercepts and sample-weight scaling, on integer-valued data whose residuals tie exactly."""

import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from sparselm_b200 import _lib  # noqa: E402

EPS = np.finfo(np.float64).eps
ALL = _lib.SLM_STAT_MAX | _lib.SLM_STAT_MAPE | _lib.SLM_STAT_MEDIAN
SIZES = [1, 2, 3, 255, 256, 257, 4096, 80001]
KS = [1, 7, 8, 9, 104]
N, P = 80001, 13


@pytest.fixture(scope="module")
def eng():
    from sparselm_b200.engine import get_engine

    return get_engine()


@pytest.fixture(scope="module")
def data(eng):
    rng = np.random.default_rng(0)
    X = rng.integers(-3, 4, (N, P)).astype(np.float64)
    B = rng.integers(-2, 3, (P, 104)).astype(np.float64)
    # column 0 leaves the residual 3 on every row (an all-equal column); the others tie on small integers
    y = X @ B[:, 0] + 3.0  # zero on some rows: percentage terms of |r| / eps
    icpt = rng.integers(-2, 3, 104).astype(np.float64)
    icpt[0] = 0.0
    # powers of two as weights: the sqrt(sw) scaling and its division are exact, so the ties survive
    sw = rng.choice([0.25, 1.0, 4.0], N)
    return dict(X=X, y=y, B=B, icpt=icpt, sw=sw, Bd=eng.to_device(B), icd=eng.to_device(icpt),
                Xa={False: eng.pack(X, y), True: eng.pack(X, y, sw)})


def _problems():
    """(m, K, intercept?) for every size and column count: 40 problems, more than one 32-problem batch."""
    return [(m, K, (i + j) % 2 == 0) for i, m in enumerate(SIZES) for j, K in enumerate(KS)]


@pytest.mark.parametrize("rows_scaled", [False, True], ids=["plain", "weighted"])
@pytest.mark.parametrize("feed", ["ranges", "lists"])
def test_score_stats_matches_numpy(eng, data, feed, rows_scaled):
    rng = np.random.default_rng(1 + rows_scaled)
    Xa = data["Xa"][rows_scaled]
    items, idx = [], []
    for m, K, with_icpt in _problems():
        ic = data["icd"] if with_icpt else None
        if feed == "ranges":
            r0 = int(rng.integers(0, N - m + 1))
            items.append((r0, r0 + m, data["Bd"], K, ic))
            idx.append(np.arange(r0, r0 + m))
        else:
            rows = np.sort(rng.choice(N, m, replace=False))
            items.append((eng.to_device(rows.astype(np.int32)), data["Bd"], K, ic))
            idx.append(rows)
    out, res = eng.cv_score_stats(Xa, P, items, rows_scaled=rows_scaled, stats=ALL, return_residuals=True)
    out = out.cpu().numpy()
    res = [r.cpu().numpy() for r in res]
    sums = (eng.cv_score_many if feed == "ranges" else eng.cv_score_rows)(Xa, P, items, rows_scaled=rows_scaled)
    sums = sums.cpu().numpy()
    again = eng.cv_score_stats(Xa, P, items, rows_scaled=rows_scaled, stats=ALL).cpu().numpy()
    assert np.array_equal(out, again)  # bitwise repeatable
    X, y, B, icpt = data["X"], data["y"], data["B"], data["icpt"]
    for i, (it, rows) in enumerate(zip(items, idx)):
        K, with_icpt = it[-2], it[-1] is not None
        m = len(rows)
        # rows 0 and 1: bitwise the residual sums of slm_cv_score_many / slm_cv_score_rows
        assert np.array_equal(out[i, :2, :K], sums[i, :, :K]), (i, m, K)
        want_r = y[rows, None] - X[rows] @ B[:, :K] - (icpt[:K] if with_icpt else 0.0)
        r = res[i][:m, :K]
        np.testing.assert_allclose(r, want_r, rtol=1e-13, atol=1e-13 * np.abs(want_r).max(), err_msg=f"{i} {m} {K}")
        a = np.abs(r)
        assert np.array_equal(out[i, 2, :K], a.max(0)), (i, m, K)
        assert np.array_equal(out[i, 4, :K], np.median(a, axis=0)), (i, m, K)
        den = np.maximum(np.abs(y[rows]), EPS)
        want_pct = np.array([math.fsum(a[:, k] / den) for k in range(K)])
        np.testing.assert_allclose(out[i, 3, :K], want_pct, rtol=1e-13, err_msg=f"{i} {m} {K}")
        assert out[i, 4, 0] == 3.0 and out[i, 2, 0] == 3.0  # the all-equal column


def test_only_the_requested_statistics_are_written(eng, data):
    Xa = data["Xa"][False]
    items = [(10, 310, data["Bd"], 9, data["icd"]), (0, 1, data["Bd"], 9, None)]
    med = eng.cv_score_stats(Xa, P, items, stats=_lib.SLM_STAT_MEDIAN).cpu().numpy()
    full = eng.cv_score_stats(Xa, P, items, stats=ALL).cpu().numpy()
    assert not med[:, 2:4].any()
    assert np.array_equal(med[:, 4], full[:, 4]) and np.array_equal(med[:, :2], full[:, :2])
    mx = eng.cv_score_stats(Xa, P, items, stats=_lib.SLM_STAT_MAX).cpu().numpy()
    assert np.array_equal(mx[:, 2], full[:, 2]) and not mx[:, 3:].any()
    from sparselm_b200.engine import EngineError

    with pytest.raises(EngineError, match="unknown statistic"):
        eng.cv_score_stats(Xa, P, items, stats=1 << 5)

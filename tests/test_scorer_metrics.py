"""The residual-statistics scorers of the batched search (neg_median_absolute_error, neg_max_error,
neg_mean_absolute_percentage_error, d2_absolute_error_score): accepted forms, formulas against sklearn's functions,
and routing (no GPU needed)."""

import warnings
from types import SimpleNamespace

import numpy as np
import pytest
from sklearn.exceptions import UndefinedMetricWarning
from sklearn.metrics import (d2_absolute_error_score, max_error, mean_absolute_percentage_error,
                             median_absolute_error)

from sparselm_b200.model import Lasso
from sparselm_b200.model_selection import (GridSearchCV, _abs_dev_median, _device_metrics, _metric, _split_metric,
                                           _stat_mask)

NEW = ["neg_median_absolute_error", "neg_max_error", "neg_mean_absolute_percentage_error", "d2_absolute_error_score"]


def test_device_metrics_accepts_the_statistics_scorers():
    for name in NEW:
        assert _device_metrics(name) == name
    assert _device_metrics(NEW + ["r2"]) == {nm: nm for nm in NEW + ["r2"]}
    assert _device_metrics(tuple(NEW)) == {nm: nm for nm in NEW}
    assert _device_metrics({"med": NEW[0], "d2": NEW[3]}) == {"med": NEW[0], "d2": NEW[3]}
    assert _device_metrics("explained_variance") is None
    assert _device_metrics("max_error") is None
    assert _device_metrics({"a": NEW[1], "b": "max_error"}) is None
    assert _device_metrics([NEW[0], "explained_variance"]) is None
    assert _device_metrics(lambda est, X, y: 0.0) is None


def test_stat_mask():
    assert _stat_mask({"a": "r2", "b": "neg_mean_absolute_error"}) == 0
    assert _stat_mask({"a": "d2_absolute_error_score"}) == 0  # the sums and y suffice
    assert _stat_mask({"a": "neg_max_error"}) == 1 << 2
    assert _stat_mask({"a": "neg_mean_absolute_percentage_error"}) == 1 << 3
    assert _stat_mask({nm: nm for nm in NEW}) == (1 << 2) | (1 << 3) | (1 << 4)


def _inputs(y, yp):
    """What the device hands _metric: per-column sums and statistics of r = y - yp, one column per prediction."""
    r = y[:, None] - yp
    a = np.abs(r)
    stats = dict(max=a.max(0), median=np.median(a, axis=0),
                 mape=(a / np.maximum(np.abs(y), np.finfo(np.float64).eps)[:, None]).sum(0), sad=_abs_dev_median(y))
    return (r * r).sum(0), a.sum(0), stats


SK = {"neg_median_absolute_error": lambda y, p: -median_absolute_error(y, p),
      "neg_max_error": lambda y, p: -max_error(y, p),
      "neg_mean_absolute_percentage_error": lambda y, p: -mean_absolute_percentage_error(y, p),
      "d2_absolute_error_score": d2_absolute_error_score}


def _cases():
    rng = np.random.default_rng(0)
    y = rng.standard_normal(41)
    yield "random_odd", y, y[:, None] + rng.standard_normal((41, 3))
    y = rng.standard_normal(40)
    yield "random_even", y, y[:, None] + rng.standard_normal((40, 3))
    y = np.round(3 * rng.standard_normal(30))
    y[::4] = 0.0  # zeros in y: MAPE terms of |r| / eps
    yield "zeros_in_y", y, y[:, None] + np.round(rng.standard_normal((30, 3)))
    y = np.full(12, 2.5)
    yield "constant_y", y, np.stack([y, y + 0.5, y - rng.random(12)], axis=1)  # perfect / imperfect, zero denominator
    y = rng.standard_normal(9)
    yield "perfect", y, np.stack([y, y + 1.0], axis=1)
    y = np.array([1.0, 2.0, 2.0, 3.0, 3.0, 3.0])
    yield "ties", y, np.stack([y - 1.0, np.full(6, 2.0)], axis=1)


@pytest.mark.parametrize("case", [c[0] for c in _cases()])
@pytest.mark.parametrize("scoring", NEW)
def test_metric_matches_sklearn(case, scoring):
    _, y, yp = next(c for c in _cases() if c[0] == case)
    sse, sae, stats = _inputs(y, yp)
    want = np.array([SK[scoring](y, yp[:, k]) for k in range(yp.shape[1])])
    for fn in (_metric, _split_metric):
        got = fn(scoring, sse, sae, len(y), 0.0, stats)
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=0)
    if case == "zeros_in_y" and scoring == "neg_mean_absolute_percentage_error":
        assert np.all(np.abs(want) > 1e13)  # MAPE near 1e14 where y is zero


def test_d2_force_finite_rules():
    y = np.full(5, 1.0)
    sse, sae, stats = _inputs(y, np.stack([y, y + 1.0], axis=1))
    assert stats["sad"] == 0.0
    assert _metric("d2_absolute_error_score", sse, sae, 5, 0.0, stats).tolist() == [1.0, 0.0]


@pytest.mark.parametrize("fn", [_metric, _split_metric])
def test_d2_on_one_row_is_nan_with_a_warning(fn):
    y, yp = np.array([1.5]), np.array([[1.0, 1.5]])
    sse, sae, stats = _inputs(y, yp)
    with pytest.warns(UndefinedMetricWarning):
        want = d2_absolute_error_score(y, yp[:, 0])
    assert np.isnan(want)
    with pytest.warns(UndefinedMetricWarning):
        got = fn("d2_absolute_error_score", sse, sae, 1, 0.0, stats)
    assert np.isnan(got).all() and got.shape == (2,)
    # the median and max of one row are |r| itself
    assert fn("neg_median_absolute_error", sse, sae, 1, 0.0, stats).tolist() == [-0.5, -0.0]


def test_abs_dev_median_matches_sklearn_quantile():
    from sklearn.utils.stats import _weighted_percentile

    rng = np.random.default_rng(3)
    for y in (rng.standard_normal(11), rng.standard_normal(12), np.round(rng.standard_normal(20))):
        q = _weighted_percentile(y, np.ones_like(y), 50, average=True)
        assert q == np.median(y)
        assert _abs_dev_median(y) == pytest.approx(np.abs(y - q).sum(), rel=1e-15)


@pytest.mark.parametrize("scoring", NEW + [{"r2": "r2", "med": "neg_median_absolute_error"}])
def test_sharded_search_with_a_statistics_scorer_keeps_the_per_fit_loop(scoring):
    rng = np.random.default_rng(0)
    X, y = rng.standard_normal((40, 6)), rng.standard_normal(40)
    refit = "med" if isinstance(scoring, dict) else True
    gs = GridSearchCV(Lasso(), {"alpha": [0.1, 0.2]}, cv=4, scoring=scoring, refit=refit)
    gs._shard = SimpleNamespace(world=2, rank=0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        assert gs._batch_plan(X, y, {}) is None

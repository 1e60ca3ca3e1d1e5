"""Batched CV searches with the residual-statistics scorers (neg_median_absolute_error, neg_max_error,
neg_mean_absolute_percentage_error, d2_absolute_error_score): cv_results_, ranks and best_params_ equal sklearn's
per-fit loop over the same engine-backed estimator, on fold partitions, direct and downdated split builds,
leave-one-out and weighted searches."""

import warnings

import numpy as np
import numpy.testing as npt
import pytest
import sklearn
from sklearn.base import clone
from sklearn.exceptions import UndefinedMetricWarning
from sklearn.metrics import get_scorer
from sklearn.model_selection import GridSearchCV as SkGS
from sklearn.model_selection import KFold, LeaveOneOut, RepeatedKFold, ShuffleSplit

pytestmark = pytest.mark.gpu

from sparselm_b200.model import Lasso, SparseGroupLasso  # noqa: E402
from sparselm_b200.model_selection import GridSearchCV, LineSearchCV, _select_best_index_onestd  # noqa: E402

# both sides stop at this relative duality gap, as in test_gpu_split_search.py
OPTS = {"tol": 1e-14}
NEW = ["neg_median_absolute_error", "neg_max_error", "neg_mean_absolute_percentage_error", "d2_absolute_error_score"]
ALL = {nm: nm for nm in NEW + ["r2"]}


def _data(n, p, seed, intercept=0.0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    y = X[:, :4] @ [2.0, -1.0, 1.0, 0.5] + 0.4 * rng.standard_normal(n) + intercept
    return X, y, rng


def _sk_search(est, grid, cv, scoring, X, y, fit_params, **kw):
    """sklearn's per-fit loop; with sample_weight, metadata routing sends the weights to fit only (the project's
    batched searches score unweighted residuals)."""
    if fit_params.get("sample_weight") is None:
        return SkGS(est, grid, cv=cv, scoring=scoring, **kw).fit(X, y, **fit_params)
    with sklearn.config_context(enable_metadata_routing=True):
        if isinstance(scoring, dict):
            scorer = {k: get_scorer(v).set_score_request(sample_weight=False) for k, v in scoring.items()}
        else:
            scorer = get_scorer(scoring).set_score_request(sample_weight=False)
        return SkGS(clone(est).set_fit_request(sample_weight=True), grid, cv=cv, scoring=scorer, **kw).fit(
            X, y, **fit_params)


def _compare(gs, sk, n_splits, metrics, train):
    assert gs.batched_ and gs.n_splits_ == n_splits
    for m in metrics:
        for kind in ("test", "train") if train else ("test",):
            for key in [f"split{i}_{kind}_{m}" for i in range(n_splits)] + [f"mean_{kind}_{m}", f"std_{kind}_{m}"]:
                npt.assert_allclose(gs.cv_results_[key], sk.cv_results_[key], rtol=1e-7, atol=1e-10, equal_nan=True,
                                    err_msg=key)
        npt.assert_array_equal(gs.cv_results_[f"rank_test_{m}"], sk.cv_results_[f"rank_test_{m}"])
    assert gs.best_index_ == sk.best_index_
    assert gs.best_params_ == sk.best_params_


def _case(name):
    """(estimator, grid, cv, X, y, fit params)"""
    grid = {"alpha": [0.004, 0.03, 0.15]}
    if name == "kfold":
        X, y, _ = _data(120, 20, 1)
        return Lasso(solver_options=OPTS), grid, KFold(4), X, y, {}
    if name == "kfold_intercept":
        X, y, _ = _data(120, 20, 2, intercept=1.5)
        return Lasso(fit_intercept=True, solver_options=OPTS), grid, KFold(4), X, y, {}
    if name == "kfold_weighted":
        X, y, rng = _data(120, 24, 3, intercept=0.8)
        groups = np.repeat(np.arange(6), 4)
        return (SparseGroupLasso(groups=groups, l1_ratio=0.4, fit_intercept=True, solver_options=OPTS), grid,
                KFold(4), X, y, {"sample_weight": 0.2 + 2.0 * rng.random(120)})
    if name == "shuffle_split_direct":  # rows in neither set, training rows built directly
        X, y, _ = _data(130, 16, 4, intercept=-0.5)
        return (Lasso(fit_intercept=True, solver_options=OPTS), grid,
                ShuffleSplit(5, test_size=0.2, train_size=0.3, random_state=1), X, y, {})
    if name == "repeated_kfold_downdate":
        X, y, _ = _data(120, 16, 5)
        return Lasso(solver_options=OPTS), grid, RepeatedKFold(n_splits=4, n_repeats=2, random_state=0), X, y, {}
    raise KeyError(name)


CASES = ["kfold", "kfold_intercept", "kfold_weighted", "shuffle_split_direct", "repeated_kfold_downdate"]


@pytest.mark.parametrize("scoring", NEW + ["all"])
@pytest.mark.parametrize("name", CASES)
def test_statistics_scorers_match_sklearn_loop(name, scoring):
    est, grid, cv, X, y, fit_params = _case(name)
    n_splits = cv.get_n_splits(X, y)
    if scoring == "all":
        kw = dict(refit="neg_median_absolute_error", return_train_score=True)
        gs = GridSearchCV(est, grid, cv=cv, scoring=ALL, **kw).fit(X, y, **fit_params)
        sk = _sk_search(est, grid, cv, ALL, X, y, fit_params, **kw)
        assert gs.multimetric_
        _compare(gs, sk, n_splits, tuple(ALL), train=True)
    else:
        gs = GridSearchCV(est, grid, cv=cv, scoring=scoring).fit(X, y, **fit_params)
        sk = _sk_search(est, grid, cv, scoring, X, y, fit_params)
        _compare(gs, sk, n_splits, ("score",), train=False)
    assert (gs.solver_info_["status"] == 0).all()


def test_leave_one_out_d2_is_nan_and_the_median_is_the_residual():
    X, y, _ = _data(30, 10, 6)
    est = Lasso(solver_options=OPTS)
    grid = {"alpha": [0.01, 0.1]}
    kw = dict(refit="neg_median_absolute_error", return_train_score=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        gs = GridSearchCV(est, grid, cv=LeaveOneOut(), scoring=ALL, **kw).fit(X, y)
        sk = SkGS(est, grid, cv=LeaveOneOut(), scoring=ALL, **kw).fit(X, y)
    _compare(gs, sk, 30, tuple(ALL), train=True)
    for s in range(30):
        assert np.isnan(gs.cv_results_[f"split{s}_test_d2_absolute_error_score"]).all()
        # one test row: median |r| = max |r| = |r|
        npt.assert_array_equal(gs.cv_results_[f"split{s}_test_neg_median_absolute_error"],
                               gs.cv_results_[f"split{s}_test_neg_max_error"])
    b = gs.best_estimator_
    assert b.coef_.shape == (10,)
    with pytest.warns(UndefinedMetricWarning):
        GridSearchCV(est, grid, cv=LeaveOneOut(), scoring="d2_absolute_error_score").fit(X, y)
    for scoring in NEW[:3]:
        g = GridSearchCV(est, grid, cv=LeaveOneOut(), scoring=scoring).fit(X, y)
        k = SkGS(est, grid, cv=LeaveOneOut(), scoring=scoring).fit(X, y)
        _compare(g, k, 30, ("score",), train=False)


def test_one_std_rule_with_the_median_scorer():
    X, y, _ = _data(120, 20, 7)
    est = Lasso(solver_options=OPTS)
    grid = {"alpha": list(np.logspace(-3, -0.5, 8))}
    gs = GridSearchCV(est, grid, cv=KFold(4), scoring="neg_median_absolute_error",
                      opt_selection_method="one_std_score").fit(X, y)
    sk = SkGS(est, grid, cv=KFold(4), scoring="neg_median_absolute_error").fit(X, y)
    assert gs.batched_
    npt.assert_allclose(gs.cv_results_["mean_test_score"], sk.cv_results_["mean_test_score"], rtol=1e-7)
    assert gs.best_index_ == _select_best_index_onestd(True, "score", sk.cv_results_)


def test_line_search_with_the_median_scorer_batches_every_line():
    X, y, _ = _data(100, 20, 8)
    groups = np.repeat(np.arange(5), 4)
    cv = KFold(4)
    grid = [("alpha", [0.01, 0.05, 0.2]), ("l1_ratio", [0.2, 0.8])]
    est = SparseGroupLasso(groups=groups, solver_options=OPTS)
    ls = LineSearchCV(est, grid, cv=cv, n_iter=3, scoring="neg_median_absolute_error").fit(X, y)
    assert all(h.batched_ for h in ls.history_)
    best = {"alpha": 0.01, "l1_ratio": 0.2}
    for i in range(3):
        name, values = grid[i % 2]
        line = {k: ([best[k]] if k != name else values) for k, _ in grid}
        g = SkGS(est, line, cv=cv, scoring="neg_median_absolute_error").fit(X, y)
        npt.assert_allclose(ls.history_[i].cv_results_["mean_test_score"], g.cv_results_["mean_test_score"], rtol=1e-7)
        best = dict(g.best_params_)
    assert ls.best_params_ == best

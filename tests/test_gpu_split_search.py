"""Batched CV searches over splits that are not one partition of the rows (repeated, shuffled, leave-one-out,
time-series and grouped splitters): cv_results_, best_params_ and the refit equal sklearn's per-fit loop over the
same engine-backed estimator, and single cells equal the CPU oracle on X[train]."""

import warnings

import numpy as np
import numpy.testing as npt
import pytest
import sklearn
from sklearn.base import clone
from sklearn.metrics import get_scorer
from sklearn.model_selection import GridSearchCV as SkGS
from sklearn.model_selection import (GroupKFold, KFold, LeaveOneGroupOut, LeaveOneOut, RepeatedKFold, ShuffleSplit,
                                     TimeSeriesSplit)

pytestmark = pytest.mark.gpu

import oracle.reference as R  # noqa: E402
from sparselm_b200.model import AdaptiveLasso, GroupLasso, Lasso, OverlapGroupLasso, SparseGroupLasso  # noqa: E402
from sparselm_b200.model_selection import GridSearchCV, LineSearchCV  # noqa: E402

# both sides of a comparison stop at this relative duality gap along different paths: at 1e-12 the CV scores of a
# KFold(20) standardized search still differ by 3e-7 relative, at 1e-14 by 4e-9 (B200), below the rtol 1e-7 checked
OPTS = {"tol": 1e-14}


def _data(n, p, seed, intercept=0.0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    y = X[:, :4] @ [2.0, -1.0, 1.0, 0.5] + 0.4 * rng.standard_normal(n) + intercept
    return X, y, rng


def _sk_search(est, grid, cv, scoring, X, y, fit_params):
    """sklearn's per-fit loop with this project's contract for fit params: sample_weight reaches fit only and the
    CV scores stay unweighted (as the reference's loop and the partition path score).  Recent sklearn forwards
    sample_weight to the scorer by default; metadata routing asks for the project's semantics explicitly."""
    if fit_params.get("sample_weight") is None:
        return SkGS(est, grid, cv=cv, scoring=scoring).fit(X, y, **fit_params)
    with sklearn.config_context(enable_metadata_routing=True):
        scorer = get_scorer(scoring).set_score_request(sample_weight=False)
        return SkGS(clone(est).set_fit_request(sample_weight=True), grid, cv=cv, scoring=scorer).fit(X, y, **fit_params)


def _compare(gs, sk, n_splits, metrics=("score",), train=False):
    assert gs.batched_ and gs.n_splits_ == n_splits
    for m in metrics:
        kinds = ("test", "train") if train else ("test",)
        for kind in kinds:
            for key in [f"split{i}_{kind}_{m}" for i in range(n_splits)] + [f"mean_{kind}_{m}", f"std_{kind}_{m}"]:
                npt.assert_allclose(gs.cv_results_[key], sk.cv_results_[key], rtol=1e-7, atol=1e-10, equal_nan=True,
                                    err_msg=key)
        npt.assert_array_equal(gs.cv_results_[f"rank_test_{m}"], sk.cv_results_[f"rank_test_{m}"])
    assert gs.best_params_ == sk.best_params_
    npt.assert_allclose(gs.best_estimator_.coef_, sk.best_estimator_.coef_, atol=1e-7)


def _case(name):
    """(estimator, grid, cv, X, y, fit params, oracle name, oracle kwargs)"""
    if name == "repeated_kfold_lasso":
        X, y, _ = _data(120, 30, 1, intercept=1.5)
        return (Lasso(fit_intercept=True, solver_options=OPTS), {"alpha": [0.005, 0.03, 0.2]},
                RepeatedKFold(n_splits=5, n_repeats=2, random_state=0), X, y, {}, "Lasso", dict(fit_intercept=True))
    if name == "shuffle_split_sgl_weighted":
        X, y, rng = _data(130, 24, 2, intercept=0.8)
        groups = rng.permutation(np.repeat(np.arange(6), 4))
        sw = 0.2 + 2.0 * rng.random(130)
        return (SparseGroupLasso(groups=groups, l1_ratio=0.4, fit_intercept=True, solver_options=OPTS),
                {"alpha": [0.003, 0.02, 0.1]}, ShuffleSplit(6, test_size=0.2, train_size=0.5, random_state=1), X, y,
                {"sample_weight": sw}, "SparseGroupLasso", dict(groups=groups, l1_ratio=0.4, fit_intercept=True))
    if name == "leave_one_out_adaptive":
        X, y, _ = _data(40, 12, 3)
        return (AdaptiveLasso(solver_options=OPTS), {"alpha": [0.01, 0.05, 0.2]}, LeaveOneOut(), X, y, {},
                "AdaptiveLasso", {})
    if name == "time_series_overlap":
        X, y, _ = _data(100, 20, 4)
        # the groups of every feature: groups of four, the last feature of each also in the next group
        group_list = [[j // 4] + ([j // 4 + 1] if j % 4 == 3 and j < 19 else []) for j in range(20)]
        return (OverlapGroupLasso(group_list=group_list, solver_options=OPTS), {"alpha": [0.01, 0.05, 0.3]},
                TimeSeriesSplit(4), X, y, {}, "OverlapGroupLasso", dict(group_list=group_list))
    if name == "kfold20_group_standardize":
        X, y, _ = _data(120, 20, 5, intercept=-1.0)
        groups = np.repeat(np.arange(5), 4)
        return (GroupLasso(groups=groups, standardize=True, fit_intercept=True, solver_options=OPTS),
                {"alpha": [0.01, 0.05, 0.3]}, KFold(20), X, y, {}, "GroupLasso",
                dict(groups=groups, standardize=True, fit_intercept=True))
    if name == "group_kfold_lasso":
        X, y, rng = _data(120, 16, 6)
        return (Lasso(solver_options=OPTS), {"alpha": [0.01, 0.05, 0.2]}, GroupKFold(16), X, y,
                {"groups": rng.integers(0, 20, 120)}, "Lasso", {})
    if name == "leave_one_group_out_sgl":
        X, y, rng = _data(120, 16, 7, intercept=0.5)
        groups = np.repeat(np.arange(4), 4)
        sw = 0.5 + rng.random(120)
        return (SparseGroupLasso(groups=groups, fit_intercept=True, solver_options=OPTS), {"alpha": [0.01, 0.05, 0.2]},
                LeaveOneGroupOut(), X, y, {"groups": np.arange(120) % 20, "sample_weight": sw}, "SparseGroupLasso",
                dict(groups=groups, fit_intercept=True))
    raise KeyError(name)


CASES = ["repeated_kfold_lasso", "shuffle_split_sgl_weighted", "leave_one_out_adaptive", "time_series_overlap",
         "kfold20_group_standardize", "group_kfold_lasso", "leave_one_group_out_sgl"]


@pytest.mark.parametrize("name", CASES)
def test_split_search_matches_sklearn_loop_and_oracle(name):
    est, grid, cv, X, y, fit_params, oname, okw = _case(name)
    scoring = "neg_mean_squared_error"
    gs = GridSearchCV(est, grid, cv=cv, scoring=scoring).fit(X, y, **fit_params)
    sk = _sk_search(est, grid, cv, scoring, X, y, fit_params)
    splits = list(cv.split(X, y, fit_params.get("groups")))
    _compare(gs, sk, len(splits))
    assert (gs.solver_info_["status"] == 0).all()
    sw = fit_params.get("sample_weight")
    # a few cells against the CPU oracle fitted on the split's training rows
    for s in (0, len(splits) - 1):
        tr, te = splits[s]
        for ci in (0, len(grid["alpha"]) - 1):
            b, icpt = R.fit(oname, X[tr], y[tr], alpha=grid["alpha"][ci], sample_weight=None if sw is None else sw[tr],
                            **okw)
            ref = -np.mean((y[te] - X[te] @ b - icpt) ** 2)
            assert gs.cv_results_[f"split{s}_test_score"][ci] == pytest.approx(ref, rel=1e-6, abs=1e-9)


def test_leave_one_out_r2_is_nan_like_sklearn():
    X, y, _ = _data(40, 10, 8)
    est = Lasso(solver_options=OPTS)
    grid = {"alpha": [0.01, 0.1]}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        gs = GridSearchCV(est, grid, cv=LeaveOneOut(), scoring="r2").fit(X, y)
        sk = SkGS(est, grid, cv=LeaveOneOut(), scoring="r2").fit(X, y)
    assert np.isnan(sk.cv_results_["split0_test_score"]).all()
    _compare(gs, sk, 40)
    from sklearn.exceptions import UndefinedMetricWarning

    with pytest.warns(UndefinedMetricWarning):
        GridSearchCV(est, grid, cv=LeaveOneOut(), scoring="r2").fit(X, y)


def test_multi_metric_with_train_scores_on_shuffle_split():
    X, y, _ = _data(90, 16, 9, intercept=1.0)
    groups = np.repeat(np.arange(4), 4)
    est = GroupLasso(groups=groups, fit_intercept=True, solver_options=OPTS)
    grid = {"alpha": [0.01, 0.05, 0.2, 0.8]}
    scoring = {"rmse": "neg_root_mean_squared_error", "mae": "neg_mean_absolute_error", "r2": "r2"}
    # train_size 0.3: training rows built directly; 0.6: downdated (train scores = all rows - rows outside)
    for train_size in (0.3, 0.6):
        cv = ShuffleSplit(5, test_size=0.2, train_size=train_size, random_state=2)
        gs = GridSearchCV(est, grid, cv=cv, scoring=scoring, refit="mae", return_train_score=True).fit(X, y)
        sk = SkGS(est, grid, cv=cv, scoring=scoring, refit="mae", return_train_score=True).fit(X, y)
        assert gs.multimetric_
        _compare(gs, sk, 5, metrics=tuple(scoring), train=True)


def test_line_search_with_repeated_kfold_prepares_the_splits_once(monkeypatch):
    from sparselm_b200.engine import Engine

    X, y, _ = _data(100, 20, 10)
    groups = np.repeat(np.arange(5), 4)
    cv = RepeatedKFold(n_splits=4, n_repeats=2, random_state=3)
    grid = [("alpha", [0.01, 0.05, 0.2]), ("l1_ratio", [0.2, 0.8])]
    est = SparseGroupLasso(groups=groups, solver_options=OPTS)
    calls = {"prepare": 0, "prepare_splits": 0}
    for name in calls:
        def spy(self, *a, _name=name, _orig=getattr(Engine, name), **k):
            calls[_name] += 1
            return _orig(self, *a, **k)

        monkeypatch.setattr(Engine, name, spy)
    # a KFold partition takes the fold path: its folds are prepared once too, whatever the identity of the y view
    # check_X_y returns at every line
    kf = LineSearchCV(est, grid, cv=KFold(4), n_iter=3).fit(X, y)
    assert calls == {"prepare": 1, "prepare_splits": 0}
    assert all(h.batched_ for h in kf.history_)
    ls = LineSearchCV(est, grid, cv=cv, n_iter=3).fit(X, y)
    assert calls["prepare_splits"] == 1
    assert all(h.batched_ for h in ls.history_)
    # the explicit loop of 1-D searches
    best = {"alpha": 0.01, "l1_ratio": 0.2}
    for i in range(3):
        name, values = grid[i % 2]
        line = {k: ([best[k]] if k != name else values) for k, _ in grid}
        g = SkGS(est, line, cv=cv, scoring="neg_root_mean_squared_error").fit(X, y)
        npt.assert_allclose(ls.history_[i].cv_results_["mean_test_score"], g.cv_results_["mean_test_score"], rtol=1e-7)
        best = dict(g.best_params_)
    assert ls.best_params_ == best

"""Host side of StabilitySelection: the subsample draws, parameter checks, the stability statistics and the
candidate descriptions it shares with GridSearchCV.  No GPU needed."""

import warnings
from types import SimpleNamespace

import numpy as np
import numpy.testing as npt
import pytest
from sklearn.base import clone
from sklearn.linear_model import Lasso as SkLasso
from sklearn.model_selection import ParameterGrid

from sparselm_b200.model import (AdaptiveLasso, GroupLasso, Lasso, OrdinaryLeastSquares, OverlapGroupLasso,
                                 SparseGroupLasso)
from sparselm_b200.model_selection import describe_candidates
from sparselm_b200.stability import StabilitySelection, draw_subsamples, selection_summary


@pytest.mark.parametrize("n", [40, 41])
def test_subsamples_have_the_right_size_and_no_repeated_row(n):
    subs = draw_subsamples(n, 10, 0.3, False, random_state=0)
    assert len(subs) == 10
    for s in subs:
        assert len(s) == int(np.floor(0.3 * n)) and len(np.unique(s)) == len(s)
        assert s.min() >= 0 and s.max() < n and np.all(np.diff(s) > 0)
    again = draw_subsamples(n, 10, 0.3, False, random_state=0)
    assert all(np.array_equal(a, b) for a, b in zip(subs, again))
    other = draw_subsamples(n, 10, 0.3, False, random_state=1)
    assert not all(np.array_equal(a, b) for a, b in zip(subs, other))


@pytest.mark.parametrize("n", [40, 41])
def test_complementary_pairs_are_disjoint_and_cover_every_row(n):
    subs = draw_subsamples(n, 8, 0.5, True, random_state=np.random.RandomState(3))
    assert len(subs) == 8
    for a, b in zip(subs[0::2], subs[1::2]):
        assert len(a) == n // 2 and len(b) == n - n // 2  # the complement of an odd n has ceil(n / 2) rows
        assert len(np.intersect1d(a, b)) == 0
        npt.assert_array_equal(np.union1d(a, b), np.arange(n))


def _data(n=30, p=12):
    rng = np.random.default_rng(0)
    return rng.standard_normal((n, p)), rng.standard_normal(n)


@pytest.mark.parametrize("kwargs", [
    dict(sample_fraction=0.0), dict(sample_fraction=1.0), dict(sample_fraction=1.5),
    dict(threshold=0.0), dict(threshold=1.01), dict(threshold=-0.2),
    dict(complementary_pairs=True, sample_fraction=0.6),
    dict(complementary_pairs=True, n_subsamples=5),
    dict(complementary_pairs=False, sample_fraction=0.05),  # one row of 30
    dict(selection_tol=-1.0),
])
def test_bad_parameters_raise(kwargs):
    X, y = _data()
    with pytest.raises(ValueError):
        StabilitySelection(Lasso(), {"alpha": [0.1]}, **kwargs).fit(X, y)


def test_a_subsample_of_fewer_than_two_rows_raises():
    with pytest.raises(ValueError):
        draw_subsamples(3, 2, 0.5, True)  # halves of one row
    with pytest.raises(ValueError):
        draw_subsamples(5, 2, 0.3, False)


@pytest.mark.parametrize("est", [OrdinaryLeastSquares(), SkLasso(), "lasso"])
def test_estimators_without_an_engine_penalty_raise(est):
    X, y = _data()
    with pytest.raises(ValueError):
        StabilitySelection(est, {"alpha": [0.1]}).fit(X, y)


@pytest.mark.parametrize("sw", [np.zeros(30), -np.ones(30), np.r_[np.ones(29), np.nan], np.ones(29)])
def test_weights_that_are_not_strictly_positive_raise(sw):
    X, y = _data()
    with pytest.raises(ValueError):
        StabilitySelection(Lasso(), {"alpha": [0.1]}).fit(X, y, sample_weight=sw)


def test_unknown_grid_parameter_raises():
    X, y = _data()
    with pytest.raises(ValueError):
        StabilitySelection(Lasso(), {"beta": [0.1]}).fit(X, y)


def test_selection_summary_matches_a_hand_computation():
    # 4 subsamples, p = 5 features, 2 candidates
    counts = np.array([[4, 3], [0, 1], [2, 2], [0, 0], [1, 4]])
    union = np.array([[1, 0, 1, 0, 1],
                      [1, 1, 0, 0, 1],
                      [1, 0, 1, 0, 1],
                      [1, 0, 0, 0, 1]], dtype=bool)
    stab, scores, q, bound = selection_summary(counts, union, 0.75)
    npt.assert_array_equal(stab, counts / 4.0)
    npt.assert_array_equal(scores, [1.0, 0.25, 0.5, 0.0, 1.0])
    assert q == (3 + 3 + 3 + 2) / 4
    assert bound == pytest.approx(2.75 ** 2 / (0.5 * 5), rel=1e-15)
    assert selection_summary(counts, union, 0.5)[3] == np.inf
    assert selection_summary(counts, union, 0.3)[3] == np.inf


def _plan_before_refactor(est, candidates, X, y):
    """The candidate descriptions GridSearchCV's plan made before describe_candidates: a fresh estimator per
    candidate, every parameter validated."""
    ests, specs = [], []
    for c in candidates:
        work = clone(est).set_params(**c)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)
            work._validate_hyperparams(X, y)
        ests.append(SimpleNamespace(fit_intercept=bool(work.fit_intercept)))
        specs.append(work._problem_spec(X.shape[1]))
    return ests, specs


def _same(a, b):
    if isinstance(a, dict):
        return isinstance(b, dict) and a.keys() == b.keys() and all(_same(a[k], b[k]) for k in a)
    if isinstance(a, np.ndarray) or isinstance(b, np.ndarray):
        return np.array_equal(a, b)
    return a == b


@pytest.mark.parametrize("est,grid", [
    (Lasso(), {"alpha": [0.3, 0.1, 0.01], "fit_intercept": [True, False]}),
    (GroupLasso(groups=np.arange(12) % 4), {"alpha": [0.2, 0.05]}),
    (SparseGroupLasso(groups=np.arange(12) % 3), {"alpha": [0.2, 0.05], "l1_ratio": [0.3, 0.8]}),
    (OverlapGroupLasso(group_list=[[j % 4, (j + 1) % 4] for j in range(12)]), {"alpha": [0.2, 0.05]}),
    (AdaptiveLasso(), {"alpha": [0.2, 0.05]}),
    (SparseGroupLasso(groups=np.arange(12) % 3, standardize=True), {"alpha": [0.2, 0.05]}),
])
def test_describe_candidates_gives_the_specs_of_the_old_plan(est, grid):
    X, y = _data()
    candidates = list(ParameterGrid(grid))
    ests, specs = describe_candidates(est, candidates, X, y)
    ref_ests, ref_specs = _plan_before_refactor(est, candidates, X, y)
    assert [e.fit_intercept for e in ests] == [e.fit_intercept for e in ref_ests]
    for s, r in zip(specs, ref_specs):
        for name in s.__dataclass_fields__:
            assert _same(getattr(s, name), getattr(r, name)), name


def test_describe_candidates_calls_on_first_once_with_the_first_candidate():
    X, y = _data()
    seen = []
    ests, specs = describe_candidates(Lasso(), [{"alpha": 0.5}, {"alpha": 0.1}], X, y,
                                      on_first=lambda e, s: seen.append((e, s)))
    assert len(seen) == 1 and seen[0][1] is specs[0] and seen[0][0] is ests[0]


def test_clone_and_get_params_round_trip():
    sel = StabilitySelection(Lasso(fit_intercept=True), {"alpha": [0.1, 0.2]}, n_subsamples=20, threshold=0.7,
                             random_state=4)
    c = clone(sel)
    assert c.get_params(deep=False).keys() == sel.get_params(deep=False).keys()
    assert c.threshold == 0.7 and c.n_subsamples == 20 and c.random_state == 4
    assert c.estimator.fit_intercept and c.param_grid == {"alpha": [0.1, 0.2]}

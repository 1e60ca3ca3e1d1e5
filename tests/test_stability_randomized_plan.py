"""Host side of randomized stability selection and of the group-level frequencies: the weakness parameter, the weight
draws, the group statistics, when the group attributes exist, and which device calls the drivers make (a mocked
engine on the CPU).  No GPU needed."""

from types import SimpleNamespace

import numpy as np
import numpy.testing as npt
import pytest
import torch
from sklearn.base import clone

import sparselm_b200.model_selection as MS
import sparselm_b200.stability as ST
from sparselm_b200.model import (AdaptiveGroupLasso, AdaptiveLasso, AdaptiveOverlapGroupLasso,
                                 AdaptiveRidgedGroupLasso, AdaptiveSparseGroupLasso, GroupLasso, Lasso,
                                 OverlapGroupLasso, RidgedGroupLasso, SparseGroupLasso)
from sparselm_b200.model_selection import describe_candidates
from sparselm_b200.stability import StabilitySelection, draw_subsamples, draw_weights, selection_summary


def _data(n=31, p=12):
    rng = np.random.default_rng(0)
    return rng.standard_normal((n, p)), rng.standard_normal(n)


class _FakeEngine:
    """The engine calls of batched_selection on CPU tensors: chunk Grams are left as they are, every fit is all
    zeros, and the scaling and group-count calls are recorded."""

    def __init__(self):
        self.torch = torch
        self.device = torch.device("cpu")
        self.scale_calls = []
        self.group_calls = []

    def to_device(self, a, dtype=None):
        t = torch.as_tensor(np.ascontiguousarray(a))
        return t if dtype is None else t.to(dtype)

    def prepare_splits(self, X, y, splits, fit_intercept=False, sample_weight=None, col_perm=None):
        n, p = X.shape
        return SimpleNamespace(pa=p + 4, p=p, direct=np.array([len(tr) <= n - len(tr) for tr, _ in splits]))

    def split_chunk(self, sd, s0, s1, buf):
        d = sd.direct[s0:s1]
        order = np.concatenate([s0 + np.flatnonzero(d), s0 + np.flatnonzero(~d)])
        return order, SimpleNamespace(G_train=buf[:s1 - s0])

    def gram_scale(self, G, p, weights, slots):
        self.scale_calls.append((G.shape[0], p, weights.numpy().copy(), np.asarray(slots).copy()))

    def support_counts(self, coef, K, rel_tol, counts, union):
        pass

    def group_support_counts(self, coef, K, rel_tol, gptr_dev, counts, union):
        self.group_calls.append(gptr_dev.numpy().copy())


def _fake_solve(engine, fd, specs, **opts):
    F = fd.G_train.shape[0]
    K = len(specs)
    ldz = max(8, (K + 7) // 8 * 8)
    z = np.zeros((F, ldz))
    return dict(coef=torch.zeros((F, specs[0].p, ldz), dtype=torch.float64), n_iter=z.astype(int),
                status=z.astype(int), gap=z, n_pass=z.astype(int), n_unconverged=0, iters_run=0)


@pytest.fixture
def fake(monkeypatch):
    eng = _FakeEngine()
    monkeypatch.setattr(ST, "get_engine", lambda *a, **k: eng)
    monkeypatch.setattr(MS, "solve_specs", _fake_solve)
    return eng


# ---- parameters and draws -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("weakness", [0.0, -0.5, 1.5, np.nan, np.inf, -np.inf, "0.5"])
def test_bad_weakness_raises(weakness):
    X, y = _data()
    with pytest.raises(ValueError):
        StabilitySelection(Lasso(), {"alpha": [0.1]}, weakness=weakness).fit(X, y)
    if not isinstance(weakness, str):
        with pytest.raises(ValueError):
            draw_weights(4, 3, weakness, 0)


@pytest.mark.parametrize("weakness", [1.0, 1, 0.5, 1e-3])
def test_weakness_in_range_is_accepted(weakness):
    StabilitySelection(Lasso(), {"alpha": [0.1]}, weakness=weakness)._check_params()


@pytest.mark.parametrize("weakness", [1.0, 0.5, 0.2])
@pytest.mark.parametrize("pairs", [True, False])
def test_subsamples_do_not_depend_on_the_weakness(fake, weakness, pairs):
    X, y = _data()
    frac = 0.5 if pairs else 0.4
    sel = StabilitySelection(Lasso(), {"alpha": [0.1, 0.01]}, n_subsamples=6, sample_fraction=frac,
                             complementary_pairs=pairs, weakness=weakness, random_state=7).fit(X, y)
    ref = draw_subsamples(31, 6, frac, pairs, random_state=7)
    assert len(sel.subsamples_) == len(ref)
    assert all(np.array_equal(a, b) for a, b in zip(sel.subsamples_, ref))


def test_weights_take_the_two_values_and_follow_the_subsamples(fake):
    X, y = _data(p=40)
    sel = StabilitySelection(Lasso(), {"alpha": [0.1]}, n_subsamples=10, weakness=0.3, random_state=3).fit(X, y)
    w = sel.weights_
    assert w.dtype == np.float64 and w.shape == (10, 40)
    assert set(np.unique(w)) == {0.3, 1.0}
    # drawn from the same generator, after the subsamples
    rng = np.random.RandomState(3)
    draw_subsamples(31, 10, 0.5, True, rng)
    npt.assert_array_equal(w, draw_weights(10, 40, 0.3, rng))


def test_weights_are_ones_at_weakness_one(fake):
    X, y = _data()
    sel = StabilitySelection(Lasso(), {"alpha": [0.1]}, n_subsamples=4, random_state=0).fit(X, y)
    npt.assert_array_equal(sel.weights_, np.ones((4, 12)))
    assert sel.weights_.dtype == np.float64
    npt.assert_array_equal(draw_weights(3, 5, 1.0, 0), np.ones((3, 5)))


def test_clone_and_get_params_round_trip_keep_the_weakness():
    sel = StabilitySelection(Lasso(), {"alpha": [0.1]}, weakness=0.25, random_state=4)
    assert sel.get_params(deep=False)["weakness"] == 0.25
    c = clone(sel)
    assert c.weakness == 0.25 and c.get_params(deep=False).keys() == sel.get_params(deep=False).keys()
    assert StabilitySelection(Lasso(), {"alpha": [0.1]}).weakness == 1.0


# ---- group statistics ---------------------------------------------------------------------------------------------
def test_group_summary_matches_a_hand_computation():
    # 4 subsamples, G = 3 groups, 2 candidates
    counts = np.array([[4, 2], [1, 3], [0, 0]])
    union = np.array([[1, 1, 0],
                      [1, 0, 0],
                      [1, 1, 0],
                      [1, 1, 0]], dtype=bool)
    stab, scores, q, bound = selection_summary(counts, union, 0.8)
    npt.assert_array_equal(stab, [[1.0, 0.5], [0.25, 0.75], [0.0, 0.0]])
    npt.assert_array_equal(scores, [1.0, 0.75, 0.0])
    assert q == (2 + 1 + 2 + 2) / 4
    assert bound == pytest.approx(1.75 ** 2 / (0.6 * 3), rel=1e-15)  # G = 3 in place of p


_GROUPS = np.array([3, 1, 1, 7, 3, 3, 1, 7, 7, 7, 2, 2])  # labels in no order: col_perm is not the identity


@pytest.mark.parametrize("est", [
    GroupLasso(groups=_GROUPS), SparseGroupLasso(groups=_GROUPS), RidgedGroupLasso(groups=_GROUPS),
    AdaptiveGroupLasso(groups=_GROUPS), AdaptiveSparseGroupLasso(groups=_GROUPS),
    AdaptiveRidgedGroupLasso(groups=_GROUPS), SparseGroupLasso(groups=_GROUPS, standardize=True),
])
def test_partition_estimators_have_group_results(fake, est):
    X, y = _data()
    sel = StabilitySelection(est, {"alpha": [0.1, 0.01]}, n_subsamples=4, random_state=0).fit(X, y)
    npt.assert_array_equal(sel.group_labels_, [1, 2, 3, 7])
    assert sel.group_stability_scores_.shape == (4, 2) and sel.group_scores_.shape == (4,)
    assert sel.group_selected_size_ == 0.0 and sel.group_expected_false_positives_ == 0.0
    # one group count per chunk, with the group table in the design's column order
    assert len(fake.group_calls) == 1
    npt.assert_array_equal(fake.group_calls[0], [0, 3, 5, 8, 12])


def test_a_group_lasso_without_groups_has_one_group_per_feature(fake):
    X, y = _data()
    sel = StabilitySelection(GroupLasso(), {"alpha": [0.1]}, n_subsamples=4, random_state=0)
    with pytest.warns(UserWarning):
        sel.fit(X, y)
    npt.assert_array_equal(sel.group_labels_, np.arange(12))
    assert sel.group_stability_scores_.shape == (12, 1)


@pytest.mark.parametrize("est,grid", [
    (Lasso(), {"alpha": [0.1]}),
    (AdaptiveLasso(), {"alpha": [0.1]}),
    (OverlapGroupLasso(group_list=[[j % 4, (j + 1) % 4] for j in range(12)]), {"alpha": [0.1]}),
    (AdaptiveOverlapGroupLasso(group_list=[[j % 3] for j in range(12)]), {"alpha": [0.1]}),
    (GroupLasso(groups=_GROUPS), {"alpha": [0.1], "groups": [_GROUPS, np.arange(12) // 3]}),
])
def test_group_results_are_none_without_a_partition(fake, est, grid):
    X, y = _data()
    sel = StabilitySelection(est, grid, n_subsamples=4, random_state=0).fit(X, y)
    for name in ("group_labels_", "group_stability_scores_", "group_scores_", "group_selected_size_",
                 "group_expected_false_positives_"):
        assert getattr(sel, name) is None, name
    assert fake.group_calls == []


# ---- which calls the drivers make ---------------------------------------------------------------------------------
@pytest.mark.parametrize("est", [Lasso(), SparseGroupLasso(groups=_GROUPS)])
def test_no_scaling_call_at_weakness_one(fake, est):
    X, y = _data()
    StabilitySelection(est, {"alpha": [0.1, 0.01]}, n_subsamples=20, random_state=0).fit(X, y)
    assert fake.scale_calls == []


@pytest.mark.parametrize("est", [Lasso(), SparseGroupLasso(groups=_GROUPS)])
def test_one_scaling_call_per_chunk_with_the_weights_in_column_order(fake, est):
    X, y = _data()
    sel = StabilitySelection(est, {"alpha": [0.1, 0.01], "fit_intercept": [False, True]}, n_subsamples=20,
                             weakness=0.5, random_state=0).fit(X, y)
    _, specs = describe_candidates(est, sel.candidates_, X, y)
    perm = specs[0].col_perm
    table = sel.weights_ if perm is None else sel.weights_[:, perm]
    # two batches (fit_intercept) x two chunks (16 + 4 subsamples)
    assert [c[0] for c in fake.scale_calls] == [16, 4, 16, 4]
    seen = []
    for S, p, w, slots in fake.scale_calls:
        assert p == 12 and len(slots) == S
        npt.assert_array_equal(w, table)
        seen.append(np.sort(slots))
    npt.assert_array_equal(np.concatenate(seen[:2]), np.arange(20))
    npt.assert_array_equal(np.concatenate(seen[2:]), np.arange(20))


def test_a_cv_split_search_passes_no_chunk_hook(monkeypatch):
    X, y = _data()
    est = Lasso()
    ests, specs = describe_candidates(est, [{"alpha": 0.1}], X, y)
    seen = []

    class Stop(Exception):
        pass

    def spy(*args, **kwargs):
        seen.append(kwargs)
        raise Stop

    monkeypatch.setattr(MS, "split_batches", spy)
    splits = [(np.arange(0, 20), np.arange(20, 31)), (np.arange(11, 31), np.arange(0, 11))]
    with pytest.raises(Stop):
        MS.batched_cv_splits(_FakeEngine(), X, y, splits, ests, specs, {}, "r2")
    assert len(seen) == 1 and seen[0].get("on_chunk") is None

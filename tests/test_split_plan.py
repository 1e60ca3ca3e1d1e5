"""Host side of the batched search over arbitrary CV splits: which path a search takes, the build mode and row
lists of every split, chunking, and sklearn's r2 rule for one-row test sets.  No GPU needed."""

import warnings

import numpy as np
import pytest
from sklearn.exceptions import UndefinedMetricWarning
from sklearn.model_selection import (GroupKFold, KFold, LeaveOneGroupOut, LeaveOneOut, RepeatedKFold, ShuffleSplit,
                                     TimeSeriesSplit)

from sparselm_b200.engine import plan_splits, split_chunks
from sparselm_b200.model_selection import _split_metric, _split_route

N = 40
X = np.zeros((N, 3))


def _splits(cv, groups=None):
    return list(cv.split(X, np.zeros(N), groups))


def test_partitions_of_at_most_15_folds_keep_the_fold_path():
    assert _split_route(_splits(KFold(5)), N) == "partition"
    assert _split_route(_splits(KFold(15)), N) == "partition"
    assert _split_route(_splits(KFold(5, shuffle=True, random_state=0)), N) == "partition"
    assert _split_route(_splits(GroupKFold(4), np.arange(N) % 8), N) == "partition"


def test_other_splitters_take_the_split_path():
    groups = np.arange(N) % 20
    for splits in (_splits(KFold(20)), _splits(LeaveOneOut()), _splits(RepeatedKFold(n_splits=5, n_repeats=2, random_state=0)),
                   _splits(ShuffleSplit(10, test_size=0.2, train_size=0.6, random_state=0)),
                   _splits(TimeSeriesSplit(4)), _splits(LeaveOneGroupOut(), groups), _splits(GroupKFold(16), groups)):
        assert _split_route(splits, N) == "splits"


def test_per_fit_loop_cases():
    splits = _splits(RepeatedKFold(n_splits=5, n_repeats=2, random_state=0))
    assert _split_route(splits, N, world=2) is None  # sharded search
    # a partition keeps the fold path on a sharded search too
    assert _split_route(_splits(KFold(5)), N, world=2) == "partition"
    tr = np.arange(10, N)
    assert _split_route([(tr, np.arange(10)), (tr, np.array([], dtype=int))], N) is None  # empty test set
    assert _split_route([(np.array([5]), np.arange(10))], N) is None  # one training row
    assert _split_route([(np.r_[tr, 11], np.arange(10))], N) is None  # repeated training row
    assert _split_route([(tr, np.r_[np.arange(10), 3])], N) is None  # repeated test row
    assert _split_route([(tr, np.r_[np.arange(10), 12])], N) is None  # a row in both sets
    assert _split_route([(tr, np.arange(N - 5, N + 1))], N) is None  # out of range


def _rows(ptr, vals, i):
    return vals[ptr[i]:ptr[i + 1]]


def test_build_mode_and_lists_leave_one_out():
    splits = _splits(LeaveOneOut())
    plan = plan_splits(splits, N)
    assert not plan["direct"].any()  # n-1 training rows, one row outside: downdate
    assert len(plan["direct_rows"]) == 0 and len(plan["out_rows"]) == N  # n indices, not n^2
    for s in range(N):
        assert list(_rows(plan["out_ptr"], plan["out_rows"], s)) == [s]
        assert list(_rows(plan["test_ptr"], plan["test_rows"], s)) == [s]
    np.testing.assert_array_equal(plan["n_obs"], N - 1)


def test_build_mode_and_lists_time_series():
    splits = _splits(TimeSeriesSplit(4))
    plan = plan_splits(splits, N)
    # training prefixes of 8, 16, 24, 32 rows: direct while the prefix is at most half of the rows
    np.testing.assert_array_equal(plan["direct"], [True, True, False, False])
    assert list(_rows(plan["direct_ptr"], plan["direct_rows"], 1)) == list(range(16))
    assert list(_rows(plan["out_ptr"], plan["out_rows"], 0)) == list(range(24, N))  # split 2
    assert list(_rows(plan["out_ptr"], plan["out_rows"], 1)) == list(range(32, N))  # split 3
    np.testing.assert_array_equal(plan["n_train"], [8, 16, 24, 32])


def test_build_mode_and_lists_shuffle_split_with_rows_in_neither_set():
    sw = 0.5 + np.arange(N) / N
    splits = _splits(ShuffleSplit(5, test_size=0.2, train_size=0.6, random_state=3))
    plan = plan_splits(splits, N, sw)
    assert not plan["direct"].any()  # 24 training rows vs 16 outside
    for s, (tr, te) in enumerate(splits):
        out = _rows(plan["out_ptr"], plan["out_rows"], s)
        np.testing.assert_array_equal(out, np.setdiff1d(np.arange(N), tr))
        assert set(te) < set(out)  # test rows and rows in neither set
        np.testing.assert_array_equal(_rows(plan["test_ptr"], plan["test_rows"], s), np.sort(te))
        assert plan["n_obs"][s] == pytest.approx(sw[tr].sum(), rel=1e-15)
    plan = plan_splits(_splits(ShuffleSplit(5, test_size=0.2, train_size=0.3, random_state=3)), N)
    assert plan["direct"].all() and len(plan["out_rows"]) == 0


def test_chunks_of_at_most_16_splits():
    assert [b - a for a, b in split_chunks(37)] == [16, 16, 5]
    assert split_chunks(37)[-1] == (32, 37)
    assert split_chunks(16) == [(0, 16)] and split_chunks(1) == [(0, 1)]


def test_r2_is_nan_on_a_one_row_test_set():
    sse, sae = np.array([0.5, 2.0]), np.array([0.7, 1.4])
    with pytest.warns(UndefinedMetricWarning):
        got = _split_metric("r2", sse, sae, 1, 0.0)
    assert np.isnan(got).all() and got.shape == (2,)
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        np.testing.assert_allclose(_split_metric("r2", sse, sae, 2, 4.0), 1.0 - sse / 4.0)
        np.testing.assert_allclose(_split_metric("neg_mean_squared_error", sse, sae, 1, 0.0), -sse)

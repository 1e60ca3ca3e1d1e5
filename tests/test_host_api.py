"""CPU tests: host-side logic of the estimator API, the C-ABI surface and the oracle."""

import ctypes
import os
import re

import numpy as np
import pytest

import oracle.reference as R
from sparselm_b200 import _build, _lib
from sparselm_b200.model import (
    AdaptiveGroupLasso,
    AdaptiveLasso,
    AdaptiveOverlapGroupLasso,
    AdaptiveRidgedGroupLasso,
    AdaptiveSparseGroupLasso,
    GroupLasso,
    Lasso,
    OverlapGroupLasso,
    RidgedGroupLasso,
    SparseGroupLasso,
)
from sparselm_b200.model._base import stack_specs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- C ABI surface ----------------------------------------------------------------------
def test_library_builds_and_exports_every_declared_symbol():
    path = _build.build()
    assert os.path.exists(path)
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "sparselm_b200.h")).read()
    declared = set(re.findall(r"\b(slm_[a-z_0-9]+)\s*\(", header))
    declared -= {"slm_ctx", "slm_batch"}
    assert declared, "no declarations found"
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
    assert lib.slm_version() >= 1
    assert lib.slm_padded_cols(4096) == 4104 and lib.slm_padded_cols(6) == 8


def test_batch_struct_layout_matches_header():
    # field order of the ctypes mirror == declaration order in the header
    header = open(os.path.join(ROOT, "include", "sparselm_b200.h")).read()
    body = header[header.index("typedef struct slm_batch {"):header.index("} slm_batch;")]
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = re.findall(r"\b([A-Za-z_0-9]+)(?:\[SLM_MAX_FOLDS\])?\s*;", body)
    assert names == [f[0] for f in _lib.SlmBatch._fields_]


def test_no_gpu_means_loud_failure():
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from sparselm_b200.engine import EngineError

    with pytest.raises(EngineError):
        Lasso(alpha=0.1).fit(np.eye(3), np.ones(3))
    h = ctypes.c_void_p()
    assert _lib.load().slm_create(0, ctypes.byref(h)) != 0


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "sparselm_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in src and "from oracle" not in src, f


# ---- error / warning contract (reference tests/test_lasso.py:203-260) -------------------
@pytest.fixture
def data():
    rng = np.random.default_rng(0)
    X = rng.standard_normal((25, 20))
    y = rng.standard_normal(25)
    groups = rng.integers(0, 4, size=20)
    groups[:4] = np.arange(4)
    return X, y, groups


def test_bad_inputs(data):
    X, y, groups = data
    rng = np.random.default_rng(1)
    bad_groups = rng.integers(0, 6, size=X.shape[1] - 1)
    gw = np.ones(len(np.unique(bad_groups)))
    with pytest.raises(ValueError):
        GroupLasso(bad_groups, group_weights=gw).fit(X, y)
    with pytest.raises(TypeError):
        GroupLasso("groups", group_weights=gw).fit(X, y)
    with pytest.raises(ValueError):
        GroupLasso(bad_groups, group_weights=np.ones(len(np.unique(bad_groups)) - 1)).fit(X, y)
    with pytest.raises(TypeError):
        GroupLasso(groups, group_weights="weights").fit(X, y)
    lasso = SparseGroupLasso(groups)
    for bad in (-1.0, 2.0):
        lasso.l1_ratio = bad
        with pytest.raises(ValueError):
            lasso.fit(X, y)
        with pytest.raises(ValueError):
            SparseGroupLasso(groups, l1_ratio=bad).fit(X, y)
    with pytest.raises(ValueError):
        OverlapGroupLasso(group_list=[[0]] * (X.shape[1] - 1)).fit(X, y)
    with pytest.raises(ValueError):
        RidgedGroupLasso(groups, delta=(1.0, 2.0)).fit(X, y)
    with pytest.raises(ValueError):
        Lasso(alpha=-1.0).fit(X, y)
    with pytest.raises(TypeError):
        Lasso(solver_options=[1]).fit(X, y)


def test_constructor_signatures_match_reference():
    import inspect

    sig = lambda c: list(inspect.signature(c).parameters)  # noqa: E731
    assert sig(Lasso) == ["alpha", "fit_intercept", "copy_X", "warm_start", "solver", "solver_options"]
    assert sig(GroupLasso)[:4] == ["groups", "alpha", "group_weights", "standardize"]
    assert sig(OverlapGroupLasso)[:4] == ["group_list", "alpha", "group_weights", "standardize"]
    assert sig(SparseGroupLasso)[:4] == ["groups", "l1_ratio", "alpha", "group_weights"]
    assert sig(RidgedGroupLasso)[:4] == ["groups", "alpha", "delta", "group_weights"]
    assert sig(AdaptiveLasso)[:5] == ["alpha", "max_iter", "eps", "tol", "update_function"]
    assert sig(AdaptiveGroupLasso)[:7] == ["groups", "alpha", "group_weights", "max_iter", "eps", "tol",
                                           "update_function"]
    for cls in (AdaptiveLasso, AdaptiveGroupLasso, AdaptiveOverlapGroupLasso, AdaptiveSparseGroupLasso,
                AdaptiveRidgedGroupLasso):
        e = cls()
        assert (e.max_iter, e.eps, e.tol, e.warm_start) == (3, 1e-6, 1e-10, True)
    assert RidgedGroupLasso().delta == (1.0,) and SparseGroupLasso().l1_ratio == 0.5


def test_get_set_params_clone_roundtrip(data):
    from sklearn.base import clone

    _, _, groups = data
    for est in (Lasso(alpha=0.3), SparseGroupLasso(groups, l1_ratio=0.2, alpha=2.0),
                AdaptiveOverlapGroupLasso(group_list=[[0, 1]] * 20, max_iter=5),
                AdaptiveRidgedGroupLasso(groups, delta=(3.0,))):
        c = clone(est)
        assert type(c) is type(est)
        for k, v in est.get_params().items():
            assert c.get_params()[k] is v or np.array_equal(c.get_params()[k], v)
        c.set_params(alpha=7.0)
        assert c.alpha == 7.0


# ---- penalty plumbing (reference tests/test_lasso.py:263-309) -----------------------------
def test_problem_specs_follow_reference_rules(data):
    _, _, groups = data
    p = 20
    G = len(np.unique(groups))
    gw = np.arange(1, G + 1, dtype=float)
    s = SparseGroupLasso(groups, l1_ratio=0.25, alpha=0.5, group_weights=gw)._problem_spec(p)
    assert s.lam1 == 0.25 * 0.5
    np.testing.assert_allclose(s.w2, 0.75 * 0.5 * gw)
    # groups made contiguous: permuted labels are sorted
    assert np.all(np.diff(groups[s.col_perm]) >= 0)
    assert s.gptr[-1] == p and len(s.gptr) == G + 1
    r = RidgedGroupLasso(groups, alpha=2.0, delta=(4.0,))._problem_spec(p)
    np.testing.assert_array_equal(r.d2, 4.0 * np.ones(G))
    r = RidgedGroupLasso(groups, alpha=2.0, delta=3.0 * np.ones(G))._problem_spec(p)
    np.testing.assert_array_equal(r.d2, 3.0 * np.ones(G))
    a = AdaptiveGroupLasso(groups, alpha=0.5, group_weights=gw)._problem_spec(p)
    np.testing.assert_array_equal(a.w2, 0.5 * np.ones(G))  # no group_weights in pass 1
    assert a.adaptive["a2"] == 0.5 and a.adaptive["a1"] is None
    np.testing.assert_array_equal(a.gw, gw)
    asg = AdaptiveSparseGroupLasso(groups, l1_ratio=0.5, alpha=0.5)._problem_spec(p)
    assert asg.lam1 == 0.25 and asg.adaptive["a1"] == 0.25 and asg.adaptive["a2"] == 0.25
    al = AdaptiveLasso(alpha=0.3)._problem_spec(p)
    assert al.lam1 == 0.3 and al.adaptive["a1"] == 0.3 and al.adaptive["alpha"] == 0.3


def test_overlap_expansion_matches_reference_scan():
    rng = np.random.default_rng(2)
    p = 17
    group_list = [list(rng.choice(6, size=rng.integers(1, 4), replace=False)) for _ in range(p)]
    est = OverlapGroupLasso(group_list=group_list)
    ext_idx, gptr, ng = est._expansion(p)
    ref_idx, ref_groups, ref_ng = R.expand_overlap(group_list, p)
    np.testing.assert_array_equal(ext_idx, ref_idx)
    assert ng == ref_ng
    np.testing.assert_array_equal(np.repeat(np.arange(ng), np.diff(gptr)), ref_groups)


def test_stack_specs_shapes(data):
    _, _, groups = data
    specs = [SparseGroupLasso(groups, alpha=a)._problem_spec(20) for a in (0.1, 0.2, 0.3)]
    assert len({s.key for s in specs}) == 1
    g = stack_specs(specs)
    assert g.K == 3 and g.W2.shape == (len(np.unique(groups)), 3)
    np.testing.assert_allclose(g.lam1, [0.05, 0.1, 0.15])
    assert SparseGroupLasso(groups, alpha=0.1, fit_intercept=True)._problem_spec(20).key != specs[0].key


# ---- model selection host logic --------------------------------------------------------------
def test_one_std_rule_and_partition_helpers():
    from sklearn.model_selection import KFold, ShuffleSplit

    from sparselm_b200.model_selection import _is_partition, _metric, _select_best_index_onestd

    res = {
        "rank_test_score": np.array([3, 1, 2, 4]),
        "mean_test_score": np.array([-1.3, -1.0, -1.05, -2.0]),
        "std_test_score": np.array([0.1, 0.1, 0.1, 0.1]),
        "param_alpha": np.ma.MaskedArray([0.01, 0.1, 1.0, 10.0]),
        "params": [{}] * 4,
    }
    # candidates with alpha >= 0.1: target mean = -1.0 - 0.1 = -1.1 -> alpha=1.0 (-1.05) is closest
    assert _select_best_index_onestd(True, "score", res) == 2
    n = 23
    assert _is_partition(list(KFold(5).split(np.zeros(n))), n)
    assert _is_partition(list(KFold(5, shuffle=True, random_state=0).split(np.zeros(n))), n)
    assert not _is_partition(list(ShuffleSplit(3, random_state=0).split(np.zeros(n))), n)
    sse, sae = np.array([4.0, 0.0]), np.array([2.0, 0.0])
    np.testing.assert_allclose(_metric("neg_root_mean_squared_error", sse, sae, 4, 8.0), [-1.0, 0.0])
    np.testing.assert_allclose(_metric("neg_mean_squared_error", sse, sae, 4, 8.0), [-1.0, 0.0])
    np.testing.assert_allclose(_metric("neg_mean_absolute_error", sse, sae, 4, 8.0), [-0.5, 0.0])
    np.testing.assert_allclose(_metric("r2", sse, sae, 4, 8.0), [0.5, 1.0])


def test_miqp_names_exist_and_fail_loudly():
    from sparselm_b200.model import L1L0, L2L0, BestSubsetSelection, RegularizedL0, RidgedBestSubsetSelection

    for cls in (L1L0, L2L0, BestSubsetSelection, RegularizedL0, RidgedBestSubsetSelection):
        with pytest.raises(NotImplementedError):
            cls().fit(np.eye(3), np.ones(3))


# ---- host logic added with the widening rows (no GPU needed) ------------------------------
def test_device_metrics_forms():
    from sparselm_b200.model_selection import _device_metrics

    assert _device_metrics(None) == "r2"
    assert _device_metrics("neg_mean_absolute_error") == "neg_mean_absolute_error"
    assert _device_metrics("explained_variance") is None
    assert _device_metrics(["r2", "neg_mean_squared_error"]) == {"r2": "r2",
                                                                 "neg_mean_squared_error": "neg_mean_squared_error"}
    assert _device_metrics(("r2", "r2")) is None  # duplicate names: sklearn's own error path
    assert _device_metrics({"a": "r2", "b": "neg_root_mean_squared_error"}) == {
        "a": "r2", "b": "neg_root_mean_squared_error"}
    assert _device_metrics({"a": "r2", "b": "max_error"}) is None
    assert _device_metrics(lambda est, X, y: 0.0) is None
    assert _device_metrics([]) is None


def test_metric_formulas_match_sklearn():
    from sklearn.metrics import mean_absolute_error, mean_squared_error, r2_score

    from sparselm_b200.model_selection import _metric

    rng = np.random.default_rng(0)
    y, yp = rng.normal(size=40), rng.normal(size=40)
    sse, sae, sst = ((y - yp) ** 2).sum(), np.abs(y - yp).sum(), ((y - y.mean()) ** 2).sum()
    assert _metric("r2", sse, sae, 40, sst) == pytest.approx(r2_score(y, yp))
    assert _metric("neg_mean_squared_error", sse, sae, 40, sst) == pytest.approx(-mean_squared_error(y, yp))
    assert _metric("neg_root_mean_squared_error", sse, sae, 40, sst) == pytest.approx(-np.sqrt(mean_squared_error(y, yp)))
    assert _metric("neg_mean_absolute_error", sse, sae, 40, sst) == pytest.approx(-mean_absolute_error(y, yp))
    # constant target: sklearn's force_finite convention
    assert _metric("r2", np.array([0.0, 1.0]), None, 5, 0.0).tolist() == [1.0, 0.0]


def test_warm_start_views_are_lazy_and_first_fold_wins():
    import torch

    from sparselm_b200.model_selection import _WarmStarts

    B = torch.arange(2 * 3 * 8, dtype=torch.float64).reshape(2, 3, 8)  # [F, p, ldz]
    w = _WarmStarts()
    idxs = np.array([5, 2, 9])  # batch columns -> candidate indices
    w.add(B, idxs, [np.array([0, 2]), np.array([1, 2])])  # fold 0 solved 5 and 9, fold 1 solved 2 and 9
    assert torch.equal(w.get(5), B[0, :, 0])
    assert torch.equal(w.get(9), B[0, :, 1])  # the first fold that solved it
    assert torch.equal(w[2], B[1, :, 0])
    assert w.get(7) is None
    with pytest.raises(KeyError):
        w[7]


def _solve_out(rng, F, ldz):
    """The info part of a solve_specs output with F slots of ldz columns."""
    return dict(n_iter=rng.integers(1, 999, (F, ldz)).astype(np.int32),
                status=rng.integers(0, 3, (F, ldz)).astype(np.int32), gap=rng.random((F, ldz)),
                n_pass=rng.integers(1, 9, (F, ldz)).astype(np.int32), n_unconverged=int(rng.integers(1, 5)),
                iters_run=int(rng.integers(1, 99)), newton={"steps": F})


def test_candidate_batches_and_solve_info_of_sharded_folds_and_split_chunks():
    from types import SimpleNamespace

    from sparselm_b200.model_selection import _SolveInfo, candidate_batches
    from sparselm_b200.parallel import assign_columns

    specs = [SimpleNamespace(key=k, strength=s) for k, s in (("a", 0.3), ("a", 0.1), ("b", 0.2), ("a", 0.1))]
    batches = candidate_batches(specs)
    assert list(batches) == ["a", "b"] and batches["a"].tolist() == [1, 3, 0] and batches["b"].tolist() == [2]

    rng = np.random.default_rng(0)
    F, n_cand = 5, 9
    idxs = np.array([4, 0, 7, 2, 8, 1, 3, 6, 5])  # batch column k -> candidate
    full = _solve_out(rng, F, 16)  # one process solving every (fold, column)
    ref = _SolveInfo(n_cand, F)
    ref.record(full, range(F), [idxs] * F)
    for k, t in ref.tables.items():
        np.testing.assert_array_equal(t[idxs].T, full[k][:, :n_cand])
    # a sharded grid: rank r solved the columns mine[f] of fold f, packed at the front of its slot
    owner = assign_columns(F, n_cand, 2)
    ranks = []
    for r in range(2):
        mine = [np.flatnonzero(owner[f] == r) for f in range(F)]
        out = dict(full, iters_run=10 + r)
        for k in ref.tables:
            out[k] = np.zeros_like(full[k])
            for f in range(F):
                out[k][f, :len(mine[f])] = full[k][f, mine[f]]
        ranks.append(_SolveInfo(n_cand, F))
        ranks[-1].record(out, range(F), [idxs[m] for m in mine])

    class _TwoRanks:
        """All-reduce of two ranks: adds the other rank's buffer to this one's (and keeps this one's)."""
        world = 2

        def __init__(self, other=None):
            self.other = other

        def allreduce_sum_numpy(self, arr, device=None):
            self.sent = arr.copy()
            return arr if self.other is None else arr + self.other

    resid = [rng.random((2, 2, n_cand, F)) for _ in range(2)]
    first = _TwoRanks()
    ranks[1].allreduce(first, None, resid[1])
    got = ranks[0].allreduce(_TwoRanks(first.sent), None, resid[0])
    np.testing.assert_array_equal(got, resid[0] + resid[1])
    for k, t in ref.tables.items():
        assert ranks[0].tables[k].dtype == t.dtype
        np.testing.assert_array_equal(ranks[0].tables[k], t)
    assert ranks[0].n_unconverged == 2 * full["n_unconverged"]
    assert ranks[0].iters_run == 10 and ranks[0].newton == {"steps": F}  # not exchanged

    # chunks of arbitrary splits: slot f holds split order[f] (direct builds first), every slot solves the batch
    info = _SolveInfo(n_cand, 20)
    outs = []
    for c0, c1 in ((0, 16), (16, 20)):
        order = c0 + rng.permutation(c1 - c0)
        outs.append((order, _solve_out(rng, c1 - c0, 16)))
        info.record(outs[-1][1], order, [idxs] * len(order))
    for order, out in outs:
        for k, t in info.tables.items():
            np.testing.assert_array_equal(t[idxs][:, order].T, out[k][:, :n_cand])
    assert info.n_unconverged == sum(o["n_unconverged"] for _, o in outs)
    assert info.iters_run == sum(o["iters_run"] for _, o in outs) and info.newton == {"steps": 20}


def _residual_rows(r, y):
    """The [5][K] rows of slm_cv_score_stats for the residuals r [rows, K] of the targets y."""
    a = np.abs(r)
    return np.stack([(r * r).sum(0), a.sum(0), a.max(0), (a / np.maximum(np.abs(y), np.finfo(float).eps)[:, None]).sum(0),
                     np.median(a, axis=0)])


def test_score_assembly_on_a_partition_and_on_splits():
    from sklearn.exceptions import UndefinedMetricWarning
    from sklearn.metrics import (d2_absolute_error_score, mean_absolute_error, mean_absolute_percentage_error,
                                 median_absolute_error, r2_score, root_mean_squared_error)

    from sparselm_b200.model_selection import (_metric, _partition_cells, _residual_tables, _scores, _split_cells,
                                               _split_metric, _stat_mask)

    sk = {"r2": r2_score, "rmse": lambda a, b: -root_mean_squared_error(a, b),
          "mae": lambda a, b: -mean_absolute_error(a, b), "med": lambda a, b: -median_absolute_error(a, b),
          "mape": lambda a, b: -mean_absolute_percentage_error(a, b), "d2": d2_absolute_error_score}
    scoring = {"r2": "r2", "rmse": "neg_root_mean_squared_error", "mae": "neg_mean_absolute_error",
               "med": "neg_median_absolute_error", "mape": "neg_mean_absolute_percentage_error",
               "d2": "d2_absolute_error_score"}
    rng = np.random.default_rng(1)
    n, K = 23, 3
    y = rng.standard_normal(n)
    allrows = np.arange(n)

    def check(scores, cells, rows_of, preds):
        for c, rows in enumerate(rows_of):
            for m, fn in sk.items():
                if len(rows) < 2 and m in ("r2", "d2"):
                    continue
                want = [fn(y[rows], preds[c][rows, k]) for k in range(K)]
                np.testing.assert_allclose(scores[m][:, c], want, rtol=1e-10, err_msg=f"{m} cell {c}")

    # a partition in row order with a one-row fold: train sums as the pieces [0, r0) + [r1, n)
    folds = [np.arange(0, 1), np.arange(1, 12), np.arange(12, n)]
    preds = [y[:, None] + rng.standard_normal((n, K)) for _ in folds]
    resid = _residual_tables(K, len(folds), True, _stat_mask(scoring))
    trains = [np.setdiff1d(allrows, te) for te in folds]
    for f, (te, tr) in enumerate(zip(folds, trains)):
        r = y[:, None] - preds[f]
        resid[0][:, :, f] = _residual_rows(r[te], y[te])
        for lo, hi in ((0, te[0]), (te[-1] + 1, n)):
            if hi > lo:
                resid[1][:2, :, f] += _residual_rows(r[lo:hi], y[lo:hi])[:2]
        resid[1][2:, :, f] = _residual_rows(r[tr], y[tr])[2:]
    cells = _partition_cells(y, folds, scoring, True)
    for (n_tr, sst, _), te, tr in zip(cells[1], folds, trains):
        # the training sst is downdated from the sums over all rows
        s_tr, q_tr = float(y.sum()) - float(y[te].sum()), float((y * y).sum()) - float((y[te] ** 2).sum())
        assert n_tr == len(tr) and sst == q_tr - s_tr * s_tr / n_tr
        assert sst == pytest.approx(((y[tr] - y[tr].mean()) ** 2).sum(), rel=1e-12)
    with pytest.warns(UndefinedMetricWarning):  # d2 of the one-row fold
        test, train = _scores(scoring, _metric, resid, *cells)
    assert set(test) == set(train) == set(scoring)
    check(test, cells[0], folds, preds)
    check(train, cells[1], trains, preds)
    r0 = y[0] - preds[0][0]
    np.testing.assert_array_equal(test["r2"][:, 0], np.where(r0 == 0.0, 1.0, 0.0))  # force-finite r2 on one row
    assert np.isnan(test["d2"][:, 0]).all()
    # one metric: its table itself; no train cells, no train scores
    one, none = _scores("neg_mean_absolute_error", _metric, resid[:1, :2], cells[0])
    np.testing.assert_array_equal(one, test["mae"])
    assert none is None

    # arbitrary splits: a one-row test set, rows in neither set; the downdated train sums are all rows - out rows
    splits = [(np.arange(1, n), np.array([0])), (np.arange(0, 8), np.arange(15, n)), (np.arange(8, 20), np.arange(5))]
    preds = [y[:, None] + rng.standard_normal((n, K)) for _ in splits]
    resid = _residual_tables(K, len(splits), True, _stat_mask(scoring))
    for s, (tr, te) in enumerate(splits):
        r = y[:, None] - preds[s]
        out = np.setdiff1d(allrows, tr)
        resid[0][:, :, s] = _residual_rows(r[te], y[te])
        resid[1][:2, :, s] += -1.0 * _residual_rows(r[out], y[out])[:2]
        resid[1][:2, :, s] += _residual_rows(r, y)[:2]
        resid[1][2:, :, s] = _residual_rows(r[tr], y[tr])[2:]
    cells = _split_cells(y, splits, scoring, True)
    with pytest.warns(UndefinedMetricWarning):  # r2 and d2 of the one-row test set
        test, train = _scores(scoring, _split_metric, resid, *cells)
    check(test, cells[0], [te for _, te in splits], preds)
    check(train, cells[1], [tr for tr, _ in splits], preds)
    assert np.isnan(test["r2"][:, 0]).all() and np.isnan(test["d2"][:, 0]).all()

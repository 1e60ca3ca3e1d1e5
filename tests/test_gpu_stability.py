"""Stability selection on the GPU: slm_support_counts against numpy, StabilitySelection against sklearn's loop of
engine fits and against the CPU oracle over the same subsamples, known answers and the convergence warning."""

import warnings

import numpy as np
import numpy.testing as npt
import pytest
from sklearn.base import clone
from sklearn.exceptions import ConvergenceWarning

pytestmark = pytest.mark.gpu

import oracle.reference as R  # noqa: E402
from sparselm_b200.model import (AdaptiveLasso, GroupLasso, Lasso, OverlapGroupLasso, RidgedGroupLasso,  # noqa: E402
                                 SparseGroupLasso)
from sparselm_b200.stability import StabilitySelection, draw_subsamples  # noqa: E402

TOL = 1e-6
OPTS = {"tol": 1e-13}


# ---- kernel -------------------------------------------------------------------------------------------------------
def _np_counts(coef, K, tol):
    a = np.abs(coef[:, :, :K])
    mx = np.where(np.isnan(a), 0.0, a).max(axis=1)  # [F, K], NaN ignored
    with np.errstate(invalid="ignore"):
        sel = a > tol * mx[:, None, :]  # NaN is never selected
    return sel.sum(axis=0).astype(np.int32), sel.any(axis=2)


def _table(rng, F, p, ldz, K):
    c = rng.uniform(-1.0, 1.0, (F, p, ldz))
    c[rng.random((F, p, ldz)) < 0.4] = 0.0  # planted exact zeros
    top = rng.integers(0, p, (F, K))
    for f in range(F):
        for k in range(K):
            M = 8.0 * (1 + rng.random())
            c[f, top[f, k], k] = M * rng.choice([-1.0, 1.0])
            band = rng.integers(0, p, 3)
            thr = TOL * M
            c[f, band[0], k] = thr * (1 + 1e-9)   # just outside the band: selected
            c[f, band[1], k] = -thr * (1 - 1e-9)  # just inside: not selected
            c[f, band[2], k] = thr                # on the boundary: not selected (strict >)
            c[f, top[f, k], k] = M * np.sign(c[f, top[f, k], k])  # the max survives the band entries
    c[:, :, K:] = np.nan  # padding columns are never read
    if F > 1:
        c[1, :, K // 2] = 0.0  # an all-zero fit selects nothing
    c[0, p // 2, 0] = np.nan  # a NaN coefficient is not selected
    return c


@pytest.mark.parametrize("F,p,K,ldz", [(1, 45, 5, 8), (3, 301, 37, 40), (16, 97, 70, 104), (16, 33, 1, 8)])
def test_support_counts_match_numpy(engine, F, p, K, ldz):
    torch = engine.torch
    rng = np.random.default_rng(F * 1000 + p)
    t1, t2 = _table(rng, F, p, ldz, K), _table(rng, F, p, ldz, K)
    counts = torch.zeros((p, K), dtype=torch.int32, device=engine.device)
    u0 = (rng.random((F, p)) < 0.1).astype(np.uint8)  # OR-accumulated: set entries stay set
    union = engine.to_device(u0)
    for t in (t1, t2):  # two calls accumulate
        engine.support_counts(engine.to_device(t), K, TOL, counts, union)
    c1, s1 = _np_counts(t1, K, TOL)
    c2, s2 = _np_counts(t2, K, TOL)
    npt.assert_array_equal(counts.cpu().numpy(), c1 + c2)
    npt.assert_array_equal(union.cpu().numpy().astype(bool), (u0 > 0) | s1 | s2)
    # repeatable bit for bit
    counts2 = torch.zeros((p, K), dtype=torch.int32, device=engine.device)
    union2 = engine.to_device(u0)
    for t in (t1, t2):
        engine.support_counts(engine.to_device(t), K, TOL, counts2, union2)
    assert torch.equal(counts, counts2) and torch.equal(union, union2)


# ---- end to end ---------------------------------------------------------------------------------------------------
def _data(n, p, seed, intercept=0.0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    y = X[:, :6] @ [2.0, -1.5, 1.0, 0.8, -0.6, 0.5] + 0.5 * rng.standard_normal(n) + intercept
    return X, y, rng


def _alphas(X, y, fracs):
    yc = y - y.mean()
    return list(np.abs(X.T @ yc).max() / len(y) * np.asarray(fracs))


def _freqs(sel, fit_one, p):
    """Selection frequencies of fit_one(candidate, rows) -> coef over the subsamples of `sel`, and the smallest
    distance (as a factor) of a non-zero relative coefficient from the selection threshold."""
    freq = np.zeros((p, len(sel.candidates_)))
    margin = np.inf
    for ci, c in enumerate(sel.candidates_):
        for rows in sel.subsamples_:
            b = np.abs(np.asarray(fit_one(c, rows)))
            mx = b.max()
            if mx == 0:
                continue
            r = b[b > 0] / mx
            margin = min(margin, np.abs(np.log10(r / TOL)).min())
            freq[:, ci] += b > TOL * mx
    return freq / len(sel.subsamples_), margin


def _case(name):
    """(estimator, grid, X, y, sample_weight)"""
    if name == "lasso":
        X, y, _ = _data(121, 40, 0)
        return Lasso(solver_options=OPTS), {"alpha": _alphas(X, y, [0.5, 0.2, 0.08])}, X, y, None
    if name == "lasso_intercept_wide":  # p > 160: the tensor-core path
        X, y, _ = _data(501, 180, 1, intercept=3.0)
        return (Lasso(fit_intercept=True, solver_options=OPTS), {"alpha": _alphas(X, y, [0.4, 0.15])}, X, y, None)
    if name == "group":
        X, y, _ = _data(121, 40, 2)
        g = np.arange(40) // 4
        return GroupLasso(groups=g, solver_options=OPTS), {"alpha": _alphas(X, y, [0.5, 0.2])}, X, y, None
    if name == "sgl_weighted":
        X, y, rng = _data(121, 40, 3, intercept=-1.0)
        g = np.arange(40) % 8
        sw = 0.5 + rng.random(121)
        return (SparseGroupLasso(groups=g, l1_ratio=0.5, fit_intercept=True, solver_options=OPTS),
                {"alpha": _alphas(X, y, [0.5, 0.2])}, X, y, sw)
    if name == "sgl_wide":
        X, y, _ = _data(401, 200, 4)
        g = np.arange(200) // 10
        return (SparseGroupLasso(groups=g, l1_ratio=0.5, solver_options=OPTS), {"alpha": _alphas(X, y, [0.4, 0.15])},
                X, y, None)
    if name == "overlap":
        X, y, _ = _data(121, 30, 5)
        gl = [[j // 5, (j // 5 + 1) % 6] if j % 5 == 0 else [j // 5] for j in range(30)]
        return OverlapGroupLasso(group_list=gl, solver_options=OPTS), {"alpha": _alphas(X, y, [0.5, 0.2])}, X, y, None
    if name == "ridged":
        X, y, _ = _data(121, 40, 6, intercept=2.0)
        g = np.arange(40) // 4
        return (RidgedGroupLasso(groups=g, delta=(0.5,), fit_intercept=True, solver_options=OPTS),
                {"alpha": _alphas(X, y, [0.5, 0.2])}, X, y, None)
    if name == "adaptive":
        X, y, _ = _data(121, 40, 7)
        return AdaptiveLasso(solver_options=OPTS), {"alpha": _alphas(X, y, [0.3, 0.1])}, X, y, None
    if name == "sgl_standardized":  # the method-of-multipliers path, small
        X, y, _ = _data(61, 12, 8)
        g = np.arange(12) // 3
        return (SparseGroupLasso(groups=g, l1_ratio=0.5, standardize=True, solver_options={"tol": 1e-14}),
                {"alpha": _alphas(X, y, [0.5, 0.25])}, X, y, None)
    raise KeyError(name)


@pytest.mark.parametrize("name", ["lasso", "lasso_intercept_wide", "group", "sgl_weighted", "sgl_wide", "overlap",
                                  "ridged", "adaptive", "sgl_standardized"])
def test_scores_equal_sklearn_loop_of_engine_fits(name):
    est, grid, X, y, sw = _case(name)
    n, p = X.shape
    assert n % 2 == 1  # complementary halves of floor(n/2) and ceil(n/2) rows: direct and downdated builds
    sel = StabilitySelection(est, grid, n_subsamples=8, random_state=11).fit(X, y, sample_weight=sw)

    def fit_one(c, rows):
        kw = {} if sw is None else {"sample_weight": sw[rows]}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)
            return clone(est).set_params(**c).fit(X[rows], y[rows], **kw).coef_

    ref, margin = _freqs(sel, fit_one, p)
    assert margin > 1.0, f"a reference coefficient lies within a factor 10 of the threshold ({margin})"
    npt.assert_array_equal(sel.stability_scores_, ref)
    npt.assert_array_equal(sel.scores_, ref.max(axis=1))
    assert sel.stability_scores_.shape == (p, len(sel.candidates_))
    assert sel.solver_info_["status"].shape == (len(sel.candidates_), 8)


@pytest.mark.parametrize("name", ["Lasso", "SparseGroupLasso"])
def test_scores_equal_the_oracle(name):
    X, y, _ = _data(61, 20, 9)
    g = np.arange(20) // 4
    alphas = _alphas(X, y, [0.5, 0.2, 0.1])
    if name == "Lasso":
        est, kw = Lasso(solver_options=OPTS), {}
    else:
        est, kw = SparseGroupLasso(groups=g, l1_ratio=0.5, solver_options=OPTS), dict(groups=g, l1_ratio=0.5)
    sel = StabilitySelection(est, {"alpha": alphas}, n_subsamples=6, random_state=2).fit(X, y)
    ref, margin = _freqs(sel, lambda c, rows: R.fit(name, X[rows], y[rows], alpha=c["alpha"], **kw)[0], 20)
    assert margin > 1.0, margin
    npt.assert_array_equal(sel.stability_scores_, ref)


def test_known_answers():
    rng = np.random.default_rng(12)
    n, p = 200, 30
    X = rng.standard_normal((n, p))
    y = X[:, :3] @ [3.0, -2.5, 2.0] + 0.1 * rng.standard_normal(n)
    subs = draw_subsamples(n, 10, 0.5, True, random_state=5)
    amax = max(np.abs(X[r].T @ y[r]).max() / len(r) for r in subs)
    grid = {"alpha": [2.0 * amax, 0.05, 0.01]}
    sel = StabilitySelection(Lasso(solver_options=OPTS), grid, n_subsamples=10, threshold=0.9,
                             random_state=5).fit(X, y)
    assert all(np.array_equal(a, b) for a, b in zip(sel.subsamples_, subs))
    cols = {c["alpha"]: i for i, c in enumerate(sel.candidates_)}
    npt.assert_array_equal(sel.stability_scores_[:, cols[2.0 * amax]], 0.0)  # above every subsample's alpha_max
    npt.assert_array_equal(sel.stability_scores_[:3, cols[0.01]], 1.0)  # the planted features
    npt.assert_array_equal(sel.scores_[:3], 1.0)
    mask = sel.scores_ >= 0.9
    npt.assert_array_equal(sel.get_support(), mask)
    npt.assert_array_equal(sel.get_support(indices=True), np.flatnonzero(mask))
    npt.assert_array_equal(sel.transform(X), X[:, mask])
    assert sel.n_features_in_ == p
    q = sel.selected_size_
    assert 3 <= q <= p
    assert sel.expected_false_positives_ == pytest.approx(q * q / (0.8 * p), rel=1e-12)


def test_too_few_iterations_warn():
    X, y, _ = _data(121, 40, 13)
    est = Lasso(solver_options={"max_iter": 2, "tol": 1e-14})
    with pytest.warns(ConvergenceWarning):
        StabilitySelection(est, {"alpha": _alphas(X, y, [0.1, 0.01])}, n_subsamples=4, random_state=0).fit(X, y)

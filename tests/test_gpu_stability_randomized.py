"""Randomized stability selection and group-level frequencies on the GPU: slm_gram_scale and slm_group_support_counts
against numpy, StabilitySelection(weakness < 1) against the per-fit loop of engine fits on the rescaled designs, and
a randomized-Lasso known answer where the plain Lasso keeps a noise column."""

import warnings

import numpy as np
import numpy.testing as npt
import pytest
from sklearn.base import clone

pytestmark = pytest.mark.gpu

from sparselm_b200.model import (AdaptiveLasso, GroupLasso, Lasso, OverlapGroupLasso, RidgedGroupLasso,  # noqa: E402
                                 SparseGroupLasso)
from sparselm_b200.stability import StabilitySelection  # noqa: E402

TOL = 1e-6
OPTS = {"tol": 1e-13}


# ---- slm_gram_scale -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 7, 16])
@pytest.mark.parametrize("p", [5, 37, 301, 1100])
@pytest.mark.parametrize("kind", ["two_point", "arbitrary"])
def test_gram_scale_is_bitwise_numpy(engine, S, p, kind):
    rng = np.random.default_rng(S * 10000 + p)
    pa = engine.padded_cols(p)
    assert p % 8 and pa >= p + 2
    n_rows = 20
    if kind == "two_point":
        w = np.where(rng.random((n_rows, p)) < 0.5, 0.3, 1.0)
    else:
        w = np.exp(rng.uniform(-3.0, 3.0, (n_rows, p)))
    slots = rng.permutation(n_rows)[:S]
    A = rng.standard_normal((S, pa, pa))
    G0 = A + A.transpose(0, 2, 1)
    G = engine.to_device(G0)
    wd = engine.to_device(w)
    engine.gram_scale(G, p, wd, slots)
    out = G.cpu().numpy()
    for s in range(S):
        d = np.ones(pa)
        d[:p] = w[slots[s]]
        npt.assert_array_equal(out[s], G0[s] * np.outer(d, d))
    npt.assert_array_equal(out, out.transpose(0, 2, 1))  # exactly symmetric
    npt.assert_array_equal(out[:, p:, p:], G0[:, p:, p:])  # the y / ones rows and the padding keep their block
    npt.assert_array_equal(wd.cpu().numpy(), w)  # the weights table is read, not written


def test_gram_scale_rejects_a_slot_outside_the_table(engine):
    from sparselm_b200.engine import EngineError

    G = engine.to_device(np.zeros((2, 8, 8)))
    with pytest.raises(EngineError):
        engine.gram_scale(G, 5, engine.to_device(np.ones((3, 5))), [0, 3])


# ---- slm_group_support_counts -------------------------------------------------------------------------------------
def _table(rng, F, p, ldz, K):
    """Coefficient tables with planted exact zeros, values on and around the threshold, an all-zero fit, a NaN
    coefficient and NaN padding columns (as tests/test_gpu_stability.py)."""
    c = rng.uniform(-1.0, 1.0, (F, p, ldz))
    c[rng.random((F, p, ldz)) < 0.6] = 0.0
    c[rng.random((F, p, ldz)) < 0.7] *= TOL  # most entries below the threshold: whole groups go unselected
    top = rng.integers(0, p, (F, K))
    for f in range(F):
        for k in range(K):
            M = 8.0 * (1 + rng.random())
            band = rng.integers(0, p, 3)
            thr = TOL * M
            c[f, band[0], k] = thr * (1 + 1e-9)
            c[f, band[1], k] = -thr * (1 - 1e-9)
            c[f, band[2], k] = thr
            c[f, top[f, k], k] = M * rng.choice([-1.0, 1.0])
    c[:, :, K:] = np.nan
    if F > 1:
        c[1, :, K // 2] = 0.0
    c[0, p // 2, 0] = np.nan
    return c


def _np_feature_sel(coef, K, tol):
    a = np.abs(coef[:, :, :K])
    mx = np.where(np.isnan(a), 0.0, a).max(axis=1)
    with np.errstate(invalid="ignore"):
        return a > tol * mx[:, None, :]  # [F, p, K]


def _np_group_counts(coef, K, tol, gptr):
    sel = _np_feature_sel(coef, K, tol)
    gsel = np.stack([sel[:, gptr[g]:gptr[g + 1], :].any(axis=1) for g in range(len(gptr) - 1)], axis=1)  # [F, G, K]
    return gsel.sum(axis=0).astype(np.int32), gsel.any(axis=2)


def _gptr(sizes, p):
    sizes = list(sizes)
    assert sum(sizes) <= p
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)


_GROUP_CASES = {
    "size1_p45": (1, 45, 5, 8, [1] * 45),
    "size3_p301": (3, 301, 37, 40, [3] * 100 + [1]),
    "size33_p990": (16, 990, 70, 72, [33] * 30),
    "size300_p4000": (16, 4000, 104, 104, [300] * 13 + [100]),
    "mixed_p2000": (9, 2000, 1, 8, [1, 3, 33, 300, 1, 1, 300, 33, 3] * 2 + [2000 - 2 * 675]),
    "one_group_p1500": (4, 1500, 40, 40, [1500]),
}


@pytest.mark.parametrize("case", list(_GROUP_CASES))
def test_group_support_counts_match_numpy(engine, case):
    F, p, K, ldz, sizes = _GROUP_CASES[case]
    torch = engine.torch
    gptr = _gptr(sizes, p)
    G = len(gptr) - 1
    rng = np.random.default_rng(len(case) * 1000 + p)
    t1, t2 = _table(rng, F, p, ldz, K), _table(rng, F, p, ldz, K)
    gdev = engine.to_device(gptr)
    counts = torch.zeros((G, K), dtype=torch.int32, device=engine.device)
    u0 = (rng.random((F, G)) < 0.1).astype(np.uint8)
    union = engine.to_device(u0)
    for t in (t1, t2):  # two calls accumulate
        engine.group_support_counts(engine.to_device(t), K, TOL, gdev, counts, union)
    c1, s1 = _np_group_counts(t1, K, TOL, gptr)
    c2, s2 = _np_group_counts(t2, K, TOL, gptr)
    npt.assert_array_equal(counts.cpu().numpy(), c1 + c2)
    npt.assert_array_equal(union.cpu().numpy().astype(bool), (u0 > 0) | s1 | s2)
    assert 0 < (c1 + c2).sum() < 2 * F * G * K or G == 1  # some groups selected, some not
    # repeatable bit for bit
    counts2 = torch.zeros((G, K), dtype=torch.int32, device=engine.device)
    union2 = engine.to_device(u0)
    for t in (t1, t2):
        engine.group_support_counts(engine.to_device(t), K, TOL, gdev, counts2, union2)
    assert torch.equal(counts, counts2) and torch.equal(union, union2)


def test_group_counts_are_the_or_of_the_feature_predicates(engine):
    torch = engine.torch
    F, p, K, ldz = 16, 700, 45, 48
    rng = np.random.default_rng(5)
    gptr = _gptr([1, 3, 33, 300, 3, 1, 33, 300, 26], p)
    t = _table(rng, F, p, ldz, K)
    coef = engine.to_device(t)
    G = len(gptr) - 1
    counts = torch.zeros((G, K), dtype=torch.int32, device=engine.device)
    union = torch.zeros((F, G), dtype=torch.uint8, device=engine.device)
    engine.group_support_counts(coef, K, TOL, engine.to_device(gptr), counts, union)
    ref = np.zeros((G, K), dtype=np.int64)
    for f in range(F):  # the per-fit feature predicates of slm_support_counts: counts of one fit
        cf = torch.zeros((p, K), dtype=torch.int32, device=engine.device)
        uf = torch.zeros((1, p), dtype=torch.uint8, device=engine.device)
        engine.support_counts(coef[f:f + 1].contiguous(), K, TOL, cf, uf)
        sel = cf.cpu().numpy() > 0
        ref += np.stack([sel[gptr[g]:gptr[g + 1]].any(axis=0) for g in range(G)])
    npt.assert_array_equal(counts.cpu().numpy(), ref)


# ---- end to end ---------------------------------------------------------------------------------------------------
def _data(n, p, seed, intercept=0.0):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    y = X[:, :6] @ [2.0, -1.5, 1.0, 0.8, -0.6, 0.5] + 0.5 * rng.standard_normal(n) + intercept
    return X, y, rng


def _alphas(X, y, fracs):
    yc = y - y.mean()
    return list(np.abs(X.T @ yc).max() / len(y) * np.asarray(fracs))


def _case(name):
    """(estimator, grid, X, y, sample_weight, group labels or None): the cases of tests/test_gpu_stability.py"""
    if name == "lasso":
        X, y, _ = _data(121, 40, 0)
        return Lasso(solver_options=OPTS), {"alpha": _alphas(X, y, [0.5, 0.2, 0.08])}, X, y, None, None
    if name == "lasso_intercept_wide":
        X, y, _ = _data(501, 180, 1, intercept=3.0)
        return (Lasso(fit_intercept=True, solver_options=OPTS), {"alpha": _alphas(X, y, [0.4, 0.15])}, X, y, None,
                None)
    if name == "group":
        X, y, _ = _data(121, 40, 2)
        g = np.arange(40) // 4
        return GroupLasso(groups=g, solver_options=OPTS), {"alpha": _alphas(X, y, [0.5, 0.2])}, X, y, None, g
    if name == "sgl_weighted":
        X, y, rng = _data(121, 40, 3, intercept=-1.0)
        g = np.arange(40) % 8
        sw = 0.5 + rng.random(121)
        return (SparseGroupLasso(groups=g, l1_ratio=0.5, fit_intercept=True, solver_options=OPTS),
                {"alpha": _alphas(X, y, [0.5, 0.2])}, X, y, sw, g)
    if name == "sgl_wide":
        X, y, _ = _data(401, 200, 4)
        g = np.arange(200) // 10
        return (SparseGroupLasso(groups=g, l1_ratio=0.5, solver_options=OPTS), {"alpha": _alphas(X, y, [0.4, 0.15])},
                X, y, None, g)
    if name == "overlap":
        X, y, _ = _data(121, 30, 5)
        gl = [[j // 5, (j // 5 + 1) % 6] if j % 5 == 0 else [j // 5] for j in range(30)]
        return (OverlapGroupLasso(group_list=gl, solver_options=OPTS), {"alpha": _alphas(X, y, [0.5, 0.2])}, X, y,
                None, None)
    if name == "ridged":
        X, y, _ = _data(121, 40, 6, intercept=2.0)
        g = np.arange(40) // 4
        return (RidgedGroupLasso(groups=g, delta=(0.5,), fit_intercept=True, solver_options=OPTS),
                {"alpha": _alphas(X, y, [0.5, 0.2])}, X, y, None, g)
    if name == "adaptive":
        X, y, _ = _data(121, 40, 7)
        return AdaptiveLasso(solver_options=OPTS), {"alpha": _alphas(X, y, [0.3, 0.1])}, X, y, None, None
    if name == "sgl_standardized":
        X, y, _ = _data(61, 12, 8)
        g = np.arange(12) // 3
        return (SparseGroupLasso(groups=g, l1_ratio=0.5, standardize=True, solver_options={"tol": 1e-14}),
                {"alpha": _alphas(X, y, [0.5, 0.25])}, X, y, None, g)
    raise KeyError(name)


def _freqs(sel, fit_one, p, labels):
    """Feature and group selection frequencies of fit_one(candidate, s) -> coef over the subsamples of `sel`, and
    the smallest distance (as a factor) of a non-zero relative coefficient from the selection threshold."""
    ids = None if labels is None else np.unique(labels, return_inverse=True)[1]
    G = 0 if labels is None else ids.max() + 1
    freq = np.zeros((p, len(sel.candidates_)))
    gfreq = np.zeros((G, len(sel.candidates_)))
    margin = np.inf
    for ci, c in enumerate(sel.candidates_):
        for s in range(len(sel.subsamples_)):
            b = np.abs(np.asarray(fit_one(c, s)))
            mx = b.max()
            if mx == 0:
                continue
            r = b[b > 0] / mx
            margin = min(margin, np.abs(np.log10(r / TOL)).min())
            chosen = b > TOL * mx
            freq[:, ci] += chosen
            if labels is not None:
                gfreq[:, ci] += np.bincount(ids, weights=chosen, minlength=G) > 0
    n_sub = len(sel.subsamples_)
    return freq / n_sub, gfreq / n_sub, margin


_NAMES = ["lasso", "lasso_intercept_wide", "group", "sgl_weighted", "sgl_wide", "overlap", "ridged", "adaptive",
          "sgl_standardized"]


@pytest.mark.parametrize("name,weakness", [(n, 0.5) for n in _NAMES] + [("sgl_weighted", 0.2)])
def test_scores_equal_the_loop_of_engine_fits_on_rescaled_designs(name, weakness):
    est, grid, X, y, sw, labels = _case(name)
    n, p = X.shape
    assert n % 2 == 1  # complementary halves of floor(n/2) and ceil(n/2) rows: direct and downdated builds
    sel = StabilitySelection(est, grid, n_subsamples=8, weakness=weakness, random_state=11).fit(X, y,
                                                                                              sample_weight=sw)
    w = sel.weights_
    assert set(np.unique(w)) == {weakness, 1.0}

    def fit_one(c, s):
        rows = sel.subsamples_[s]
        kw = {} if sw is None else {"sample_weight": sw[rows]}
        with warnings.catch_warnings():
            warnings.simplefilter("ignore", UserWarning)
            return clone(est).set_params(**c).fit(X[rows] * w[s], y[rows], **kw).coef_

    ref, gref, margin = _freqs(sel, fit_one, p, labels)
    assert margin > 1.0, f"a reference coefficient lies within a factor 10 of the threshold ({margin})"
    npt.assert_array_equal(sel.stability_scores_, ref)
    npt.assert_array_equal(sel.scores_, ref.max(axis=1))
    if labels is None:
        assert sel.group_stability_scores_ is None and sel.group_labels_ is None
    else:
        npt.assert_array_equal(sel.group_labels_, np.unique(labels))
        npt.assert_array_equal(sel.group_stability_scores_, gref)
        npt.assert_array_equal(sel.group_scores_, gref.max(axis=1))
        assert 0.0 < sel.group_selected_size_ <= len(np.unique(labels))


def test_weakness_one_is_plain_stability_selection():
    est, grid, X, y, sw, labels = _case("sgl_weighted")
    a = StabilitySelection(est, grid, n_subsamples=8, random_state=11).fit(X, y, sample_weight=sw)
    b = StabilitySelection(est, grid, n_subsamples=8, weakness=1.0, random_state=11).fit(X, y, sample_weight=sw)
    npt.assert_array_equal(a.stability_scores_, b.stability_scores_)
    npt.assert_array_equal(a.group_stability_scores_, b.group_stability_scores_)
    npt.assert_array_equal(b.weights_, 1.0)


def test_randomized_lasso_drops_a_column_the_lasso_keeps():
    # x2 = 0.6 (x0 + x1) + noise violates the Lasso's irrepresentable condition (|Sigma_NS Sigma_SS^-1 sign| = 1.2):
    # the Lasso selects x2 on every subsample, the randomized Lasso keeps x0 and x1 and drops x2.  Seed, grid and
    # threshold checked against the CPU oracle (oracle.reference) on the same subsamples and weights: at weakness 0.2
    # the scores of x0, x1, x2 are 0.92, 0.94, 0.58; at weakness 1 they are all 1.
    rng = np.random.default_rng(0)
    n, p = 201, 8
    X = rng.standard_normal((n, p))
    X[:, 2] = 0.6 * (X[:, 0] + X[:, 1]) + 0.4 * rng.standard_normal(n)
    y = X[:, 0] + X[:, 1] + 0.5 * rng.standard_normal(n)
    amax = np.abs(X.T @ y).max() / n
    grid = {"alpha": list(amax * np.array([0.6, 0.4, 0.2, 0.1, 0.05]))}
    kw = dict(n_subsamples=50, threshold=0.75, random_state=0)
    plain = StabilitySelection(Lasso(solver_options=OPTS), grid, **kw).fit(X, y)
    rand = StabilitySelection(Lasso(solver_options=OPTS), grid, weakness=0.2, **kw).fit(X, y)
    assert all(np.array_equal(a, b) for a, b in zip(plain.subsamples_, rand.subsamples_))
    assert plain.get_support()[:3].all()  # the noise column x2 is selected
    assert rand.get_support()[:2].all() and not rand.get_support()[2]
    npt.assert_array_equal(plain.scores_[:3], 1.0)
    npt.assert_allclose(rand.scores_[:3], [0.92, 0.94, 0.58], atol=0.021)

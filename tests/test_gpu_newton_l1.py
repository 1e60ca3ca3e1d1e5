"""The l1 Newton step (slm_newton_step_l1, csrc/newton_kernels.cuh) column by column against the float64 reference
(tests/newton_l1_reference.py), and ``solver_options={"newton": "l1"}`` at estimator level: Lasso, AdaptiveLasso,
SparseGroupLasso and AdaptiveSparseGroupLasso on a strongly correlated design give the answers of the plain
iterations in at most half their iterations."""

import ctypes
import warnings

import numpy as np
import pytest

import newton_l1_reference as L1
import oracle.reference as R
import test_gpu_newton_kernels as NK

pytestmark = pytest.mark.gpu

from sparselm_b200.model import AdaptiveLasso, AdaptiveSparseGroupLasso, Lasso, SparseGroupLasso  # noqa: E402
from sparselm_b200.model_selection import GridSearchCV  # noqa: E402

EPS = np.finfo(np.float64).eps
SIZES = [0, 1, 2, 15, 16, 17, 63, 64, 65, 127, 128, 129, 191, 192, 193, 257, 500]


# ---- kernel level ---------------------------------------------------------------------------------------------
def run_step_l1(engine, case, X0w, W1w, work=None, fill=0.0):
    """One slm_newton_step_l1 (W1w None: NULL) on a copy of X0w [k][ldv]; returns (X, out [k][4], workspace)."""
    import torch

    p, F, k = case["p"], case["F"], X0w.shape[0]
    Gn = len(case["gptr"]) - 1
    nbytes = engine.lib.slm_newton_workspace(p, Gn, k, F)
    if work is None:
        work = torch.full(((nbytes + 7) // 8,), fill, dtype=torch.float64, device=engine.device)
    X = X0w.clone()
    out = torch.full((k, 4), fill, dtype=torch.float64, device=engine.device)
    fh = np.ascontiguousarray(case["fold"], dtype=np.int32)
    Gs, pa = case["Gs_dev"], case["Gs_dev"].shape[-1]
    engine._ck(engine.lib.slm_newton_step_l1(
        engine.h, engine._ptr(Gs), pa * pa, pa, p, F, k, fh.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
        engine._ptr(case["nobs_dev"]), engine._ptr(X), engine._ptr(case["w2_dev"]), engine._ptr(case["d2_dev"]),
        engine._ptr(W1w), engine._ptr(case["gptr_dev"]), engine._ptr(case["gid_dev"]), Gn, engine._ptr(work), nbytes,
        engine._ptr(out), engine.stream), "slm_newton_step_l1")
    torch.cuda.synchronize(engine.device)
    return X, out, work


def _l1_case(engine, seed, p, F, ms, sgl):
    """Columns with exactly ms[c] non-zero coordinates at random places (so SparseGroupLasso groups are active with
    zero coordinates in them), per-coordinate l1 weights, random folds and row counts."""
    import torch

    rng = np.random.default_rng(seed)
    sizes = (NK.MULTI + [1] * (p - sum(NK.MULTI))) if sgl else [p]
    gptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    Gn, k, n = len(sizes), len(ms), 3 * p
    X0 = np.zeros((k, p))
    for c, m in enumerate(rng.permutation(ms)):
        X0[c, rng.choice(p, m, replace=False)] = rng.standard_normal(m)
    w1 = 0.02 * (0.5 + rng.random((k, p)))
    w2 = 0.05 * (0.5 + rng.random((k, Gn))) if sgl else np.zeros((k, 1))
    case = dict(p=p, F=F, gptr=gptr, fold=rng.integers(0, F, k), nobs=n * (0.5 + rng.random(k)), X0=X0, w2=w2,
                d2=None, w1=w1, Gs_dev=NK._grams(engine, rng, p, F, n))
    NK._finish(engine, case)  # device copies (its pure group reference is not used here)
    ldv = NK._round_up(p, 8)
    W1w = np.zeros((k, ldv))
    W1w[:, :p] = w1
    case["W1w"] = torch.from_numpy(W1w).to(engine.device)
    case["l1ref"] = [L1.l1_step(case["Gs"][case["fold"][c]], p, case["nobs"][c], X0[c], w1[c], w2[c], None, gptr)
                     for c in range(k)]
    return case


def _check_l1_column(case, c, Xk, outk, views, x0w):
    ref = case["l1ref"][c]
    p = case["p"]
    G, n = case["Gs"][case["fold"][c]], case["nobs"][c]
    x0 = case["X0"][c]
    act, m = ref["act"], len(ref["act"])
    acc, t, dec, flag = outk
    assert np.isfinite(Xk[:p]).all() and np.isfinite(outk).all(), c
    assert ref["ok"] and flag == 0.0, c
    assert np.array_equal(act, np.flatnonzero(x0)), c                  # active = the non-zero coordinates
    if m:
        U = np.triu(views["H"][c, :m, :m])
        asm = 4 * EPS * (np.abs(np.diag(G)[act]) / n + ref["kk"][act]).max()
        err = np.abs(U.T @ U - ref["H"]).max()
        assert err <= NK.C_FACTOR * m * EPS * np.abs(ref["H"]).max() + asm, (c, m, err)
    d = views["DIR"][c, :p]
    assert np.all(d[x0 == 0] == 0.0), c
    assert np.abs(d - ref["d"]).max() <= 1e-8 * max(np.abs(ref["d"]).max(), 1e-300), c
    assert abs(dec - ref["dec"]) <= 1e-8 * abs(ref["dec"]) + 1e-300, (c, dec, ref["dec"])
    close = any(abs(dphi - thr) <= 1e-7 * size for (_, dphi, thr, size) in ref["trials"])
    if not close:
        assert bool(acc) == ref["accepted"], c
        assert t == pytest.approx(ref["t"], rel=1e-8, abs=0.0), (c, t, ref["t"])
    if acc:
        assert 0.0 < t <= min(1.0, ref["t_cross"] * (1 + 1e-8)), c
        if not close:
            assert np.all(Xk[ref["zeroed"]] == 0.0), c                 # exact zeros at the sign change
            assert np.array_equal(Xk[:p] == 0, ref["x_new"] == 0), c
            assert np.abs(Xk[:p] - ref["x_new"]).max() <= 1e-8 * np.abs(x0).max(), c
        assert L1.objective_change(G, p, n, x0, Xk[:p], case["w1"][c], case["w2"][c], None, case["gptr"]) < 0.0, c
    else:
        assert t == 0.0 and np.array_equal(NK._bits(Xk), NK._bits(x0w)), c
    assert np.array_equal(NK._bits(Xk[:p][x0 == 0]), NK._bits(x0w[:p][x0 == 0])), c   # the support never grows
    assert np.array_equal(NK._bits(Xk[p:]), NK._bits(x0w[p:])), c
    return not close, acc and len(ref["zeroed"]) > 0 and not close


_CASES = {}


def _case(engine, name):
    if name not in _CASES:
        rng = np.random.default_rng(11)
        if name == "sgl":     # m_max = 577 (odd), SparseGroupLasso groups, three Grams
            _CASES[name] = _l1_case(engine, 12, 640, 3, SIZES + [577] + list(rng.integers(65, 300, 20)), sgl=True)
        else:                 # Lasso: one zero-weight group of all coordinates, SLM_MAX_FOLDS Grams
            _CASES[name] = _l1_case(engine, 13, 700, NK.MAX_FOLDS, SIZES + [633] + list(rng.integers(65, 300, 20)),
                                    sgl=False)
    return _CASES[name]


@pytest.fixture()
def tma_mask(engine, request):
    engine.set_option("tma", request.param)
    yield request.param
    engine.set_option("tma", NK.ENGINE_TMA)


@pytest.mark.parametrize("tma_mask", [NK.DEFAULT_TMA, 0], indirect=True, ids=["tma", "cpasync"])
@pytest.mark.parametrize("name", ["sgl", "lasso"])
def test_newton_l1_step_matches_reference_across_panels(engine, tma_mask, name):
    case = _case(engine, name)
    p, k = case["p"], len(case["fold"])
    x0w = case["X0w"].cpu().numpy()
    X, out, work = run_step_l1(engine, case, case["X0w"], case["W1w"])
    Xh, outh = X.cpu().numpy(), out.cpu().numpy()
    m_max = max(len(r["act"]) for r in case["l1ref"])
    views = {kk: v.cpu().numpy() for kk, v in NK.workspace_views(work, p, k, m_max).items()}
    res = [_check_l1_column(case, c, Xh[c], outh[c], views, x0w[c]) for c in range(k)]
    assert sum(r[0] for r in res) >= k - 2
    assert sum(r[1] for r in res) >= 3                                  # steps truncated at a sign change
    # the same call again, and on a NaN-poisoned workspace: bitwise the same
    for fill in (0.0, float("nan")):
        X2, out2, _ = run_step_l1(engine, case, case["X0w"], case["W1w"], fill=fill)
        assert np.array_equal(NK._bits(X2.cpu().numpy()), NK._bits(Xh))
        assert np.array_equal(NK._bits(out2.cpu().numpy()), NK._bits(outh))


def test_newton_l1_entry_point_without_l1_weights_is_the_group_step(engine):
    """W1 = NULL: bitwise the result of slm_newton_step (pure group penalty, ridge, backtracking)."""
    case = NK._sized_case(engine, 8, 600, 2, [0, 17, 65, 130, 200, 257], ridge=True, backtrack=1)
    Xa, outa, _ = NK.run_step(engine, case, case["X0w"])
    Xb, outb, _ = run_step_l1(engine, case, case["X0w"], None)
    assert np.array_equal(NK._bits(Xa.cpu().numpy()), NK._bits(Xb.cpu().numpy()))
    assert np.array_equal(NK._bits(outa.cpu().numpy()), NK._bits(outb.cpu().numpy()))


# ---- estimator level ------------------------------------------------------------------------------------------
def _ar1_problem(seed=0, n=1200, p=300, rho=0.99, n_true=30):
    rng = np.random.default_rng(seed)
    X = np.empty((n, p))
    X[:, 0] = rng.standard_normal(n)
    for j in range(1, p):
        X[:, j] = rho * X[:, j - 1] + np.sqrt(1 - rho * rho) * rng.standard_normal(n)
    b = np.zeros(p)
    b[rng.choice(p, n_true, replace=False)] = rng.standard_normal(n_true) * 3.0
    y = X @ b + rng.standard_normal(n) + 2.0
    return X, y


GROUPS = np.repeat(np.arange(100), 3)


def _fit(cls, X, y, newton, **kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return cls(fit_intercept=True, solver_options={"tol": 1e-10, "max_iter": 200000, "newton": newton},
                   **kw).fit(X, y)


@pytest.mark.parametrize("cls", [Lasso, AdaptiveLasso, SparseGroupLasso, AdaptiveSparseGroupLasso])
def test_l1_newton_phase_matches_plain_iterations(cls):
    X, y = _ar1_problem()
    Xc, yc, _, _ = R.preprocess(X, y, None, True)
    amax = np.abs(Xc.T @ yc).max() / len(y)
    kw = dict(alpha=1e-2 * amax)
    if cls in (SparseGroupLasso, AdaptiveSparseGroupLasso):
        kw.update(groups=GROUPS, l1_ratio=0.5)
    a, b = _fit(cls, X, y, False, **kw), _fit(cls, X, y, "l1", **kw)
    assert a.solver_info_["status"] == 0 and b.solver_info_["status"] == 0
    s = np.abs(a.coef_).max()
    assert np.abs(a.coef_ - b.coef_).max() <= 1e-6 * s
    assert np.array_equal(np.abs(a.coef_) > 1e-6, np.abs(b.coef_) > 1e-6)
    assert abs(a.intercept_ - b.intercept_) <= 1e-6 * max(1.0, abs(a.intercept_))
    assert abs(a.solver_info_["objective"] - b.solver_info_["objective"]) <= 1e-8 * abs(a.solver_info_["objective"])
    assert 2 * b.solver_info_["iterations"] <= a.solver_info_["iterations"], (a.solver_info_, b.solver_info_)
    if cls in (Lasso, SparseGroupLasso):  # fixed weights: the oracle's certificate of the Newton path's answer
        p = X.shape[1]
        if cls is Lasso:
            pen = R.Penalty(np.arange(p), np.full(p, kw["alpha"]), np.zeros(p), np.zeros(p))
        else:
            pen = R.Penalty(GROUPS, np.full(p, 0.5 * kw["alpha"]), np.full(100, 0.5 * kw["alpha"]), np.zeros(100))
        cert = R.certificate(Xc, yc, b.coef_, pen)
        assert cert["gap"] <= 1e-8 * abs(cert["primal"]), cert


@pytest.mark.parametrize("cls", [Lasso, SparseGroupLasso])
def test_l1_newton_phase_in_a_cv_batch(cls, monkeypatch):
    """Five folds x five alphas: strongly penalised columns finish in the first stretch, weak ones go through
    the phase (its stats from the search's own batches, fewer iterations over all columns); per-split scores,
    best_params_ and the refit equal to the plain path."""
    import sparselm_b200.model_selection as MS

    searched = {}
    batched_cv = MS.batched_cv

    def spy(*a, **k):
        out = batched_cv(*a, **k)
        searched["newton"] = out.get("newton") or {}
        return out

    monkeypatch.setattr(MS, "batched_cv", spy)
    X, y = _ar1_problem(seed=1)
    Xc, yc, _, _ = R.preprocess(X, y, None, True)
    amax = np.abs(Xc.T @ yc).max() / len(y)
    alphas = list(amax * np.array([0.5, 0.1, 0.01, 3e-3, 1e-3]))
    kw = dict(groups=GROUPS, l1_ratio=0.5) if cls is SparseGroupLasso else {}
    out, stats = {}, {}
    for newton in (False, "l1"):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out[newton] = GridSearchCV(cls(fit_intercept=True, solver_options={
                "tol": 1e-10, "max_iter": 200000, "newton": newton}, **kw), {"alpha": alphas}, cv=5).fit(X, y)
        stats[newton] = searched.pop("newton")
    a, b = out[False], out["l1"]
    assert b.batched_ and not stats[False].get("phases")
    assert stats["l1"]["phases"] > 0 and stats["l1"]["factorizations"] > 0, stats["l1"]
    assert b.solver_info_["n_iter"].sum() < a.solver_info_["n_iter"].sum()
    for f in range(5):
        np.testing.assert_allclose(b.cv_results_[f"split{f}_test_score"], a.cv_results_[f"split{f}_test_score"],
                                   rtol=1e-6)
    assert a.best_params_ == b.best_params_
    assert np.abs(a.best_estimator_.coef_ - b.best_estimator_.coef_).max() <= 1e-6 * np.abs(a.best_estimator_.coef_).max()


def test_newton_true_is_still_a_no_op_with_an_l1_term_and_bogus_is_refused():
    X, y = _ar1_problem(seed=2, n=300, p=200)
    a = _fit(Lasso, X, y, True, alpha=0.05)
    b = _fit(Lasso, X, y, False, alpha=0.05)
    assert np.array_equal(a.coef_, b.coef_) and a.solver_info_["iterations"] == b.solver_info_["iterations"]
    with pytest.raises(ValueError, match="newton"):
        Lasso(alpha=0.05, solver_options={"newton": "bogus"}).fit(X, y)

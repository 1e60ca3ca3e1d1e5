"""The Newton phase inside the engine's batch (Engine._run_batch + newton.newton_phase): same
answers as the plain iterations on ill-conditioned overlap problems, in far fewer iterations."""

import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from sparselm_b200.model import AdaptiveOverlapGroupLasso, OverlapGroupLasso, SparseGroupLasso  # noqa: E402
from sparselm_b200.model_selection import GridSearchCV  # noqa: E402


def _overlap_problem(seed=0, n=400, p=240, G=24):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    w = np.zeros(p)
    w[rng.choice(p, p // 10, replace=False)] = 100.0 * rng.random(p // 10)
    y = X @ w + 10.0 * rng.standard_normal(n)
    base = rng.permutation(np.repeat(np.arange(G), p // G))
    extra = rng.random(p) < 0.3
    group_list = [[int(base[j])] + ([int((base[j] + 1 + rng.integers(G - 1)) % G)] if extra[j] else []) for j in range(p)]
    return X, y, group_list


@pytest.mark.parametrize("cls", [OverlapGroupLasso, AdaptiveOverlapGroupLasso])
def test_newton_phase_matches_plain_iterations_and_oracle(cls):
    X, y, group_list = _overlap_problem()
    alpha = 2e-3 * np.abs(X.T @ y).max() / len(y)        # weak penalty + duplicated columns: slow for first-order
    fits = {}
    for newton in (False, True):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            fits[newton] = cls(group_list=group_list, alpha=alpha, fit_intercept=True,
                               solver_options={"tol": 1e-11, "max_iter": 200000, "newton": newton}).fit(X, y)
    a, b = fits[False], fits[True]
    # the plain path (checked against the oracle throughout tests/test_gpu_estimators.py) is the reference here:
    # the block-coordinate-descent oracle needs minutes on this conditioning
    assert a.solver_info_["status"] == 0 and b.solver_info_["status"] == 0
    assert np.abs(a.coef_ - b.coef_).max() <= 1e-6 * np.abs(a.coef_).max()
    assert np.array_equal(np.abs(a.coef_) > 1e-6, np.abs(b.coef_) > 1e-6)
    assert abs(a.intercept_ - b.intercept_) <= 1e-6 * max(1.0, abs(a.intercept_))
    assert abs(a.solver_info_["objective"] - b.solver_info_["objective"]) <= 1e-8 * abs(a.solver_info_["objective"])
    assert b.solver_info_["iterations"] <= a.solver_info_["iterations"]


def test_newton_phase_in_a_cv_batch_with_frozen_and_finished_columns():
    """Five folds x four alphas: strongly penalised columns finish in the first stretch and are frozen,
    the weakly penalised ones go through the Newton phase; score table equal to the plain path."""
    X, y, group_list = _overlap_problem(seed=1)
    amax = np.abs(X.T @ y).max() / len(y)
    alphas = list(amax * np.array([0.3, 0.03, 3e-3, 1e-3]))
    out = {}
    for newton in (False, True):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out[newton] = GridSearchCV(AdaptiveOverlapGroupLasso(group_list=group_list, solver_options={
                "tol": 1e-10, "max_iter": 100000, "newton": newton}), {"alpha": alphas}, cv=5).fit(X, y)
    a, b = out[False], out[True]
    assert b.batched_
    for f in range(5):
        np.testing.assert_allclose(b.cv_results_[f"split{f}_test_score"], a.cv_results_[f"split{f}_test_score"], rtol=1e-6)
    assert a.best_params_ == b.best_params_
    assert np.abs(a.best_estimator_.coef_ - b.best_estimator_.coef_).max() <= 1e-6 * np.abs(a.best_estimator_.coef_).max()


def test_newton_option_is_ignored_when_the_penalty_has_an_l1_term():
    X, y, _ = _overlap_problem(seed=2)
    groups = np.repeat(np.arange(24), 10)
    kw = dict(groups=groups, alpha=0.05, l1_ratio=0.5)
    a = SparseGroupLasso(solver_options={"newton": True}, **kw).fit(X, y)
    b = SparseGroupLasso(solver_options={"newton": False}, **kw).fit(X, y)
    assert np.array_equal(a.coef_, b.coef_) and a.solver_info_["iterations"] == b.solver_info_["iterations"]


def test_newton_step_kernels_match_torch_model(engine):
    """slm_newton_step (Hessian assembly, blocked Cholesky, triangular solves, line search in
    csrc/newton_kernels.cuh) against the torch / library-Cholesky model of the same iteration:
    partly converged group-Lasso columns on two Grams, ridge on some, p not a multiple of the
    panel width."""
    import torch

    from sparselm_b200.newton import newton_phase, newton_phase_device

    rng = np.random.default_rng(4)
    n, p, Gn, F = 500, 203, 29, 2
    sizes = rng.multinomial(p - Gn, np.ones(Gn) / Gn) + 1
    gptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    gid = np.repeat(np.arange(Gn), sizes)
    pa = engine.padded_cols(p)
    Gs = torch.zeros((F, pa, pa), dtype=torch.float64, device=engine.device)
    for f in range(F):
        X = rng.standard_normal((n, p)) @ (np.eye(p) + 0.3 * rng.standard_normal((p, p)) / np.sqrt(p))
        w = np.zeros(p)
        for g in rng.choice(Gn, 6, replace=False):
            w[gptr[g]:gptr[g + 1]] = rng.standard_normal(sizes[g])
        y = X @ w + 0.3 * rng.standard_normal(n)
        Xa = np.hstack([X, y[:, None], np.ones((n, 1)), np.zeros((n, pa - p - 2))])
        Gs[f] = torch.from_numpy(Xa.T @ Xa).to(engine.device)
    K = 7
    fold = torch.from_numpy(rng.integers(0, F, K)).to(engine.device)
    nobs = torch.full((K,), float(n), dtype=torch.float64, device=engine.device)
    alphas = np.logspace(-1.0, -2.5, K)
    w2 = torch.from_numpy(alphas[:, None] * (0.5 + rng.random((K, Gn)))).to(engine.device)
    d2 = torch.from_numpy((rng.random((K, Gn)) < 0.3) * 0.2).to(engine.device)
    # start points: a few active groups per column, the rest exactly zero
    X0 = np.zeros((K, p))
    for c in range(K):
        for g in rng.choice(Gn, 8, replace=False):
            X0[c, gptr[g]:gptr[g + 1]] = rng.standard_normal(sizes[g])
    X0 = torch.from_numpy(X0).to(engine.device)
    scale = torch.ones(K, dtype=torch.float64, device=engine.device)
    gid64 = torch.from_numpy(gid.astype(np.int64)).to(engine.device)
    ref, iref = newton_phase(Gs, fold, nobs, X0, w2, d2, gid64, scale, 1e-10)
    out, iout = newton_phase_device(engine, Gs, fold, nobs, X0, w2, d2, torch.from_numpy(gptr).to(engine.device),
                                    gid64.to(torch.int32), scale, 1e-10)
    # the two differ by rounding only: same iterates; a decrement within rounding of the target may
    # flip the `finished` flag of at most one column
    assert (iref["finished"].cpu() == iout["finished"].cpu()).sum().item() >= K - 1
    assert iref["finished"].any() and iout["finished"].any()
    assert (out - ref).abs().max().item() <= 1e-7 * ref.abs().max().item()
    # inactive groups stay exactly zero
    assert torch.equal(out == 0, ref == 0)


def test_newton_kernels_and_torch_model_give_the_same_cv_search(monkeypatch):
    """One overlap CV batch at p_ext ~ 520, so that the Newton systems span several 64-wide panels, through the
    engine's kernels (SLM_NEWTON_TORCH=0) and through the torch / library-Cholesky model of the same iteration
    (=1): same status and score table, and the same amount of second-order work.  The duality-gap certificate
    would accept the points of a descending but wrong Newton direction; the work it takes to get there is
    where such a direction shows end to end."""
    from types import SimpleNamespace

    import torch
    from sklearn.model_selection import KFold

    from sparselm_b200.engine import get_engine
    from sparselm_b200.model_selection import batched_cv

    X, y, group_list = _overlap_problem(seed=3, n=600, p=400, G=40)
    amax = np.abs(X.T @ y).max() / len(y)
    est = AdaptiveOverlapGroupLasso(group_list=group_list, solver_options={"tol": 1e-10, "max_iter": 100000,
                                                                          "newton": True})
    p = X.shape[1]
    ests, specs = [], []
    for a in amax * np.array([0.03, 3e-3, 1e-3, 3e-4]):
        est.set_params(alpha=a)
        specs.append(est._problem_spec(p))
        ests.append(SimpleNamespace(fit_intercept=False))
    engine = get_engine(0)
    folds = [te for _, te in KFold(5).split(X)]
    Xd = torch.from_numpy(X).to(engine.device)
    res = {}
    for torch_model in ("0", "1"):
        monkeypatch.setenv("SLM_NEWTON_TORCH", torch_model)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            res[torch_model] = batched_cv(engine, Xd, y, folds, ests, specs, dict(est._engine_options()),
                                          "neg_root_mean_squared_error")
    a, b = res["0"], res["1"]
    assert len(specs[0].ext_idx) > 6 * 64
    assert max(int((a["warm"][ci] != 0).sum()) for ci in range(len(specs))) > 2 * 64  # multi-panel systems
    np.testing.assert_array_equal(a["info"]["status"], b["info"]["status"])
    assert (a["info"]["status"] == 0).all()
    np.testing.assert_allclose(a["test_scores"], b["test_scores"], rtol=1e-6)
    na, nb = a["newton"], b["newton"]
    counts = (na, nb, a["iters_run"], b["iters_run"])
    assert na["factorizations"] > 0 and abs(na["phases"] - nb["phases"]) <= 1, counts
    assert abs(na["factorizations"] - nb["factorizations"]) <= 0.05 * nb["factorizations"] + 2, counts
    assert abs(a["iters_run"] - b["iters_run"]) <= 0.05 * b["iters_run"] + 20, counts
    ia, ib = a["info"]["n_iter"].sum(), b["info"]["n_iter"].sum()
    assert abs(ia - ib) <= 0.05 * ib + 20, (ia, ib)

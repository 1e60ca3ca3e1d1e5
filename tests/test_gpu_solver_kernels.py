"""The proximal-iteration and duality-gap kernels (csrc/solver_kernels.cuh, coop_kernels.cuh) against float64
references (tests/solver_reference.py), kernel path by kernel path.

A. The certificate (gap_partial_kernel + gap_final_kernel, final mode) on given iterates: Engine.solve with
   max_iter = 0 only certifies B0.  Compared with the Gram-form model (bisection dual norm) and with the oracle's
   certificate from X and y.
B. The iterate after exactly m steps in every solver mode (small-design kernel, fused kernel in each register
   instantiation and its two-pass form, two-kernel iteration, cooperative and cluster kernels, compaction), with
   a tolerance no column can meet, against the same m steps of the model.
C. Groups left unpenalised (smooth groups) are certified: end-to-end fits converge with status 0."""

import warnings

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import engine_model as M  # noqa: E402
import oracle.reference as R  # noqa: E402
import solver_reference as S  # noqa: E402
from sparselm_b200.engine import PenaltyGrid, get_engine  # noqa: E402

# largest deviation of an m-step iterate from the float64 model, relative to max |B| of the case
ITER_RTOL = 1e-13  # observed on a B200: at most 7.5e-16


@pytest.fixture()
def switches():
    """fused_prox / coop as the test sets them, restored afterwards."""
    eng = get_engine()
    yield eng
    eng.set_option("fused_prox", 1)
    eng.set_option("coop", 1)


def _ldz(Ks):
    return max(8, -(-max(Ks) // 8) * 8)


def _stack(eng, arrs, Ks, rows):
    out = np.zeros((len(Ks), rows, _ldz(Ks)))
    for f, a in enumerate(arrs):
        out[f, :, : Ks[f]] = a
    return eng.to_device(out)


def _grid(p, gptr, lam1, W2, D2):
    if gptr is None:
        return PenaltyGrid(p=p, lam1=lam1)
    return PenaltyGrid(p=p, lam1=lam1, gptr=gptr, W2=W2, D2=D2)


def _solve(eng, G, p, n_obs, L, gptr, cols, tol, max_iter, per_row_w1=True):
    """Engine.solve on the columns cols[f] = (W1, W2, D2, B0) of every fold; W1 goes in as W1_init unless every
    row of a column carries the same weight and per_row_w1 is False."""
    Ks = [c[0].shape[1] for c in cols]
    p_ = cols[0][0].shape[0]
    grids = []
    for W1, W2, D2, _ in cols:
        lam1 = W1[0].copy() if not per_row_w1 else np.zeros(W1.shape[1])
        grids.append(_grid(p, gptr, lam1, None if gptr is None else W2, None if (gptr is None or not D2.any()) else D2))
    B0 = _stack(eng, [c[3] for c in cols], Ks, p_)
    W1 = _stack(eng, [c[0] for c in cols], Ks, p_) if per_row_w1 else None
    return eng.solve(G, p, n_obs, L, grids, B0=B0, tol=tol, max_iter=max_iter, newton=False, W1_init=W1)


# ================================================================================================================
# A. certificate on given iterates
# ================================================================================================================
def _cert_case(name):
    """(X, y, folds, gptr, cols per fold, penalised-from-X labels) of one certificate case.  Each column of a
    fold gets its own penalty and iterate: zero, sparse and dense iterates, omega < 1 and >> 1, the oracle's
    optimum."""
    cfg = {
        # name: (n, p, group sizes or None, K per fold, kind)
        "lasso_folds": (150, 120, None, [13, 8, 1], "lasso"),
        "lasso_many_rows": (400, 2100, None, [9], "lasso"),
        "sgl_sizes": (260, 260, [1, 3, 7, 8, 2, 10, 12, 13, 17, 20, 22, 31, 32, 45, 5, 4, 9, 6, 11, 2], [10, 3],
                      "sgl"),
        "group_sizes": (150, 110, [2, 5, 9, 14, 21, 33, 1, 6, 4, 15], [9], "group"),
        "ridged_sizes": (200, 240, [4, 8, 12, 16, 20, 24, 28, 32, 36, 40, 20], [8], "ridged"),
        "sgl_many_groups": (300, 1100, "many", [11], "sgl"),
        "smooth_groups": (200, 96, [8] * 12, [6], "smooth"),
    }[name]
    n, p, sizes, Ks, kind = cfg
    seed = sum(map(ord, name))
    X, y, rng = S.design(seed, n, p)
    if sizes is None:
        gptr = None
    elif sizes == "many":
        s = list(rng.integers(1, 4, size=p))
        s = s[: int(np.searchsorted(np.cumsum(s), p))]
        s.append(p - sum(s))
        gptr = S.gptr_of(s)
    else:
        gptr = S.gptr_of(sizes)
    assert gptr is None or gptr[-1] == p
    ge = np.arange(p + 1, dtype=np.int32) if gptr is None else gptr
    Gn = len(ge) - 1
    gw = np.sqrt(np.diff(ge)).astype(float)
    folds = None if len(Ks) == 1 else np.array_split(rng.permutation(n), len(Ks))
    amax = np.abs(X.T @ y).max() / n
    cols = []
    for f, K in enumerate(Ks):
        rows = np.arange(n) if folds is None else np.setdiff1d(np.arange(n), folds[f])
        Xf, yf = X[rows], y[rows]
        alphas = amax * np.geomspace(0.6, 0.02, K)
        W1 = np.zeros((p, K))
        W2 = np.zeros((Gn, K))
        D2 = np.zeros((Gn, K))
        if kind == "lasso":
            W1[:] = alphas * (0.5 + rng.random((p, 1)))
        elif kind in ("sgl", "ridged"):
            W1[:] = 0.4 * alphas * (0.5 + rng.random((p, 1)))
            W2[:] = gw[:, None] * (0.4 * alphas)[None, :]
            if kind == "ridged":
                D2[:] = 0.1 + rng.random((Gn, 1))
        elif kind == "group":
            W2[:] = gw[:, None] * alphas[None, :]
        if kind in ("sgl", "ridged", "group", "smooth") and Gn > 6:
            # rows without l1 weight inside groups with w2 > 0 (the infinite ratio bound of the Newton refinement),
            # and groups with w2 = 0 and w1 > 0 (closed-form ratio)
            W1[rng.random(p) < 0.2] = 0.0
            W1[ge[1]:ge[2]] = 0.3 * alphas
            W2[1] = 0.0
        if kind == "smooth":
            W1[:] = 0.0
            W2[:] = gw[:, None] * alphas[None, :]
            W2[[2, 7]] = 0.0  # two groups without any penalty
            if K > 3:
                D2[:, 3:] = 0.3
        B = np.zeros((p, K))
        lab = np.repeat(np.arange(Gn), np.diff(ge))
        for k in range(K):
            pen = R.Penalty(labels=lab, w1=W1[:, k], w2=W2[:, k], delta=D2[:, k])
            pick = k % 5
            if pick == 1:  # sparse
                B[:, k] = np.where(rng.random(p) < 0.1, rng.standard_normal(p), 0.0)
            elif pick == 2:  # dense, far from optimal (omega >> 1)
                B[:, k] = 0.3 * rng.standard_normal(p)
            elif pick == 3 and p <= 400:  # the oracle's optimum
                B[:, k] = R.solve(Xf, yf, pen, tol=1e-14)[0]
            elif pick == 4:  # a heavily penalised column at 0 (omega < 1, gap exactly 0)
                W1[:, k] *= 60.0
                W2[:, k] *= 60.0
        cols.append((W1, W2, D2, B))
    if kind == "smooth":  # every column at the oracle's optimum except the dense one
        for f, (W1, W2, D2, B) in enumerate(cols):
            for k in range(B.shape[1]):
                if k % 5 != 2:
                    pen = R.Penalty(labels=np.repeat(np.arange(Gn), np.diff(ge)), w1=W1[:, k], w2=W2[:, k],
                                    delta=D2[:, k])
                    B[:, k] = R.solve(X, y, pen, tol=1e-14)[0]
    return X, y, folds, gptr, cols


CERT_CASES = ["lasso_folds", "lasso_many_rows", "sgl_sizes", "group_sizes", "ridged_sizes", "sgl_many_groups",
              "smooth_groups"]


@pytest.mark.parametrize("name", CERT_CASES)
def test_certificate_matches_float64_references(name):
    eng = get_engine()
    X, y, folds, gptr, cols = _cert_case(name)
    n, p = X.shape
    tol = 1e-8
    fd = eng.prepare(X, y, test_folds=folds)
    F = len(cols)
    G = fd.G_full[None] if F == 1 else fd.G_train
    n_obs = [fd.n_obs("full")] if F == 1 else [fd.n_obs(f) for f in range(F)]
    L = [1.0] * F  # no iteration runs
    out = _solve(eng, G, p, n_obs, L, gptr, cols, tol=tol, max_iter=0)
    Gh = G.cpu().numpy()
    ge = np.arange(p + 1) if gptr is None else gptr
    lab = np.repeat(np.arange(len(ge) - 1), np.diff(ge))
    decided = 0
    for f, (W1, W2, D2, B) in enumerate(cols):
        K = B.shape[1]
        pb = S.problem_from_gram(Gh[f], p, n_obs[f], ge, W1, W2, D2)
        ref = S.certificate(pb, B, tol)
        P, gap, st = out["primal"][f, :K], out["gap"][f, :K], out["status"][f, :K]
        rows = np.arange(n) if folds is None else np.setdiff1d(np.arange(n), folds[f])
        gscale = np.maximum(np.abs(ref["primal"]), pb.yty / (2 * pb.n))
        assert np.all(out["n_iter"][f, :K] == 0)
        np.testing.assert_allclose(P, ref["primal"], rtol=1e-12, atol=0)
        assert np.all(np.abs(gap - ref["gap"]) <= 1e-12 * gscale), (name, f, gap - ref["gap"])
        # the oracle's certificate from X and y (its dual norm counts smooth rows: compare where there are none)
        for k in range(K):
            pen = R.Penalty(labels=lab, w1=W1[:, k], w2=W2[:, k], delta=D2[:, k])
            c = R.certificate(X[rows], y[rows], B[:, k], pen)
            assert abs(P[k] - c["primal"]) <= 1e-12 * abs(c["primal"]), (name, f, k)
            if not M.smooth_rows(pb)[:, k].any():
                assert abs(gap[k] - c["gap"]) <= 1e-12 * gscale[k], (name, f, k, gap[k], c["gap"])
        # a relative error of 1e-9 in omega moves the dual value by dD * 1e-9: where that exceeds the tolerance
        # above, the gap comparison checks the kernel's dual norm to better than 1e-9
        sens = ref["dD"] * 1e-9 > 2e-12 * gscale
        assert sens.sum() >= (1 if K < 4 else 2), (name, f, ref["dD"])
        # status: only where the reference is at least 2x away from the threshold
        clear = (ref["ratio"] <= 0.5) | (ref["ratio"] >= 2.0) | ~np.isfinite(ref["ratio"])
        clear &= ref["smooth_ok"] | (M.smooth_excess(pb, B, pb.G @ B) >= 2 * M.SMOOTH_KAPPA)
        assert np.array_equal(st[clear], ref["status"][clear]), (name, f, st, ref["status"], ref["ratio"])
        decided += int(clear.sum())
        assert {0, 1} <= set(ref["status"][clear].tolist()) or K < 4
    assert decided >= sum(c[3].shape[1] for c in cols) - 2


def test_certificate_unpenalised_and_nan_columns():
    """A column without any penalty is solved by conjugate gradients and frozen: the certificate kernels must
    leave its result alone.  A NaN in an iterate gives status 2 for that column only."""
    eng = get_engine()
    X, y, folds, gptr, cols = _cert_case("lasso_folds")
    n, p = X.shape
    fd = eng.prepare(X, y, test_folds=folds)
    F = len(cols)
    n_obs = [fd.n_obs(f) for f in range(F)]
    cols = [tuple(np.array(a) for a in c) for c in cols]
    for f in range(F):
        W1, _, _, B = cols[f]
        W1[:] = W1[0]  # one l1 weight per column: lam1 (the unpenalised column is recognised from lam1 = 0)
    cols[0][0][:, 4] = 0.0
    cols[0][3][:, 4] = 1.0
    cols[0][3][7, 5] = np.nan
    out = _solve(eng, fd.G_train, p, n_obs, [1.0] * F, None, cols, tol=1e-8, max_iter=0, per_row_w1=False)
    Gh = fd.G_train.cpu().numpy()
    Bd = out["B"].cpu().numpy()
    # the conjugate-gradient result (normal equations, iteration count, gap 0) is what comes back: the final
    # certificate would have written n_iter 0 and the column's gap
    c = Gh[0][p, :p]
    assert np.linalg.norm(Gh[0][:p, :p] @ Bd[0, :, 4] - c) <= 1e-8 * np.linalg.norm(c)
    assert out["n_iter"][0, 4] > 0 and out["gap"][0, 4] == 0.0
    assert out["status"][0, 5] == 2
    ok = [k for k in range(cols[0][3].shape[1]) if k not in (4, 5)]
    assert np.all(out["status"][0, ok] != 2) and np.all(out["status"][1:, :8] != 2)
    assert np.isfinite(out["gap"][0, ok]).all()


# ================================================================================================================
# B. m-step iterates in every solver mode
# ================================================================================================================
def _freeze(cols):
    """Columns f, f+2, ... of fold f (half of them at most) penalised 50x harder: beyond alpha_max at B0 = 0,
    their gap is exactly 0 at the check of iteration 0."""
    out, frozen = [], []
    for f, (W1, W2, D2, B0) in enumerate(cols):
        W1, W2, B0 = W1.copy(), W2.copy(), B0.copy()
        fz = np.arange(f, B0.shape[1], 2)[: max(1, B0.shape[1] // 2)]
        W1[:, fz] *= 50.0
        W2[:, fz] *= 50.0
        B0[:, fz] = 0.0
        out.append((W1, W2, D2, B0))
        frozen.append(fz)
    return out, frozen


def _iter_run(eng, name, mode, lips_device=False, freeze=False):
    X, y, gptr, Ks, m, cols, kind = S.iter_case(name)
    frozen = None
    if freeze:
        cols, frozen = _freeze(cols)
    n, p = X.shape
    F = len(Ks)
    folds = None if F == 1 else np.array_split(np.arange(n), F)
    fd = eng.prepare(X, y, test_folds=folds)
    G = fd.G_full[None] if F == 1 else fd.G_train
    keys = ["full"] if F == 1 else list(range(F))
    n_obs = [fd.n_obs(k) for k in keys]
    if lips_device:
        L = fd.lipschitz_dev(eng, keys, list(range(F)))
        Lh = L.cpu().numpy()
    else:
        Lh = np.array([fd.lipschitz(eng, k) for k in keys])
        L = list(Lh)
    eng.set_option("fused_prox", 0 if mode == "two_kernel" else 1)
    eng.set_option("coop", 1 if mode in ("coop", "cluster") else 0)
    l0 = eng.launch_count()
    out = _solve(eng, G, p, n_obs, L, None if kind == "lasso" else gptr, cols, tol=1e-14, max_iter=m,
                 per_row_w1=kind != "lasso")
    launches = eng.launch_count() - l0
    Gh = G.cpu().numpy()
    refs = []
    for f, (W1, W2, D2, B0) in enumerate(cols):
        pb = S.problem_from_gram(Gh[f], p, n_obs[f], gptr, W1, W2, D2, L=float(Lh[f]))
        Bm, mg = S.fused_iterates(pb, B0, m)
        S.assert_margins(mg, f"{name} fold {f}")
        refs.append((pb, Bm))
    return out, refs, m, launches, frozen


def _check_iterates(out, refs, m, frozen=None, name=""):
    """B after m steps against the model; n_iter = m, and the final certificate's status where the model's is
    clear of the threshold (a column can reach the tolerance in the last steps); frozen columns come back as
    B0 = 0 with n_iter 0, status 0 and gap 0."""
    Bd = out["B"].cpu().numpy()
    dev = 0.0
    for f, (pb, Bm) in enumerate(refs):
        K = Bm.shape[1]
        ks = np.arange(K)
        if frozen is not None:
            fz = frozen[f]
            assert np.all(out["n_iter"][f, fz] == 0) and np.all(out["status"][f, fz] == 0), (name, f)
            assert np.all(out["gap"][f, fz] == 0.0) and np.all(Bd[f][:, fz] == 0.0), (name, f)
            ks = np.setdiff1d(ks, fz)
        ref = S.certificate(pb, Bm, 1e-14)
        clear = ks[(ref["ratio"][ks] >= 2) | (ref["ratio"][ks] <= 0.5)]
        assert np.all(out["n_iter"][f, ks] == m), (name, f, out["n_iter"][f, :K])
        assert np.array_equal(out["status"][f, clear], ref["status"][clear]), (name, f, out["status"][f, :K])
        assert np.mean(ref["status"][ks] == 1) >= 0.5, (name, f)  # most columns are still running
        scale = np.abs(Bm[:, ks]).max()
        assert scale > 0
        dev = max(dev, np.abs(Bd[f][:, ks] - Bm[:, ks]).max() / scale)
    print(f"[iterates] {name}: max |B - B_ref| / max |B_ref| = {dev:.2e}")
    assert dev <= ITER_RTOL, (name, dev)
    return dev


# case -> the kernel it reaches: fista_small_kernel (p <= 160; nsplit = 2 at p = 100, 1 at p = 150),
# prox_fused_kernel<GROUPED, FZ_RC> chosen from the largest group (<= 8 rows: 2 rows per sub-lane, <= 12: 3,
# <= 20: 5, <= 32: 8, longer: 8 with the two-pass stash path), prox_main + prox_momentum (two-kernel)
@pytest.mark.parametrize("name,mode", [
    ("small_sgl_p100", "fused"), ("small_group_p150", "fused"), ("small_lasso_p150", "fused"),
    ("lasso_p240", "fused"), ("rc2_p240", "fused"), ("rc3_p240", "fused"), ("rc5_p240", "fused"),
    ("rc8_p240", "fused"), ("twopass_p240", "fused"),
    ("lasso_p240", "two_kernel"), ("rc3_p240", "two_kernel"), ("twopass_p240", "two_kernel"),
    ("rc5_p240", "two_kernel"),
])
def test_m_step_iterates_match_model(name, mode, switches):
    out, refs, m, _, _ = _iter_run(switches, name, mode)
    _check_iterates(out, refs, m, name=f"{name}/{mode}")


@pytest.mark.parametrize("name", ["few_lasso_p300", "few_sgl_p300", "many_sgl_p400"])
def test_m_step_iterates_cooperative_and_cluster(name, switches):
    """At most four columns: the cooperative kernel iterates between checks.  Twenty columns of which half
    converge at the first check (frozen beyond alpha_max): the ten left, with empty supports (cold start), are
    under the cluster threshold and the cluster kernel takes over.  Either way far fewer launches than the
    per-iteration kernels on the same problem, and the same iterates."""
    many = name.startswith("many")
    mode = "cluster" if many else "coop"
    out, refs, m, la, frozen = _iter_run(switches, name, mode, freeze=many)
    _check_iterates(out, refs, m, frozen=frozen, name=f"{name}/{mode}")
    _, _, _, lb, _ = _iter_run(switches, name, "fused", freeze=many)
    assert la < lb // 2, (la, lb)  # the cooperative / cluster path really ran


@pytest.mark.parametrize("mode", ["fused", "two_kernel"])
def test_m_step_iterates_after_compaction(mode, switches):
    """Folds of 13, 8 and 5 columns, several of them penalised beyond alpha_max from B0 = 0: they converge at the
    check of iteration 0 (gap exactly 0), leave the batch (compaction: scatter, renumbering, the restart dot
    carried over), come back as B0 with n_iter 0 -- and the other columns still walk the model's iterates.
    Lipschitz constants on the device."""
    out, refs, m, _, frozen = _iter_run(switches, "folds_sgl_p260", mode, lips_device=True, freeze=True)
    _check_iterates(out, refs, m, frozen=frozen, name=f"compaction/{mode}")


# ================================================================================================================
# C. groups left unpenalised
# ================================================================================================================
@pytest.mark.parametrize("p", [90, 300])
@pytest.mark.parametrize("fit_intercept", [False, True])
@pytest.mark.parametrize("est", ["GroupLasso", "SparseGroupLasso", "RidgedGroupLasso"])
def test_zero_weight_group_fits_converge(est, fit_intercept, p):
    """A group weight of 0 (no l1 weight either) leaves the group unpenalised: its dual constraint is
    X_g' theta = 0, met only to rounding.  The certificate tests those rows for stationarity instead of
    putting an infinite dual norm into the gap, so the fit converges early with status 0."""
    from sparselm_b200 import model

    cls = getattr(model, est)
    rng = np.random.default_rng(p + 2 * fit_intercept)
    n = 2 * p
    X = rng.standard_normal((n, p)) + (0.5 if fit_intercept else 0.0)
    w = np.zeros(p)
    w[rng.choice(p, p // 8, replace=False)] = 2 * rng.standard_normal(p // 8)
    y = X @ w + 0.5 * rng.standard_normal(n) + (1.0 if fit_intercept else 0.0)
    groups = np.repeat(np.arange(p // 6), 6)
    gw = 0.5 + rng.random(p // 6)
    gw[2] = 0.0
    kw = {"groups": groups, "group_weights": gw}
    if est == "SparseGroupLasso":
        kw["l1_ratio"] = 0.0
    if est == "RidgedGroupLasso":
        kw["delta"] = (0.3,)
    alpha = 0.1 * np.abs(X.T @ y).max() / n
    from sklearn.exceptions import ConvergenceWarning

    with warnings.catch_warnings():
        warnings.simplefilter("error", ConvergenceWarning)
        a = cls(alpha=alpha, fit_intercept=fit_intercept, **kw).fit(X, y)
    info = a.solver_info_
    assert info["status"] == 0 and info["iterations"] <= 2000, info
    b_ref, i_ref = R.fit(est, X, y, alpha=alpha, fit_intercept=fit_intercept, **kw)
    assert np.abs(a.coef_ - b_ref).max() <= 1e-6 * np.abs(b_ref).max()
    assert abs(a.intercept_ - i_ref) <= 1e-6 * max(1.0, abs(i_ref))
    Xc, yc = (X - X.mean(0), y - y.mean()) if fit_intercept else (X, y)
    labels, Gn = R.group_labels(groups, p)
    delta = np.full(Gn, 0.3) if est == "RidgedGroupLasso" else np.zeros(Gn)
    pen = R.Penalty(labels=labels, w1=np.zeros(p), w2=alpha * gw, delta=delta)
    assert abs(R.objective(Xc, yc, a.coef_, pen) - R.objective(Xc, yc, b_ref, pen)) <= 1e-8 * R.objective(Xc, yc, b_ref, pen)
    assert R.kkt_residual(Xc, yc, a.coef_, pen) <= 1e-9
    # how far from stationary the smooth rows of the fit are, in units of the kappa = 1 rounding bound
    gptr = np.arange(0, p + 1, 6)
    pb = S.problem_from_design(Xc, yc, gptr, np.zeros((p, 1)), (alpha * gw)[:, None], delta[:, None])
    print(f"[smooth] {est} p={p} intercept={fit_intercept}: iterations {info['iterations']}, "
          f"max |g_j| / tau_j(kappa=1) = {M.smooth_excess(pb, a.coef_[:, None], pb.G @ a.coef_[:, None])[0]:.3f}")

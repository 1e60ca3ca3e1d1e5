"""l1 step of the lock-step Newton phase (``newton_phase(..., w1=...)``, sparselm_b200/newton.py) on CPU tensors
against the float64 per-column reference (tests/newton_l1_reference.py): Lasso (one zero-weight group of all
coordinates), SparseGroupLasso and per-coordinate adaptive weights; a step truncated at a sign change; an
optimal column; the values the ``newton`` solver option accepts."""

import numpy as np
import pytest
import torch

import engine_model as M
import newton_l1_reference as L1
from sparselm_b200.newton import newton_phase


def _ar1_design(rng, n, p, rho):
    X = np.empty((n, p))
    X[:, 0] = rng.standard_normal(n)
    for j in range(1, p):
        X[:, j] = rho * X[:, j - 1] + np.sqrt(1 - rho * rho) * rng.standard_normal(n)
    return X


def _case(kind, seed=0, n=240, p=48, K=6):
    """Columns of one kind at partly converged proximal-gradient points (engine model, loose tolerance).
    Returns (Ga [1, pa, pa], n, gptr, X0 [K, p], w1 [K, p], w2 [K, Gn])."""
    rng = np.random.default_rng(seed)
    X = _ar1_design(rng, n, p, 0.9)
    b = np.zeros(p)
    b[rng.choice(p, 8, replace=False)] = rng.standard_normal(8) * 2.0
    y = X @ b + 0.3 * rng.standard_normal(n)
    pa = p + 2
    Ga = np.zeros((1, pa, pa))
    Ga[0, :p, :p] = X.T @ X
    Ga[0, p, :p] = Ga[0, :p, p] = X.T @ y
    Ga[0, p, p] = y @ y
    amax = np.abs(X.T @ y).max() / n
    alphas = amax * np.geomspace(0.3, 0.01, K)
    if kind == "sgl":
        gptr = np.arange(0, p + 1, 4)
        Gn = len(gptr) - 1
        W1 = np.tile(0.5 * alphas, (p, 1))
        W2 = np.tile(0.5 * alphas, (Gn, 1))
    else:
        gptr = np.array([0, p])  # Lasso: one group of every coordinate, zero weight
        W1 = np.tile(alphas, (p, 1))
        if kind == "adaptive":
            W1 *= 0.2 + 1.6 * rng.random((p, K))
        W2 = np.zeros((1, K))
    pb = M.BatchProblem(Ga[0, :p, :p], Ga[0, p, :p], Ga[0, p, p], n, gptr if kind == "sgl" else np.arange(p + 1),
                        W1, W2 if kind == "sgl" else np.zeros((p, K)), np.zeros((len(W2) if kind == "sgl" else p, K)))
    B, _ = M.solve(pb, tol=1e-3, max_iter=40)
    return Ga, n, gptr, B.T.copy(), W1.T.copy(), W2.T.copy()


def _model_step(Ga, n, gptr, X0, w1, w2):
    K, p = X0.shape
    gid = np.repeat(np.arange(len(gptr) - 1), np.diff(gptr))
    Xn, info = newton_phase(torch.from_numpy(Ga), torch.zeros(K, dtype=torch.int64), torch.full((K,), float(n)),
                            torch.from_numpy(X0), torch.from_numpy(w2), None, torch.from_numpy(gid),
                            torch.ones(K, dtype=torch.float64), 1e-10, max_steps=1, w1=torch.from_numpy(w1))
    return Xn.numpy(), info


def _close_call(ref, rel):
    return any(abs(dphi - thr) <= 8 * rel * size for (_, dphi, thr, size) in ref["trials"])


@pytest.mark.parametrize("kind", ["lasso", "sgl", "adaptive"])
def test_torch_model_l1_step_matches_reference(kind):
    Ga, n, gptr, X0, w1, w2 = _case(kind)
    K, p = X0.shape
    Xn, info = _model_step(Ga, n, gptr, X0, w1, w2)
    compared = 0
    for c in range(K):
        ref = L1.l1_step(Ga[0], p, n, X0[c], w1[c], w2[c], None, gptr)
        assert ref["ok"] and ref["dec"] > 0, c
        if _close_call(ref, 1e-9):
            continue
        compared += 1
        assert int(info["steps"][c]) == int(ref["accepted"]), c
        scale = np.abs(X0[c]).max()
        assert np.abs(Xn[c] - ref["x_new"]).max() <= 1e-9 * scale, (c, np.abs(Xn[c] - ref["x_new"]).max())
        assert np.array_equal(Xn[c] == 0, ref["x_new"] == 0), c       # same support after the step
        assert np.all(Xn[c][X0[c] == 0] == 0.0), c                     # the support never grows
        if ref["accepted"]:
            assert L1.objective_change(Ga[0], p, n, X0[c], Xn[c], w1[c], w2[c], None, gptr) < 0.0, c
    assert compared >= K - 1


def _crossing_case():
    """Orthogonal design (G = n I, n a power of two): the Newton direction lands on the unconstrained minimiser of
    the sign manifold, which for coordinate 1 lies on the other side of zero."""
    p, n = 4, 8.0
    bstar = np.array([1.5, 0.05, -0.75, 0.0])
    Ga = np.zeros((1, p + 2, p + 2))
    Ga[0, :p, :p] = n * np.eye(p)
    Ga[0, p, :p] = Ga[0, :p, p] = n * bstar
    Ga[0, p, p] = n * (bstar @ bstar) + 1.0
    lam = 0.25
    x0 = np.array([1.0, 0.1, -0.5, 0.0])
    return Ga, n, p, x0, lam


def test_step_truncated_at_a_sign_change():
    Ga, n, p, x0, lam = _crossing_case()
    gptr = np.array([0, p])
    w1 = np.full(p, lam)
    ref = L1.l1_step(Ga[0], p, n, x0, w1, np.zeros(1), None, gptr)
    # d_1 = -(x_1 - b*_1 + lam) = -0.3: coordinate 1 reaches zero at t = 0.1 / 0.3
    assert ref["t_cross"] == pytest.approx(1 / 3, rel=1e-15)
    assert ref["accepted"] and ref["t"] == ref["t_cross"]
    assert list(ref["zeroed"]) == [1] and ref["x_new"][1] == 0.0
    assert L1.objective_change(Ga[0], p, n, x0, ref["x_new"], w1, np.zeros(1), None, gptr) < 0.0
    Xn, info = _model_step(Ga, n, gptr, x0[None].copy(), w1[None].copy(), np.zeros((1, 1)))
    assert Xn[0, 1] == 0.0 and Xn[0, 3] == 0.0
    np.testing.assert_allclose(Xn[0], ref["x_new"], rtol=0, atol=1e-15)
    assert not bool(info["finished"][0])                               # a truncated step never finishes a column


def test_optimal_column_is_left_alone():
    Ga, n, p, _, lam = _crossing_case()
    gptr = np.array([0, p])
    w1 = np.full(p, lam)
    xopt = np.array([1.25, 0.0, -0.5, 0.0])                           # soft(b*, lam): the gradient is exactly zero
    ref = L1.l1_step(Ga[0], p, n, xopt, w1, np.zeros(1), None, gptr)
    assert ref["dec"] == 0.0 and not ref["accepted"]
    Xn, info = _model_step(Ga, n, gptr, xopt[None].copy(), w1[None].copy(), np.zeros((1, 1)))
    assert np.array_equal(Xn[0], xopt) and int(info["steps"][0]) == 0


@pytest.mark.parametrize("value,ok", [(None, True), (True, True), (False, True), ("l1", True), ("bogus", False),
                                      (1, False), ("L1", False)])
def test_newton_solver_option_values(value, ok):
    from sparselm_b200.model import Lasso

    est = Lasso(alpha=0.1, solver_options={"newton": value, "tol": 1e-9})
    if ok:
        assert est._engine_options()["newton"] is value
    else:
        with pytest.raises(ValueError, match="newton"):
            est._engine_options()

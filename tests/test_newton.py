"""Lock-step Newton phase (sparselm_b200/newton.py) on CPU tensors: from a partly converged
proximal-gradient point it must land on the oracle's solution, never increase the objective, and
leave columns alone whose start point is already optimal."""

import numpy as np
import pytest
import torch

import engine_model as M
import oracle.reference as R
from sparselm_b200.newton import newton_phase


def _problem(seed, n=80, p=30, G=6, ridge=False):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    groups = np.repeat(np.arange(G), p // G)
    w = np.zeros(p)
    w[: 2 * (p // G)] = rng.standard_normal(2 * (p // G)) * 2.0
    y = X @ w + 0.2 * rng.standard_normal(n)
    pa = p + 2
    Ga = np.zeros((1, pa, pa))
    Ga[0, :p, :p] = X.T @ X
    Ga[0, p, :p] = Ga[0, :p, p] = X.T @ y
    Ga[0, p, p] = y @ y
    return X, y, groups, Ga, (0.5 + rng.random(G) if ridge else None)


def _objective(X, y, b, groups, w2, d2):
    nr = np.array([np.linalg.norm(b[groups == g]) for g in np.unique(groups)])
    return np.sum((y - X @ b) ** 2) / (2 * len(y)) + (w2 * nr).sum() + (0.0 if d2 is None else 0.5 * (d2 * nr * nr).sum())


@pytest.mark.parametrize("ridge", [False, True])
def test_newton_phase_finishes_partly_converged_columns(ridge):
    X, y, groups, Ga, d2 = _problem(3, ridge=ridge)
    n, p = X.shape
    G = 6
    alphas = np.array([0.4, 0.1, 0.02])
    K = len(alphas)
    W2 = np.tile(alphas, (G, 1))
    D2 = np.zeros((G, K)) if d2 is None else np.tile(d2[:, None], (1, K))
    gptr = np.arange(0, p + 1, p // G)
    pb = M.BatchProblem(Ga[0, :p, :p], Ga[0, p, :p], Ga[0, p, p], n, gptr, np.zeros((p, K)), W2, D2)
    B, _ = M.solve(pb, tol=1e-3, max_iter=60)                      # support found, far from 1e-10
    P0, _, g0 = M.gap_terms(pb, B, pb.G @ B)
    Xn, info = newton_phase(torch.from_numpy(Ga), torch.zeros(K, dtype=torch.int64), torch.full((K,), float(n)),
                            torch.from_numpy(B.T.copy()), torch.from_numpy(W2.T.copy()),
                            None if d2 is None else torch.from_numpy(D2.T.copy()),
                            torch.from_numpy(np.repeat(np.arange(G), p // G)), torch.from_numpy(np.abs(P0)), 1e-10)
    Bn = Xn.numpy().T
    assert bool(info["finished"].all())
    P, _, g = M.gap_terms(pb, Bn, pb.G @ Bn)
    assert np.all(g <= 1e-10 * np.abs(P))
    for k, a in enumerate(alphas):
        kw = {"delta": tuple(d2)} if ridge else {}
        b_ref, _ = R.fit("RidgedGroupLasso" if ridge else "GroupLasso", X, y, alpha=a, groups=groups, **kw)
        assert np.abs(Bn[:, k] - b_ref).max() <= 1e-8 * np.abs(b_ref).max()
        assert np.array_equal(Bn[:, k] != 0, B[:, k] != 0)            # the phase never changes the support
        assert _objective(X, y, Bn[:, k], groups, W2[:, k], None if d2 is None else D2[:, k]) <= \
            _objective(X, y, B[:, k], groups, W2[:, k], None if d2 is None else D2[:, k]) + 1e-14


def test_newton_phase_leaves_zero_and_optimal_columns_alone():
    X, y, groups, Ga, _ = _problem(5)
    n, p = X.shape
    G = 6
    gid = torch.from_numpy(np.repeat(np.arange(G), p // G))
    b_ref, _ = R.fit("GroupLasso", X, y, alpha=0.1, groups=groups)
    start = np.stack([np.zeros(p), b_ref])                           # an all-zero column and an optimal one
    W2 = np.stack([np.full(G, 50.0), np.full(G, 0.1)])
    Xn, info = newton_phase(torch.from_numpy(Ga), torch.zeros(2, dtype=torch.int64), torch.full((2,), float(n)),
                            torch.from_numpy(start), torch.from_numpy(W2), None, gid, torch.ones(2), 1e-10)
    out = Xn.numpy()
    assert np.all(out[0] == 0.0)
    assert np.abs(out[1] - b_ref).max() <= 1e-9 * np.abs(b_ref).max()
    assert int(info["steps"][0]) == 0


def test_newton_phase_columns_on_different_grams():
    """Two folds with their own Gram and row count, columns mixed (fold index per column)."""
    Xa, ya, groups, Ga, _ = _problem(7, n=80)
    Xb, yb, _, Gb, _ = _problem(8, n=60)
    p, G = Xa.shape[1], 6
    Gs = torch.from_numpy(np.concatenate([Ga, Gb]))
    gid = torch.from_numpy(np.repeat(np.arange(G), p // G))
    fold = torch.tensor([1, 0, 1])
    alphas = [0.05, 0.2, 0.3]
    data = {0: (Xa, ya), 1: (Xb, yb)}
    refs = [R.fit("GroupLasso", *data[int(f)], alpha=a, groups=groups)[0] for f, a in zip(fold, alphas)]
    rng = np.random.default_rng(0)
    start = np.stack([r * (1.0 + 0.05 * rng.standard_normal(p)) for r in refs])   # same support, perturbed values
    W2 = np.stack([np.full(G, a) for a in alphas])
    n_obs = torch.tensor([60.0, 80.0, 60.0])
    Xn, info = newton_phase(Gs, fold, n_obs, torch.from_numpy(start), torch.from_numpy(W2), None, gid,
                            torch.ones(3), 1e-10, chol_batched=False)
    for k in range(3):
        assert np.abs(Xn[k].numpy() - refs[k]).max() <= 1e-8 * np.abs(refs[k]).max()


def _step_problem(seed, p=150, F=2, K=9):
    """Groups of 1..12 features (a run of singletons included), two Grams, per-column n, ridge on some
    columns, start points with a few active groups per column (a far, heavily weighted one among them)."""
    rng = np.random.default_rng(seed)
    sizes = list(rng.integers(2, 13, 14)) + [1] * 20
    sizes.append(p - sum(sizes))
    gptr = np.concatenate([[0], np.cumsum(sizes)])
    Gn = len(sizes)
    Gs = np.zeros((F, p + 2, p + 2))
    for f in range(F):
        n = 3 * p
        X = rng.standard_normal((n, p))
        y = X @ (rng.standard_normal(p) * (rng.random(p) < 0.2)) + 0.3 * rng.standard_normal(n)
        Xa = np.hstack([X, y[:, None], np.ones((n, 1))])
        Gs[f] = Xa.T @ Xa
    fold = rng.integers(0, F, K)
    n_obs = 3 * p * (0.5 + rng.random(K))
    w2 = 0.05 * (0.5 + rng.random((K, Gn)))
    d2 = (rng.random((K, Gn)) < 0.3) * 0.2
    X0 = np.zeros((K, p))
    for c in range(K):
        for g in rng.choice(Gn, 10, replace=False):
            X0[c, gptr[g]:gptr[g + 1]] = rng.standard_normal(sizes[g])
    X0[0] *= 1e-3                                                    # far from the optimum, strong penalty:
    w2[0] *= 40.0                                                    # the line search has to backtrack
    return Gs, gptr, fold, n_obs, X0, w2, d2


@pytest.mark.parametrize("ridge", [False, True])
def test_newton_reference_matches_newton_phase_after_one_step(ridge):
    """tests/newton_reference.py (float64 numpy / scipy, the kernels' line-search formulas) against the torch
    model of the phase after one step: same accept decisions, same points up to rounding."""
    import newton_reference as NR

    Gs, gptr, fold, n_obs, X0, w2, d2 = _step_problem(11)
    d2 = d2 if ridge else None
    K, p = X0.shape
    gid = torch.from_numpy(NR.group_ids(gptr))
    Xn, info = newton_phase(torch.from_numpy(Gs), torch.from_numpy(fold), torch.from_numpy(n_obs), torch.from_numpy(X0),
                            torch.from_numpy(w2), None if d2 is None else torch.from_numpy(d2), gid, torch.ones(K),
                            1e-10, max_steps=1)
    Xn = Xn.numpy()
    ts = []
    for c in range(K):
        ref = NR.newton_step(Gs[fold[c]], p, n_obs[c], X0[c], w2[c], None if d2 is None else d2[c], gptr)
        assert ref["ok"] and ref["accepted"] == bool(info["steps"][c] == 1)
        assert np.abs(Xn[c] - ref["x_new"]).max() <= 1e-10 * np.abs(X0[c]).max()
        assert np.array_equal(Xn[c] != 0, X0[c] != 0)
        ts.append(ref["t"])
        if ref["accepted"]:
            assert NR.objective_change(Gs[fold[c]], p, n_obs[c], X0[c], ref["x_new"], w2[c],
                                       None if d2 is None else d2[c], gptr) <= NR.ARMIJO / 2 * ref["t"] * -ref["dec"]
    assert min(ts) < 1.0 and max(ts) == 1.0                           # a backtracked and a full step among them

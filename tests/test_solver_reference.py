"""CPU checks of the float64 references of tests/test_gpu_solver_kernels.py (tests/solver_reference.py): the
model's dual norm (bisection) agrees with the oracle's (C, from X and y), the m-step reference runs stay clear of
the switch points of the iteration at the seeds the GPU test uses, and the model certifies groups left
unpenalised at the oracle's optimum."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import engine_model as M  # noqa: E402
import oracle.reference as R  # noqa: E402
import solver_reference as S  # noqa: E402


def _penalty(pb, k):
    return R.Penalty(labels=pb.gid, w1=pb.W1[:, k], w2=pb.W2[:, k], delta=pb.D2[:, k])


@pytest.mark.parametrize("kind", ["lasso", "sgl", "group", "ridged", "zero_w1_rows"])
def test_model_dual_norm_matches_oracle(kind):
    X, y, rng = S.design(11 + len(kind), 150, 110)
    n, p = X.shape
    gptr = S.gptr_of([2, 5, 9, 14, 21, 33, 1, 6, 4, 15]) if kind != "lasso" else np.arange(p + 1)
    Gn = len(gptr) - 1
    K = 6
    amax = np.abs(X.T @ y).max() / n
    alphas = amax * np.geomspace(0.6, 0.02, K)
    W1 = np.zeros((p, K))
    W2 = np.zeros((Gn, K))
    D2 = np.zeros((Gn, K))
    if kind == "lasso":
        W1[:] = alphas * (0.5 + rng.random((p, 1)))
    else:
        W2[:] = np.sqrt(np.diff(gptr))[:, None] * (0.5 * alphas)[None, :]
        if kind != "group":
            W1[:] = 0.5 * alphas
        if kind == "ridged":
            D2[:] = 0.1 + rng.random((Gn, 1))
        if kind == "zero_w1_rows":
            W1[:] = 0.5 * alphas
            W1[rng.random(p) < 0.3] = 0.0
            W2[3] = 0.0  # w2 = 0, w1 > 0: the closed-form ratio
            W1[gptr[3]:gptr[4]] = 0.5 * alphas
    pb = S.problem_from_design(X, y, gptr, W1, W2, D2)
    B = np.zeros((p, K))
    B[:, 1] = np.where(rng.random(p) < 0.1, rng.standard_normal(p), 0.0)
    B[:, 2] = 0.3 * rng.standard_normal(p)
    B[:, 3] = R.solve(X, y, _penalty(pb, 3), tol=1e-14)[0]
    B[:, 4] = 1e-3 * rng.standard_normal(p)
    ref = S.certificate(pb, B, 1e-8)
    for k in range(K):
        c = R.certificate(X, y, B[:, k], _penalty(pb, k))
        assert abs(ref["omega"][k] - c["omega"]) <= 1e-12 * c["omega"], (k, ref["omega"][k], c["omega"])
        assert abs(ref["primal"][k] - c["primal"]) <= 1e-12 * abs(c["primal"])
        assert abs(ref["gap"][k] - c["gap"]) <= 1e-12 * max(abs(c["primal"]), y @ y / (2 * n))
    assert ref["status"][3] == 0 and ref["omega"][2] > 1


@pytest.mark.parametrize("name", sorted(S.ITER_CASES))
def test_reference_runs_keep_clear_of_switch_points(name):
    X, y, gptr, Ks, m, cols, kind = S.iter_case(name)
    for f, (W1, W2, D2, B0) in enumerate(cols):
        pb = S.problem_from_design(X, y, gptr, W1, W2, D2)
        Bm, mg = S.fused_iterates(pb, B0, m)
        S.assert_margins(mg, name)
        # the two-kernel model (engine_model.solve) walks through the same iterates; nothing converges in m steps
        Ba, info = M.solve(pb, tol=1e-14, max_iter=m, B0=B0)
        assert not info["done"].any()
        assert np.abs(Ba - Bm).max() <= 1e-12 * np.abs(Bm).max()


def test_model_certifies_unpenalised_groups_at_the_optimum():
    """A group with w2 = 0 and no l1 weight: its dual constraint is g = 0, met only to rounding.  The model's
    certificate leaves it out of the dual norm and tests stationarity to rounding instead (status 0 at the
    oracle's optimum, status 1 away from it)."""
    X, y, rng = S.design(5, 200, 96)
    gptr = S.gptr_of([8] * 12)
    K = 3
    alphas = 0.1 * np.abs(X.T @ y).max() / 200 * np.array([1.0, 0.5, 0.25])
    W2 = np.sqrt(8.0) * np.tile(alphas, (12, 1))
    W2[[2, 7]] = 0.0
    D2 = np.zeros((12, K))
    D2[:, 2] = 0.3
    pb = S.problem_from_design(X, y, gptr, np.zeros((96, K)), W2, D2)
    B = np.stack([R.solve(X, y, _penalty(pb, k), tol=1e-15)[0] for k in range(K)], 1)
    ref = S.certificate(pb, B, 1e-10)
    assert (ref["status"] == 0).all() and np.isfinite(ref["omega"]).all()
    assert (M.smooth_excess(pb, B, pb.G @ B) <= 8).all()
    Bp = B.copy()
    Bp[gptr[2]] += 1e-6
    assert (S.certificate(pb, Bp, 1e-10)["status"] == 1).all()
    # and the iteration of the model converges on it
    Bm, info = M.solve(pb, tol=1e-10)
    assert info["done"].all() and info["iters"].max() < 2000
    assert np.abs(Bm - B).max() <= 1e-6 * np.abs(B).max()

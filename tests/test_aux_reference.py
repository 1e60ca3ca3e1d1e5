"""CPU checks of the float64 references of tests/test_gpu_aux_kernels.py (tests/aux_reference.py): the emulated block
power iteration is a tight lower bound of lambda_max on the Gaussian designs of
test_gpu_engine.py::test_lipschitz_is_tight_lower_bound and falls below lambda_max / 1.10 on the spike-over-flat-bulk
design of the convergence test; the ordered-sum references keep their order."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import aux_reference as A  # noqa: E402

ITERS, MARGIN = 12, 1.10  # Engine.LIPSCHITZ_ITERS, Engine.LIPSCHITZ_MARGIN


def test_start_vectors_are_the_kernels_hash():
    """Spot values of the 32-bit hash, computed step by step with Python integers."""
    def one(j, c, f):
        h = ((j * 8 + c) * 2654435761 + 12345 * (f + 1)) & 0xFFFFFFFF
        h ^= h >> 15
        h = (h * 2246822519) & 0xFFFFFFFF
        h ^= h >> 13
        return (h & 0xFFFFFF) / 8388608.0 - 1.0

    V = A.power_start(700, 5)
    for j, c in [(0, 0), (1, 7), (123, 3), (699, 7)]:
        assert V[j, c] == one(j, c, 5)
    assert not np.array_equal(A.power_start(50, 0), A.power_start(50, 1))
    assert (np.abs(V) <= 1.0).all()


@pytest.mark.parametrize("n,p", [(400, 100), (3000, 700), (60, 60), (6000, 1500), (500, 1000)])
def test_emulation_is_tight_on_gaussian_designs(n, p):
    rng = np.random.default_rng(3)
    X = rng.standard_normal((n, p))
    G = X.T @ X
    lam = A.power_lambda(G, ITERS)
    top = np.linalg.eigvalsh(G)[-1]
    assert lam <= top * (1 + 1e-12)
    assert lam * MARGIN >= top * 1.01, (lam / top)


def test_emulation_underestimates_spike_over_flat_bulk():
    """The design of test_gpu_aux_kernels.py::test_lasso_converges_with_underestimated_lipschitz: the margin does
    not cover lambda_max (Rayleigh quotient about 0.84 lambda_max)."""
    X = A.spike_over_bulk(1000, 1200, 1000, 0.8)
    G = X.T @ X
    ev = np.linalg.eigvalsh(G)
    np.testing.assert_allclose(ev[[0, -2, -1]], [0.8 * 1200, 0.8 * 1200, 1200], rtol=1e-10)
    lam = A.power_lambda(G, ITERS)
    assert lam * MARGIN < ev[-1]
    assert lam <= ev[-1]


def test_power_lambda_edge_spectra():
    assert A.power_lambda(np.zeros((9, 9)), ITERS) == 0.0
    v = np.arange(1.0, 8.0)
    np.testing.assert_allclose(A.power_lambda(np.outer(v, v), ITERS), v @ v, rtol=1e-14)
    assert A.power_lambda(np.array([[3.5]]), ITERS) == 3.5


def test_ordered_sums_keep_their_order():
    """On mixed magnitudes a pairwise or reversed sum gives other bits; the references add 0.0 + G_0 + G_1 + ..."""
    rng = np.random.default_rng(0)
    blocks = A.mixed_magnitudes(rng, (16, 30, 30))
    tot = A.ordered_total(blocks)
    rev = np.zeros_like(tot)
    for b in blocks[::-1]:
        rev = rev + b
    assert not np.array_equal(tot, rev)
    comp = A.ordered_complements(list(blocks))
    acc = np.zeros_like(tot)
    for b in blocks[1:]:
        acc = acc + b
    assert np.array_equal(comp[0], acc)
    assert np.array_equal(A.ordered_complements([blocks[0]])[0], np.zeros_like(tot))
    Be = A.mixed_magnitudes(rng, (7, 3))
    coef = A.fold_back(Be, np.array([0, 0, 7]), np.arange(7), 2, 3)
    assert np.array_equal(coef[0], np.zeros(3))
    want = np.zeros(3)
    for t in range(7):
        want = want + Be[t]
    assert np.array_equal(coef[1], want)

"""slm_gram_rows_update and slm_cv_score_rows against float64 numpy: Grams and residual sums of arbitrary row
lists (the batched search over CV splits that are not one partition of the rows)."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

EPS = np.finfo(np.float64).eps


@pytest.fixture(scope="module")
def eng():
    from sparselm_b200.engine import get_engine

    e = get_engine()
    yield e
    e.set_option("tma", 15)


def _design(eng, n, p, seed, sw=None):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, p))
    y = X[:, :3] @ [1.0, -2.0, 0.5] + rng.standard_normal(n)
    Xa = eng.pack(X, y, sw)
    return X, y, Xa, Xa.cpu().numpy()


def _lists(n, lens, rng):
    lists = [np.sort(rng.choice(n, int(L), replace=False)) for L in lens]
    ptr = np.concatenate([[0], np.cumsum([len(v) for v in lists])]).astype(np.int64)
    return lists, ptr, np.concatenate(lists).astype(np.int32)


@pytest.mark.parametrize("tma", [True, False], ids=["tma", "cp_async"])
@pytest.mark.parametrize("p", [126, 127, 254])
def test_gram_rows_update_matches_numpy(eng, p, tma):
    n = 300
    _, _, Xa, Xh = _design(eng, n, p, p)
    pa = Xa.shape[1]
    rng = np.random.default_rng(p)
    # list lengths across the 4-row gather and 32-row slab edges, n-1 and n, then enough problems for two launches
    lens = [0, 1, 3, 4, 5, 31, 33, n - 1, n] + list(rng.integers(0, n, 30))
    lists, ptr, rows = _lists(n, lens, rng)
    rows_dev = eng.to_device(rows)
    S = len(lists)
    G0 = rng.standard_normal((S, pa, pa))
    G0 = G0 + G0.transpose(0, 2, 1)
    eng.set_option("tma", 15 if tma else 0)
    try:
        for mode in ("plain", "accumulate", "negate"):
            G = torch.from_numpy(G0).to(eng.device)
            tma0 = eng.tma_launch_count()
            eng.gram_rows_update(Xa, ptr, rows_dev, G, accumulate=mode != "plain", negate=mode == "negate")
            assert (eng.tma_launch_count() > tma0) == tma
            got = G.cpu().numpy()
            for s, idx in enumerate(lists):
                A = Xh[idx]
                prod = A.T @ A
                if len(idx) == 0:
                    want = G0[s]  # an empty list leaves the Gram untouched
                elif mode == "plain":
                    want = prod
                elif mode == "accumulate":
                    want = G0[s] + prod
                else:
                    want = G0[s] - prod
                # DGEMM error bound of both products: 2 (k + 2) eps |A|^T |A| (+ eps |G0| for the addition)
                bound = 2 * (len(idx) + 2) * EPS * (np.abs(A).T @ np.abs(A)) + 2 * EPS * np.abs(G0[s])
                assert np.all(np.abs(got[s] - want) <= bound + 1e-300), (mode, s, len(idx))
                assert np.array_equal(got[s], got[s].T), (mode, s)  # upper tiles + bit-identical mirror
            if mode == "plain":
                G2 = torch.from_numpy(G0).to(eng.device)
                eng.gram_rows_update(Xa, ptr, rows_dev, G2)
                assert torch.equal(G, G2)  # fixed stream-K fix-up order: bitwise reproducible
    finally:
        eng.set_option("tma", 15)


@pytest.mark.parametrize("tma", [True, False], ids=["tma", "cp_async"])
def test_downdate_equals_direct_build(eng, tma):
    n, p = 3000, 127
    _, _, Xa, Xh = _design(eng, n, p, 5)
    pa = Xa.shape[1]
    rng = np.random.default_rng(6)
    train = np.sort(rng.choice(n, 2200, replace=False))
    out = np.setdiff1d(np.arange(n), train)
    eng.set_option("tma", 15 if tma else 0)
    try:
        G_full = eng.gram_blocks(Xa, np.array([0, n]))[0]
        direct = torch.empty((1, pa, pa), dtype=torch.float64, device=eng.device)
        eng.gram_rows_update(Xa, np.array([0, len(train)]), eng.to_device(train.astype(np.int32)), direct)
        down = G_full.clone()[None]
        eng.gram_rows_update(Xa, np.array([0, len(out)]), eng.to_device(out.astype(np.int32)), down, accumulate=True,
                             negate=True)
        gf, d, dd = G_full.cpu().numpy(), direct[0].cpu().numpy(), down[0].cpu().numpy()
    finally:
        eng.set_option("tma", 15)
    ref = Xh[train].T @ Xh[train]
    scale = np.abs(gf).max()
    # the downdate carries the rounding of the full Gram (3000-term sums): within 1024 eps ||G_full||_max of the
    # direct build; a wrong row or tile would be off by O(||G_full|| / n)
    assert np.abs(dd - d).max() <= 1024 * EPS * scale
    assert np.abs(d - ref).max() <= 1024 * EPS * scale
    assert np.array_equal(dd, dd.T)


def test_cv_score_rows_matches_numpy(eng):
    n, p, K = 200, 37, 13
    rng = np.random.default_rng(3)
    sw = 0.3 + rng.random(n)
    X, y, Xa, _ = _design(eng, n, p, 4, sw)
    B = rng.standard_normal((p, 16))
    icpt = rng.standard_normal(K)
    Bd, icd = eng.to_device(B), eng.to_device(icpt)
    lists = [np.array([7]), np.array([0, 5, 199]), np.sort(rng.choice(n, 57, replace=False)), np.arange(n),
             np.array([n - 1])]
    devs = [eng.to_device(v.astype(np.int32)) for v in lists]
    items = [(r, Bd, K, icd if i % 2 == 0 else None) for i, r in enumerate(devs)]
    res = eng.cv_score_rows(Xa, p, items, rows_scaled=True).cpu().numpy()
    for i, idx in enumerate(lists):
        r = y[idx, None] - X[idx] @ B[:, :K] - (icpt if i % 2 == 0 else 0.0)  # unweighted residuals
        np.testing.assert_allclose(res[i, 0, :K], (r * r).sum(0), rtol=1e-12)
        np.testing.assert_allclose(res[i, 1, :K], np.abs(r).sum(0), rtol=1e-12)
    # a row list that is a contiguous range scores bitwise as the range does
    a, b = 40, 161
    rng_res = eng.cv_score_many(Xa, p, [(a, b, Bd, K, icd)], rows_scaled=True).cpu().numpy()
    row_res = eng.cv_score_rows(Xa, p, [(eng.to_device(np.arange(a, b, dtype=np.int32)), Bd, K, icd)],
                                rows_scaled=True).cpu().numpy()
    assert np.array_equal(rng_res[0, :, :K], row_res[0, :, :K])

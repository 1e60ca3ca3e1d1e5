"""The TMA-fed GEMM path (csrc/gemm_f64_tma.cuh): ground truth of the shared-memory layout the
consumers assume, and the three kernel families (Gram build, dense apply, row-sparse apply)
against the cp.async kernels and a float64 reference, tails included."""

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture()
def tma_switch(engine):
    yield engine
    engine.set_option("tma", 15)  # the engine default: later tests run on the wide-band gather kernels


def _expected_image(A, col0, rows):
    """[len(rows)][16] box image with the 128-byte swizzle: 16-byte chunk c of row r sits at chunk
    c ^ (r & 7); elements outside the matrix read as zero."""
    img = np.zeros((len(rows), 16))
    for r, gr in enumerate(rows):
        for c in range(16):
            gc = col0 + c
            v = A[gr, gc] if (0 <= gr < A.shape[0] and 0 <= gc < A.shape[1]) else 0.0
            img[r, (((c >> 1) ^ (r & 7)) << 1) + (c & 1)] = v
    return img


@pytest.mark.parametrize("col0,row0,rows4", [(0, 0, (0, 1, 2, 3)), (16, 30, (5, 39, 0, 2)), (8, 24, (7, 7, 33, 12)),
                                             (16, 32, (39, 38, 100000, 1))])
def test_tma_box_and_gather4_layout(engine, col0, row0, rows4):
    import torch

    rows, ld = 40, 24
    A = (torch.arange(rows, dtype=torch.float64)[:, None] * 100 + torch.arange(ld, dtype=torch.float64)[None, :] + 1
         ).to(engine.device).contiguous()
    out = engine.tma_probe(A, col0, row0, rows4).cpu().numpy()
    Ah = A.cpu().numpy()
    np.testing.assert_array_equal(out[:256].reshape(16, 16), _expected_image(Ah, col0, list(range(row0, row0 + 16))))
    np.testing.assert_array_equal(out[256:].reshape(4, 16), _expected_image(Ah, col0, list(rows4)))


LAYOUTS = [7, 31]  # 128-byte swizzled boxes / wide padded-pitch bands (bits 3, 4 of the "tma" option)


@pytest.mark.parametrize("mask", LAYOUTS)
@pytest.mark.parametrize("n,p,F", [(37, 5, 1), (300, 81, 3), (1000, 250, 5), (513, 130, 4), (2050, 300, 2)])
def test_tma_gram_build(tma_switch, n, p, F, mask):
    import torch

    eng = tma_switch
    rng = np.random.default_rng(n + p)
    X, y = rng.standard_normal((n, p)), rng.standard_normal(n)
    row_ptr = np.linspace(0, n, F + 1).astype(np.int64)
    Xa = eng.pack(X, y)
    eng.set_option("tma", 0)
    G0 = eng.gram_blocks(Xa, row_ptr)
    c0 = eng.tma_launch_count()
    eng.set_option("tma", mask)
    G1 = eng.gram_blocks(Xa, row_ptr)
    assert eng.tma_launch_count() > c0, "the TMA kernel did not run"
    Xh = Xa.cpu().numpy()
    for f in range(F):
        ref = Xh[row_ptr[f]:row_ptr[f + 1]].T @ Xh[row_ptr[f]:row_ptr[f + 1]]
        scale = np.abs(ref).max()
        assert np.abs(G1[f].cpu().numpy() - ref).max() <= 1e-13 * scale * max(1, n // F) ** 0.5
        assert torch.equal(G1[f], G1[f].T)
        assert (G1[f] - G0[f]).abs().max().item() <= 1e-13 * scale * max(1, n // F) ** 0.5
    # accumulate into an existing Gram (slm_gram_block_add)
    Gacc = G1[0].clone()
    eng._gram_block_into(Xa, int(row_ptr[0]), int(row_ptr[1]), Gacc, accumulate=True)
    assert (Gacc - 2 * G1[0]).abs().max().item() <= 1e-12 * G1[0].abs().max().item()


@pytest.mark.parametrize("mask", LAYOUTS)
@pytest.mark.parametrize("p,Ks", [(80, [1]), (80, [10, 7]), (515, [100, 100, 100]), (1030, [33]), (300, [64, 0, 9])])
def test_tma_dense_apply(tma_switch, p, Ks, mask):
    import torch

    eng = tma_switch
    eng.set_option("tma", mask)
    F = len(Ks)
    pa = eng.padded_cols(p)
    g = torch.Generator(device="cpu").manual_seed(p)
    G = torch.randn((F, pa, pa), dtype=torch.float64, generator=g)
    G = (G + G.transpose(1, 2)).to(eng.device).contiguous()
    ldz = max(8, (max(Ks) + 7) // 8 * 8)
    Z = torch.randn((F, p, ldz), dtype=torch.float64, generator=g).to(eng.device)
    c0 = eng.tma_launch_count()
    GZ = eng.gram_apply(G, p, Ks, Z)
    assert eng.tma_launch_count() > c0
    for f in range(F):
        if Ks[f] == 0:
            continue
        ref = G[f, :p, :p] @ Z[f, :, :Ks[f]]
        assert (GZ[f, :, :Ks[f]] - ref).abs().max().item() <= 1e-12 * ref.abs().max().item()


@pytest.mark.parametrize("p,Ks,chunk_w,density", [(515, [100, 64], 32, 0.3), (300, [40], 8, 0.05), (1030, [33, 33, 8], 16, 0.6),
                                                  (200, [24], 32, 0.0), (257, [16, 72], 32, 1.0)])
@pytest.mark.parametrize("mask", LAYOUTS)
def test_tma_rowsparse_apply(tma_switch, p, Ks, chunk_w, density, mask):
    import torch

    eng = tma_switch
    eng.set_option("tma", mask)
    F = len(Ks)
    pa = eng.padded_cols(p)
    g = torch.Generator(device="cpu").manual_seed(p + 1)
    G = torch.randn((F, pa, pa), dtype=torch.float64, generator=g)
    G = (G + G.transpose(1, 2)).to(eng.device).contiguous()
    ldz = max(8, (max(Ks) + 7) // 8 * 8)
    Z = torch.randn((F, p, ldz), dtype=torch.float64, generator=g)
    keep = torch.rand((F, p, 1), generator=g) < density
    Z = (Z * keep).to(eng.device)
    c0 = eng.tma_launch_count()
    GZ = eng.gram_apply_rowsparse(G, p, Ks, Z, chunk_w=chunk_w)
    if chunk_w > 16 and max(Ks) > 16:  # tiles of <= 16 columns stay on the cp.async kernel (faster start)
        assert eng.tma_launch_count() > c0
    eng.set_option("tma", 0)
    GZ0 = eng.gram_apply_rowsparse(G, p, Ks, Z, chunk_w=chunk_w)
    for f in range(F):
        ref = G[f, :p, :p] @ Z[f, :, :Ks[f]]
        tol = 1e-12 * max(ref.abs().max().item(), 1e-300)
        assert (GZ[f, :, :Ks[f]] - ref).abs().max().item() <= tol
        assert (GZ[f, :, :Ks[f]] - GZ0[f, :, :Ks[f]]).abs().max().item() <= tol


def test_solver_on_tma_kernels_agrees_with_cp_async_kernels(tma_switch):
    """A whole CV search (dense cold-start phase, row-sparse middle, tail) with the TMA-fed kernels
    against the same search on the cp.async kernels."""
    from sparselm_b200.model import Lasso
    from sparselm_b200.model_selection import GridSearchCV

    rng = np.random.default_rng(12)
    n, p = 600, 400
    X = rng.standard_normal((n, p))
    y = X @ rng.standard_normal(p) + rng.standard_normal(n)     # dense truth: dense iterates
    alphas = np.abs(X.T @ y).max() / n * np.logspace(-2.0, -4.0, 40)
    eng = tma_switch
    out = []
    for mask in (15, 0):
        eng.set_option("tma", mask)
        gs = GridSearchCV(Lasso(solver_options={"tol": 1e-11}), {"alpha": list(alphas)}, cv=3).fit(X, y)
        assert gs.batched_ and (gs.solver_info_["status"] == 0).all()
        out.append((gs.cv_results_["mean_test_score"].copy(), gs.best_estimator_.coef_.copy()))
    np.testing.assert_allclose(out[0][0], out[1][0], rtol=1e-8)
    assert np.abs(out[0][1] - out[1][1]).max() <= 1e-7 * np.abs(out[1][1]).max()


def test_tma_results_are_reproducible(tma_switch):
    """Fixed-order stream-K fix-up: two launches give bit-identical Grams."""
    import torch

    eng = tma_switch
    rng = np.random.default_rng(5)
    X, y = rng.standard_normal((3000, 700)), rng.standard_normal(3000)
    Xa = eng.pack(X, y)
    row_ptr = np.array([0, 1000, 1900, 3000], dtype=np.int64)
    G1 = eng.gram_blocks(Xa, row_ptr)
    G2 = eng.gram_blocks(Xa, row_ptr)
    assert torch.equal(G1, G2)

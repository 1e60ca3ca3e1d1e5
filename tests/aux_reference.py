"""Float64 references of the kernels that run before and after the solver loop (csrc/engine.cu: pack, complement,
triangle, centering, gather, fold-back, intercept, adaptive and power-iteration kernels; whiten_kernels.cuh;
cg_kernels.cuh), shared by tests/test_gpu_aux_kernels.py and its CPU counterpart tests/test_aux_reference.py.

- Ordered sums: the complement and fold-back kernels add their terms one by one in a fixed order.  The references
  below do the same with elementwise numpy additions in a Python loop (never `ndarray.sum`, which sums pairwise), so
  a kernel that keeps its documented order matches them bit for bit.
- `power_lambda`: the block power iteration of `slm_lipschitz` (power_norm_kernel and the tensor-core apply) on the
  CPU, with the kernel's hash start vectors, its Rayleigh quotient and running maximum.  The kernel's products and
  reductions are summed in another order, so the two agree to rounding, not bitwise.
- `gamma`: the constant of the standard error bound of a k-term sum of products, gamma_k * sum |terms|.
"""

from __future__ import annotations

import numpy as np

U = np.finfo(np.float64).eps / 2  # unit roundoff


def gamma(k):
    k = np.asarray(k, dtype=np.float64)
    return k * U / (1.0 - k * U)


# ---- ordered sums ---------------------------------------------------------------------------------------------------
def ordered_total(blocks):
    """0.0 + G_0 + G_1 + ... in ascending order (gram_complement_kernel's and tri_complement_kernel's total)."""
    tot = np.zeros_like(blocks[0])
    for b in blocks:
        tot = tot + b
    return tot


def ordered_complements(blocks):
    """Complement f = 0.0 + sum of G_g over g != f, ascending (exactly 0 for a single block)."""
    out = []
    for f in range(len(blocks)):
        acc = np.zeros_like(blocks[0])
        for g, b in enumerate(blocks):
            if g != f:
                acc = acc + b
        out.append(acc)
    return out


def fold_back(Be, inv_ptr, inv_idx, p, K):
    """coef[j][k] = 0.0 + Be[inv_idx[t]][k] for t = inv_ptr[j] .. inv_ptr[j+1]-1, in that order."""
    coef = np.zeros((p, K))
    for j in range(p):
        acc = np.zeros(K)
        for t in range(inv_ptr[j], inv_ptr[j + 1]):
            acc = acc + Be[inv_idx[t], :K]
        coef[j] = acc
    return coef


def mixed_magnitudes(rng, shape, share=0.3):
    """Non-integer values of magnitude ~1 and ~1e16 side by side: any change of summation order changes bits."""
    return rng.standard_normal(shape) * np.where(rng.random(shape) < share, 1e16, 1.0)


# ---- block power iteration (slm_lipschitz) --------------------------------------------------------------------------
PN_COLS = 8  # start vectors per Gram


def power_start(p, f):
    """The kernel's start block V[p][8] of Gram f of a call: a 32-bit multiplicative hash of (row, column, f)."""
    idx = np.arange(p * PN_COLS, dtype=np.uint64).reshape(p, PN_COLS)
    m32 = np.uint64(0xFFFFFFFF)
    h = (idx * np.uint64(2654435761) + np.uint64(12345 * (f + 1))) & m32
    h ^= h >> np.uint64(15)
    h = (h * np.uint64(2246822519)) & m32
    h ^= h >> np.uint64(13)
    return (h & np.uint64(0xFFFFFF)).astype(np.float64) / 8388608.0 - 1.0


def power_lambda(G, iters, f=0):
    """Largest Rayleigh quotient v.w / v.v (0 when v.v = 0) over the 8 columns and all iterations of
    W = G V, V <- W / ||W||, from the start block of Gram f.  A lower bound of lambda_max(G)."""
    G = np.asarray(G, dtype=np.float64)
    V = power_start(G.shape[0], f)
    lam = 0.0
    for _ in range(iters):
        W = G @ V
        vw = np.einsum("ij,ij->j", V, W)
        vv = np.einsum("ij,ij->j", V, V)
        ww = np.einsum("ij,ij->j", W, W)
        q = np.where(vv > 0.0, vw / np.where(vv > 0.0, vv, 1.0), 0.0)
        lam = max(lam, float(q.max()))
        V = W * np.where(ww > 0.0, 1.0 / np.sqrt(np.where(ww > 0.0, ww, 1.0)), 0.0)
    return lam


def spike_over_bulk(seed, n, p, bulk):
    """Design X [n][p] whose Gram X^T X has one eigenvalue n and p - 1 eigenvalues bulk * n (random
    eigenvectors): the block power iteration's Rayleigh quotient stays well below lambda_max."""
    rng = np.random.default_rng(seed)
    U, _ = np.linalg.qr(rng.standard_normal((n, p)))
    Q, _ = np.linalg.qr(rng.standard_normal((p, p)))
    d = np.full(p, bulk)
    d[0] = 1.0
    return np.sqrt(n) * (U * np.sqrt(d)) @ Q.T

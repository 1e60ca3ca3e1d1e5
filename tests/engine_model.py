"""Numpy model of the CUDA engine's algorithm (kernel-by-kernel), used by tests.

This is NOT a product path and not the oracle: it mirrors the exact arithmetic of
the kernels in ``sparselm_b200/csrc`` (same recurrences, same order of
operations up to reduction order) so that GPU unit tests can compare single
kernels against it, and so that the algorithm's convergence behaviour can be
studied on CPU.  Layout mirrors the device: state matrices are (p, K) with the
batch columns contiguous.
"""

from __future__ import annotations

import numpy as np


def soft(v, t):
    return np.sign(v) * np.maximum(np.abs(v) - t, 0.0)


def group_dual_norm(g, w1, w2, iters=100):
    """Vectorised epsilon-norm for one group: g (s, K), w1 (s, K), w2 (K,)."""
    a = np.abs(g)
    g2 = np.sqrt((a * a).sum(0))
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(a > 0, np.where(w1 > 0, a / np.where(w1 > 0, w1, 1), np.inf), 0.0).max(0)
        hi = np.where(w2 > 0, np.minimum(g2 / np.where(w2 > 0, w2, 1), ratio), ratio)
    lo = np.zeros_like(hi)
    need = (w2 > 0) & (g2 > 0) & np.isfinite(hi) & (ratio > 0)
    # pure group (w1==0) or pure l1 (w2==0) have closed forms == hi already
    need &= (w1 > 0).any(0)
    for _ in range(iters):
        mid = 0.5 * (lo + hi)
        u = soft(g, mid * w1)
        feas = np.sqrt((u * u).sum(0)) <= mid * w2
        hi = np.where(need & feas, mid, hi)
        lo = np.where(need & ~feas, mid, lo)
    return np.where(g2 > 0, hi, 0.0)


class BatchProblem:
    """One fold: Gram G (p,p), c (p,), yty, n; K columns with weights."""

    def __init__(self, G, c, yty, n, gptr, W1, W2, D2, L=None):
        self.G, self.c, self.yty, self.n = G, c, float(yty), float(n)
        self.gptr = np.asarray(gptr)
        self.W1, self.W2, self.D2 = W1, W2, D2  # (p,K), (Gn,K), (Gn,K)
        self.p, self.K = W1.shape
        self.L = L if L is not None else np.linalg.eigvalsh(G)[-1] / n
        self.gid = np.repeat(np.arange(len(self.gptr) - 1), np.diff(self.gptr))


SMOOTH_KAPPA = 64.0  # kSmoothKappa of csrc/solver_kernels.cuh


def smooth_rows(pb: BatchProblem):
    """(p, K) mask of the rows without any penalty: w1_j = 0 in a group with w2_g = 0."""
    return (pb.W1 == 0) & (pb.W2[pb.gid] == 0)


def smooth_ok(pb: BatchProblem, B, GB, kappa=SMOOTH_KAPPA):
    """Per column: every smooth row is stationary to the rounding bound of (c - G b)_j,
    |g_j| <= kappa * eps * (|c_j| + sqrt(G_jj) * sum_k sqrt(G_kk) |b_k|) / n (gap kernels)."""
    return smooth_excess(pb, B, GB) <= kappa


def smooth_excess(pb: BatchProblem, B, GB):
    """Per column: max over the smooth rows of |g_j| / tau_j at kappa = 1 (0 without smooth rows)."""
    g = np.abs((pb.c[:, None] - GB) / pb.n - pb.D2[pb.gid] * B)
    d = np.sqrt(np.diag(pb.G))
    tau = np.finfo(float).eps * (np.abs(pb.c)[:, None] + d[:, None] * (d[:, None] * np.abs(B)).sum(0)) / pb.n
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(smooth_rows(pb) & (g > 0), g / tau, 0.0)
    return r.max(0)


def gap_terms(pb: BatchProblem, B, GB):
    """Primal, dual, gap per column from Gram quantities (gap kernel).  Smooth rows stay out of
    the dual norm: their dual constraint g_j = 0 is tested separately (smooth_ok)."""
    n = pb.n
    cb = pb.c @ B
    bgb = (B * GB).sum(0)
    ss = np.add.reduceat(B * B, pb.gptr[:-1], axis=0)
    pen = (pb.W1 * np.abs(B)).sum(0) + (pb.W2 * np.sqrt(ss)).sum(0)
    ridge = (pb.D2 * ss).sum(0)
    g = (pb.c[:, None] - GB) / n - pb.D2[pb.gid] * B
    g = np.where(smooth_rows(pb), 0.0, g)
    omega = np.zeros(pb.K)
    for gi in range(len(pb.gptr) - 1):
        a, b = pb.gptr[gi], pb.gptr[gi + 1]
        omega = np.maximum(omega, group_dual_norm(g[a:b], pb.W1[a:b], pb.W2[gi]))
    rr = pb.yty - 2 * cb + bgb
    rr_aug = rr + n * ridge
    yr = pb.yty - cb
    P = rr_aug / (2 * n) + pen
    s = np.where(omega > 1, 1 / np.where(omega > 1, omega, 1), 1.0)
    s = np.where(np.isfinite(omega), s, 0.0)
    D = (2 * s * yr - s * s * rr_aug) / (2 * n)
    return P, D, P - D


def prox_step(pb: BatchProblem, Z, B, GZ, GBprev, theta, tmom, done):
    """One fused epilogue: GB recurrence, prox, restart test, momentum.
    Returns (Znew, Bnew, GB, theta_new, tmom_new)."""
    step = 1.0 / pb.L
    GB = (GZ + theta * GBprev) / (1.0 + theta)
    V = Z - step * (GZ - pb.c[:, None]) / pb.n
    U = soft(V, step * pb.W1)
    ss = np.add.reduceat(U * U, pb.gptr[:-1], axis=0)
    nrm = np.sqrt(ss)
    with np.errstate(divide="ignore", invalid="ignore"):
        sc = np.where(nrm > 0, np.maximum(0.0, 1.0 - step * pb.W2 / np.where(nrm > 0, nrm, 1)), 0.0)
    sc = sc / (1.0 + step * pb.D2)
    Bn = U * sc[pb.gid]
    dot = ((Z - Bn) * (Bn - B)).sum(0)
    restart = dot > 0
    tn = (1 + np.sqrt(1 + 4 * tmom * tmom)) / 2
    th = (tmom - 1) / tn
    th = np.where(restart, 0.0, th)
    tn = np.where(restart, 1.0, tn)
    Zn = Bn + th * (Bn - B)
    # frozen columns keep their state
    Zn = np.where(done, Z, Zn)
    Bn = np.where(done, B, Bn)
    GB = np.where(done, GBprev, GB)
    th = np.where(done, theta, th)
    tn = np.where(done, tmom, tn)
    return Zn, Bn, GB, th, tn


def solve(pb: BatchProblem, tol=1e-10, floor_rel=1e-14, max_iter=20000, check_every=10, B0=None):
    p, K = pb.p, pb.K
    B = np.zeros((p, K)) if B0 is None else B0.copy()
    Z = B.copy()
    GB = pb.G @ B
    theta = np.zeros(K)
    tmom = np.ones(K)
    done = np.zeros(K, bool)
    iters = np.zeros(K, int)
    floor = max(floor_rel, 4e-15 / tol) * pb.yty / (2 * pb.n)  # rounding floor of the Gram-form gap
    gap = np.full(K, np.inf)
    for it in range(max_iter):
        GZ = pb.G @ Z
        if it % check_every == 0:
            GBk = np.where(done, GB, (GZ + theta * GB) / (1 + theta))
            P, D, g = gap_terms(pb, B, GBk)
            newly = (~done) & (g <= tol * np.maximum(np.abs(P), floor)) & smooth_ok(pb, B, GBk)
            gap = np.where(done, gap, g)
            iters[newly] = it
            if newly.any():
                # freeze at B_k: Z := B so the state is consistent
                Z = np.where(newly, B, Z)
                GB = np.where(newly, GBk, GB)
                theta = np.where(newly, 0.0, theta)
            done |= newly
            if done.all():
                break
        Z, B, GB, theta, tmom = prox_step(pb, Z, B, GZ, GB, theta, tmom, done)
    iters[~done] = max_iter
    GBx = pb.G @ B
    P, D, g = gap_terms(pb, B, GBx)
    return B, {"iters": iters, "gap": g, "primal": P, "done": done, "total_iters": it}


def solve_fused(pb: BatchProblem, tol=1e-10, floor_rel=1e-14, max_iter=20000, check_every=10, B0=None):
    """The fused iteration of csrc/solver_kernels.cuh (prox_fused_kernel) in numpy: the state is W_t, W_{t-1},
    G W_t, G W_{t-1}; the Gram acts on the iterate, the extrapolated point and its product are formed on the fly at
    the START of iteration t, when the restart test of iteration t-1 is known:

        z_t = W_t + th_t (W_t - W_{t-1}),   G z_t = (1 + th_t) G W_t - th_t G W_{t-1},
        th_t = (t_{k-1} - 1) / t_k  unless  dot_{t-1} = sum (z_{t-1} - W_t)(W_t - W_{t-1}) > 0  (then th_t = 0, t_k = 1).

    Same restart rule and theta sequence as `solve` (the two-kernel form): the iterates agree up to rounding."""
    p, K = pb.p, pb.K
    W = np.zeros((p, K)) if B0 is None else B0.copy()
    Wold = W.copy()
    GWold = np.zeros((p, K))
    tm = np.ones(K)                 # t_{k-1}
    dot = np.zeros(K)               # restart dot of the previous iteration
    done = np.zeros(K, bool)
    iters = np.zeros(K, int)
    floor = max(floor_rel, 4e-15 / tol) * pb.yty / (2 * pb.n)
    step = 1.0 / pb.L
    for it in range(max_iter):
        GW = pb.G @ W               # exact product of the iterate (the kernel contracts over its support rows)
        if it % check_every == 0:
            P, D, g = gap_terms(pb, W, GW)
            newly = (~done) & (g <= tol * np.maximum(np.abs(P), floor)) & smooth_ok(pb, W, GW)
            iters[newly] = it
            done |= newly
            if done.all():
                break
        if it == 0:
            th, tn = np.zeros(K), tm.copy()
        else:
            tn = (1 + np.sqrt(1 + 4 * tm * tm)) / 2
            th = (tm - 1) / tn
            th = np.where(dot > 0, 0.0, th)
            tn = np.where(dot > 0, 1.0, tn)
        Z = W + th * (W - Wold)
        GZ = GW + th * (GW - GWold)
        V = Z - step * (GZ - pb.c[:, None]) / pb.n
        U = soft(V, step * pb.W1)
        ss = np.add.reduceat(U * U, pb.gptr[:-1], axis=0)
        nrm = np.sqrt(ss)
        with np.errstate(divide="ignore", invalid="ignore"):
            sc = np.where(nrm > 0, np.maximum(0.0, 1.0 - step * pb.W2 / np.where(nrm > 0, nrm, 1)), 0.0)
        sc = sc / (1.0 + step * pb.D2)
        Wn = U * sc[pb.gid]
        dot_new = ((Z - Wn) * (Wn - W)).sum(0)
        # finished columns keep their state (settle_done_kernel: the final iterate sits in both buffers)
        Wold = np.where(done, W, W)
        GWold = np.where(done, GWold, GW)
        W = np.where(done, W, Wn)
        tm = np.where(done, tm, tn)
        dot = np.where(done, dot, dot_new)
    iters[~done] = max_iter
    P, D, g = gap_terms(pb, W, pb.G @ W)
    return W, {"iters": iters, "gap": g, "primal": P, "done": done, "total_iters": it}

"""Second-order phase for slow columns of a batched solve: lock-step Newton on the active manifold.

Why (DESIGN.md section 4, "C4, the ill-conditioned case"): accelerated proximal-gradient iterations need
~sqrt(condition number) iterations.  A group-penalised problem whose penalty is nearly flat on its
support (the adaptive passes weight an active group by alpha^2/||b_g||, reference
_adaptive_lasso.py:364-374) on a Gram with exactly flat directions (the duplicated columns of the
overlap expansion, _lasso.py:440-461) reaches condition numbers of 1e6 and more: the active groups
settle after a few hundred iterations and 10^4 more crawl along the flat directions.  On the
settled support the objective

    phi(b) = 1/(2n) b' G b - c' b / n + sum_g w_g ||b_g|| + 1/2 sum_g d_g ||b_g||^2,   b_g = 0 off the support,

is smooth (||b_g|| > 0 on every active group), so a damped Newton iteration finishes in a handful of
factorisations.  The conic interior-point solvers behind the reference's cvxpy call
(_base.py:512-519) are second-order methods too.

What this module does: host-side orchestration, all slow columns in lock step.  On the GPU
(``newton_phase_device``) every Newton step is ONE call into the engine (``slm_newton_step``,
csrc/newton_kernels.cuh): Hessian assembly straight from the Gram on the active coordinates of every column, a
batched blocked Cholesky whose trailing updates run on the TMA-fed FP64 tensor-core GEMM, blocked triangular solves and the Armijo line
search -- no library factorisation, no ``[k, p, p]`` copies of the Gram, no host synchronisation
inside a step.  ``newton_phase`` is the same iteration written with torch operations
(``torch.linalg.cholesky_ex``); it runs on CPU tensors in ``tests/test_newton.py`` and is the model the
kernels are tested against.  It never decides convergence: the points go back into the engine's
batch and the engine's own duality-gap certificate (exact ``G b``, all groups,
``gap_final_kernel``) judges them.  A step on a wrong support only costs time: every accepted step
decreases phi (Armijo test on the *difference* of objective values, formed without cancellation).

Scope: pure group penalties (no l1 term) with optional ridge: GroupLasso, OverlapGroupLasso,
RidgedGroupLasso and their adaptive variants (also in whitened variables, standardize=True).
On by default for 160 < p <= 2048 (engine.Engine.solve); ``solver_options={"newton": True / False}``
forces it.  ``solver_options={"newton": "l1"}`` also runs it for penalties with an l1 term (Lasso,
SparseGroupLasso and their adaptive variants; not the method-of-multipliers path of standardize=True):
steps on the manifold of fixed signs (``slm_newton_step_l1``), active set = the non-zero coordinates,
backtracking from min(1, t_cross) and exact zeros where a coordinate reaches zero -- the support only
shrinks.  Measured on an AR(1) rho = 0.99 design (n = 5000, p = 1000, DESIGN.md section 4,
profiles/r03_newton_l1_probe.jsonl): AdaptiveLasso fit 85 -> 58 ms (2717 -> 300 iterations), Lasso 20 x 5
search 384 -> 222 ms, SparseGroupLasso 20 x 5 search 430 -> 398 ms, answers equal to 2e-10.  Measured on C4 (AdaptiveOverlapGroupLasso, 20 alphas x 5 folds x 3 passes, p_ext = 1961): 0.41 s per
search against 12.4 s first-order only (round 1 with torch / cuSOLVER: 1.25 s), 1155 iterations against 129 350,
no column left on max_iter (6 before), scores equal to 3e-8 relative; 1384 factorisations per search on the active
coordinates of every column (DESIGN.md section 4).
"""

from __future__ import annotations

import os
import sys

import torch

__all__ = ["newton_phase", "newton_phase_device"]


def _gsum(v, gid, n_groups):
    """Per-column group sums: v [K, p] -> [K, n_groups]."""
    out = torch.zeros((v.shape[0], n_groups), dtype=v.dtype, device=v.device)
    out.index_add_(1, gid, v)
    return out


def newton_phase(Gs, fold, n_obs, X, w2, d2, gid, scale, tol, max_steps=12, chol_batched=True, w1=None):
    """Lock-step damped Newton iteration for K columns.

    Gs [F, pa, pa] Grams (rows/cols < p: X'X, row p: X'y), fold [K] int64 (Gram of every column),
    n_obs [K] rows of the data term, X [K, p] start points (solver feature order), w2 [K, Gn] group
    weights, d2 [K, Gn] ridge weights or None, gid [p] int64 group of every feature, scale [K] =
    max(|P|, floor) of the engine's relative test, tol its tolerance: a column is finished once the
    Newton decrement says phi - phi* <= 1e-3 * tol * scale after a full step.

    w1 [K, p]: per-coordinate l1 weights (None: pure group penalty).  Then the step works on the manifold of
    fixed signs: only the non-zero coordinates are active, the gradient gains w1 * sign(x), backtracking starts
    from min(1, t_cross) (the first sign change along the direction) and a step accepted at t_cross stores the
    coordinates that reach zero as exact zeros.

    Returns (X_new [K, p], info) with info = dict(steps [K], factorizations int, finished [K] bool).
    """
    K, p = X.shape
    Gn = w2.shape[1]
    dt, dev = X.dtype, X.device
    X = X.clone()
    same = (gid[:, None] == gid[None, :]).to(dt)                      # [p, p] shared by all columns
    steps = torch.zeros(K, dtype=torch.int64, device=dev)
    finished = torch.zeros(K, dtype=torch.bool, device=dev)
    live = torch.arange(K, device=dev)                                # columns still iterating
    target = 1e-3 * tol * scale
    n_fact = 0
    small_t = torch.zeros(K, dtype=torch.int64, device=dev)
    for _ in range(max_steps):
        if live.numel() == 0:
            break
        x = X.index_select(0, live)                                   # [k, p]
        k = x.shape[0]
        n = n_obs.index_select(0, live)[:, None]
        w = w2.index_select(0, live)
        d = torch.zeros_like(w) if d2 is None else d2.index_select(0, live)
        f = fold.index_select(0, live)
        nrm_g = torch.sqrt(_gsum(x * x, gid, Gn))                     # [k, Gn]
        act_g = nrm_g > 0
        act = act_g.index_select(1, gid)                              # [k, p]
        if w1 is not None:
            w1l = w1.index_select(0, live)
            act = act & (x != 0)
        actf = act.to(dt)
        safe = torch.where(act_g, nrm_g, torch.ones_like(nrm_g))
        nrm = safe.index_select(1, gid)
        u = x / nrm * actf
        wp = w.index_select(1, gid) * actf
        dp = d.index_select(1, gid) * actf
        kk = wp / nrm
        GA = Gs.index_select(0, f)[:, :p, :p] / n[:, :, None]         # [k, p, p]
        cA = Gs[f, p, :p] / n
        Gx = torch.bmm(GA, x[:, :, None])[:, :, 0]
        gs = (Gx - cA) * actf                                         # gradient of the quadratic part
        grad = gs + wp * u + dp * x
        if w1 is not None:
            grad = grad + w1l * torch.sign(x)
        H = GA * actf[:, :, None] * actf[:, None, :]
        H -= same[None] * (kk * u)[:, :, None] * u[:, None, :]
        H.diagonal(dim1=1, dim2=2).add_(kk + dp + (1.0 - actf))       # identity on the inactive coordinates
        if chol_batched:
            L, err = torch.linalg.cholesky_ex(H)
        else:
            L = torch.empty_like(H)
            err = torch.zeros(k, dtype=torch.int32, device=dev)
            for i in range(k):
                L[i], err[i] = torch.linalg.cholesky_ex(H[i])
        n_fact += k
        del H
        ok = err == 0
        dlt = -torch.cholesky_solve(grad[:, :, None], torch.where(ok[:, None, None], L, torch.eye(p, dtype=dt, device=dev)[None]))[:, :, 0]
        dlt = dlt * actf
        del L
        gd = (grad * dlt).sum(1)                                      # = -decrement^2
        dec = -gd
        Gd = torch.bmm(GA, dlt[:, :, None])[:, :, 0]
        del GA
        q1, q2 = (gs * dlt).sum(1), (dlt * Gd).sum(1)
        xd, dd = x * dlt, dlt * dlt
        r1, r2 = (dp * xd).sum(1), (dp * dd).sum(1)
        g1, g2 = _gsum(xd, gid, Gn), _gsum(dd, gid, Gn)
        t = torch.ones(k, dtype=dt, device=dev)
        if w1 is not None:
            l1d = (w1l * torch.sign(x) * dlt).sum(1)                  # slope of the l1 term up to t_cross
            cross = torch.where(x * dlt < 0, -x / dlt, torch.full_like(x, float("inf")))
            t = torch.clamp(cross.min(1).values, max=1.0)
        accepted = torch.zeros(k, dtype=torch.bool, device=dev)
        usable = ok & (dec > 0)
        for _ls in range(24):                                         # Armijo backtracking, per column
            dsq = 2.0 * t[:, None] * g1 + (t * t)[:, None] * g2       # ||x_g + t d_g||^2 - ||x_g||^2
            new_nrm = torch.sqrt(torch.clamp(nrm_g * nrm_g + dsq, min=0.0))
            dpen = (w * dsq / (new_nrm + safe)).sum(1)
            dphi = t * q1 + 0.5 * t * t * q2 + t * r1 + 0.5 * t * t * r2 + dpen
            if w1 is not None:
                dphi = dphi + t * l1d
            good = usable & ~accepted & (dphi <= 1e-4 * t * gd)
            accepted |= good
            t = torch.where(accepted | ~usable, t, 0.5 * t)
            if bool((accepted | ~usable).all()):
                break
        t = torch.where(accepted, t, torch.zeros_like(t))
        x_new = x + t[:, None] * dlt
        if w1 is not None:                                            # the coordinates that reach zero at t_cross
            x_new = torch.where(cross <= t[:, None], torch.zeros_like(x_new), x_new)
        X.index_copy_(0, live, x_new)
        steps.index_add_(0, live, accepted.to(torch.int64))
        full = accepted & (t == 1.0)
        fin = full & (0.5 * dec <= target.index_select(0, live))
        st = small_t.index_select(0, live)
        st = torch.where(accepted & (t < 1e-4), st + 1, torch.zeros_like(st))
        small_t.index_copy_(0, live, st)
        finished.index_copy_(0, live, fin)
        keep = accepted & ~fin & (st < 2)                             # not accepted / crawling: back to the engine
        live = live[keep]
    return X, {"steps": steps, "factorizations": n_fact, "finished": finished}


def newton_phase_device(engine, Gs, fold, n_obs, X, w2, d2, gptr_dev, gid_dev, scale, tol, max_steps=12, w1=None):
    """The same lock-step iteration as ``newton_phase`` with every step done by the engine's kernels
    (``slm_newton_step``; ``slm_newton_step_l1`` with l1 weights).  Gs [F, pa, pa] device Grams, fold [K] int64,
    n_obs [K], X [K, p] start points, w2 [K, Gn], d2 [K, Gn] or None, gptr_dev int32 [Gn+1], gid_dev int32 [p],
    scale [K], tol, w1 [K, p] or None.
    One small device-to-host read per step (accepted / step length / decrement of every column)."""
    import ctypes

    import numpy as np

    K, p = X.shape
    Gn = w2.shape[1]
    dev, dt = X.device, X.dtype
    F, pa = Gs.shape[0], Gs.shape[-1]
    ldv = (p + 7) // 8 * 8
    Xw = torch.zeros((K, ldv), dtype=dt, device=dev)
    Xw[:, :p] = X
    fold_h = fold.cpu().numpy().astype(np.int32)
    steps = torch.zeros(K, dtype=torch.int64)
    finished = torch.zeros(K, dtype=torch.bool)
    small_t = torch.zeros(K, dtype=torch.int64)
    live = torch.arange(K)
    target = (1e-3 * tol * scale).cpu()
    n_obs = n_obs.to(dt).contiguous()
    w2 = w2.contiguous()
    d2 = None if d2 is None else d2.contiguous()
    W1w = None
    if w1 is not None:
        W1w = torch.zeros((K, ldv), dtype=dt, device=dev)
        W1w[:, :p] = w1
    nbytes = engine.lib.slm_newton_workspace(p, Gn, K, F)
    work = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    out = torch.zeros((K, 4), dtype=dt, device=dev)
    n_fact = 0
    for _ in range(max_steps):
        k = int(live.numel())
        if k == 0:
            break
        ld = live.to(dev)
        xs = Xw.index_select(0, ld).contiguous()
        fh = np.ascontiguousarray(fold_h[live.numpy()])
        # the gathered operands are named: a temporary would hand its memory back to the caching allocator
        # (and to the next temporary) before the call that reads it is enqueued
        nn_s = n_obs.index_select(0, ld).contiguous()
        w2_s = w2.index_select(0, ld).contiguous()
        d2_s = None if d2 is None else d2.index_select(0, ld).contiguous()
        fp = fh.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))
        if W1w is None:
            engine._ck(engine.lib.slm_newton_step(
                engine.h, engine._ptr(Gs), pa * pa, pa, p, F, k, fp, engine._ptr(nn_s), engine._ptr(xs),
                engine._ptr(w2_s), engine._ptr(d2_s), engine._ptr(gptr_dev), engine._ptr(gid_dev), Gn,
                engine._ptr(work), nbytes, engine._ptr(out), engine.stream), "slm_newton_step")
        else:
            w1_s = W1w.index_select(0, ld).contiguous()
            engine._ck(engine.lib.slm_newton_step_l1(
                engine.h, engine._ptr(Gs), pa * pa, pa, p, F, k, fp, engine._ptr(nn_s), engine._ptr(xs),
                engine._ptr(w2_s), engine._ptr(d2_s), engine._ptr(w1_s), engine._ptr(gptr_dev), engine._ptr(gid_dev),
                Gn, engine._ptr(work), nbytes, engine._ptr(out), engine.stream), "slm_newton_step_l1")
        info = out[:k].cpu()  # the step's only host synchronisation
        n_fact += k
        accepted = info[:, 0] > 0
        t, dec = info[:, 1], info[:, 2]
        Xw.index_copy_(0, ld, xs)
        steps[live] += accepted.to(torch.int64)
        fin = accepted & (t == 1.0) & (0.5 * dec <= target[live])
        st = small_t[live]
        st = torch.where(accepted & (t < 1e-4), st + 1, torch.zeros_like(st))
        small_t[live] = st
        finished[live] = fin
        if os.environ.get("SLM_TRACE"):
            print(f"[slm newton step] k={k} accepted={int(accepted.sum())} full={int((t == 1.0).sum())} finished={int(fin.sum())} "
                  f"dec max {float(dec.max()):.3e} min {float(dec.min()):.3e} chol failures {int((info[:, 3] != 0).sum())} "
                  f"active coordinates of p={p}: max {int((xs[:, :p] != 0).sum(1).max())} mean {float((xs[:, :p] != 0).sum(1).double().mean()):.0f}",
                  file=sys.stderr)
        live = live[accepted & ~fin & (st < 2)]
    return Xw[:, :p].contiguous(), {"steps": steps.to(dev), "factorizations": n_fact, "finished": finished.to(dev)}

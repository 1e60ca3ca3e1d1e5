"""Float64 reference of one step of the second-order phase (``slm_newton_step``, csrc/newton_kernels.cuh;
``sparselm_b200/newton.py``), one column at a time, in plain numpy / scipy.

On the active manifold of a column (groups with ||x_g|| > 0)

    phi(x) = 1/(2n) x'Gx - c'x/n + sum_g w_g ||x_g|| + 1/2 sum_g d_g ||x_g||^2,      c = row p of the Gram,

the step factors the compacted Hessian H = G_AA/n + blockdiag_g(w_g/||x_g|| (I - u_g u_g')) + diag(d) on the
ordered active coordinates, solves H d = -grad and backtracks on phi(x + t d) - phi(x).  The line search
here uses the kernel's formulas in the kernel's order (q2 = dec - cdd, the dpen form of the penalty
difference, 24 halvings, slope 1e-4), so that its accept decision and step length can be compared with
the kernel's exactly; every tried step is recorded with its Armijo margin so that a caller can tell a
decision that rounding could flip.
"""

from __future__ import annotations

import numpy as np
import scipy.linalg as sla

ARMIJO = 1e-4
HALVINGS = 24


def group_ids(gptr):
    gptr = np.asarray(gptr, dtype=np.int64)
    return np.repeat(np.arange(len(gptr) - 1), np.diff(gptr))


def hessian_terms(G, p, n, x, w2, d2, gptr):
    """Per-coordinate quantities of the step: (act [m] ascending active coordinates, on [p] activity, nrm [Gn]
    group norms, u [p], kk [p] = w_g/||x_g||, dp [p] = d_g, gs [p] = (Gx - c)/n, grad [p]; zero off the support)."""
    gid = group_ids(gptr)
    Gn = len(gptr) - 1
    x = np.asarray(x, dtype=np.float64)
    nrm = np.sqrt(np.array([np.dot(x[gptr[g]:gptr[g + 1]], x[gptr[g]:gptr[g + 1]]) for g in range(Gn)]))
    on = (nrm > 0)[gid]
    act = np.flatnonzero(on)
    safe = np.where(nrm > 0, nrm, 1.0)[gid]
    u = np.where(on, x / safe, 0.0)
    kk = np.where(on, np.asarray(w2)[gid] / safe, 0.0)
    dp = np.where(on, 0.0 if d2 is None else np.asarray(d2)[gid], 0.0)
    gs = np.where(on, (G[:p, :p] @ x - G[p, :p]) / n, 0.0)
    grad = gs + (kk + dp) * x
    return act, on, nrm, u, kk, dp, gs, grad


def compact_hessian(G, n, act, gid, u, kk, dp):
    """H[act][act] in the kernel's order of operations: G/n, minus the group curvature, plus the diagonal."""
    H = G[np.ix_(act, act)] / n
    same = gid[act][:, None] == gid[act][None, :]
    H = H - np.where(same, (kk[act] * u[act])[:, None] * u[act][None, :], 0.0)
    H[np.diag_indices_from(H)] += kk[act] + dp[act]
    return H


def newton_step(G, p, n, x, w2, d2, gptr):
    """One damped Newton step of one column.  G [>= p+1, >= p+1] Gram (rows/cols < p: X'X, row p: X'y), n the
    row count of the data term, x [p] start point, w2 [Gn] group weights, d2 [Gn] ridge weights or None,
    gptr [Gn+1] group pointers.  Returns a dict:

    act, on ([p] activity), kk ([p] w_g/||x_g||), H (compacted, [m, m]), grad_a (grad[act]), gs, grad ([p]), d ([p], zero off the support), ok (H
    factored), dec = -grad'd, accepted, t (0 when not accepted), x_new, and trials: one (t, dphi, threshold,
    size) per tried step, size = sum of the magnitudes of the terms of dphi (the scale of its rounding)."""
    gptr = np.asarray(gptr, dtype=np.int64)
    gid = group_ids(gptr)
    x = np.asarray(x, dtype=np.float64)
    act, on, nrm, u, kk, dp, gs, grad = hessian_terms(G, p, n, x, w2, d2, gptr)
    H = compact_hessian(G, n, act, gid, u, kk, dp)
    d = np.zeros(p)
    ok = True
    if len(act):
        try:
            d[act] = -sla.cho_solve(sla.cho_factor(H, lower=False, check_finite=False), grad[act], check_finite=False)
        except np.linalg.LinAlgError:
            ok = False
    ls = line_search(x, d, on, gs, grad, u, kk, dp, np.asarray(w2, dtype=np.float64), nrm, gptr, ok)
    return dict(act=act, on=on, kk=kk, H=H, grad_a=grad[act], gs=gs, grad=grad, d=d, ok=ok, **ls)


def line_search(x, d, on, gs, grad, u, kk, dp, w2, nrm, gptr, ok=True):
    """newton_linesearch_kernel for one column: the same sums and the same tests in the same order."""
    Gn = len(gptr) - 1
    g1 = np.array([np.dot(x[gptr[g]:gptr[g + 1]], d[gptr[g]:gptr[g + 1]]) for g in range(Gn)])
    g2 = np.array([np.dot(d[gptr[g]:gptr[g + 1]], d[gptr[g]:gptr[g + 1]]) for g in range(Gn)])
    q1 = float(np.dot(gs, d))
    gd = float(np.dot(grad, d))
    r1 = float(np.sum(np.where(on, dp * x * d, 0.0)))
    r2 = float(np.sum(np.where(on, dp * d * d, 0.0)))
    ud = np.array([np.dot(u[gptr[g]:gptr[g + 1]], d[gptr[g]:gptr[g + 1]]) for g in range(Gn)])
    kkg = np.array([kk[gptr[g]] if gptr[g + 1] > gptr[g] else 0.0 for g in range(Gn)])
    cdd = float(np.sum(np.where(on, (kk + dp) * d * d, 0.0)) - np.sum(kkg * ud * ud))
    dec = -gd
    q2 = dec - cdd  # d'(G_AA/n)d through the Newton system: d'Hd = -grad'd
    usable = ok and dec > 0.0 and np.isfinite(dec)
    t, accepted, trials = 1.0, False, []
    safe = np.where(nrm > 0, nrm, 1.0)
    if usable:
        for _ in range(HALVINGS):
            dsq = 2.0 * t * g1 + t * t * g2  # ||x_g + t d_g||^2 - ||x_g||^2
            nn = np.sqrt(np.maximum(nrm * nrm + dsq, 0.0))
            terms = w2 * dsq / (nn + safe)
            dpen = float(np.sum(terms))
            dphi = t * q1 + 0.5 * t * t * q2 + t * r1 + 0.5 * t * t * r2 + dpen
            thr = ARMIJO * t * gd
            size = (abs(t * q1) + 0.5 * t * t * (abs(dec) + abs(cdd)) + abs(t * r1) + 0.5 * t * t * abs(r2)
                    + float(np.sum(np.abs(terms))) + abs(thr))
            trials.append((t, dphi, thr, size))
            if dphi <= thr:
                accepted = True
                break
            t *= 0.5
    ts = t if accepted else 0.0
    x_new = x + ts * d if accepted else x.copy()
    return dict(dec=dec, accepted=accepted, t=ts, x_new=x_new, trials=trials)


def objective_change(G, p, n, x, x_new, w2, d2, gptr):
    """phi(x_new) - phi(x) formed without cancellation (s = x_new - x): gs's + s'Gs/(2n) + penalty changes."""
    gptr = np.asarray(gptr, dtype=np.int64)
    x = np.asarray(x, dtype=np.float64)
    s = np.asarray(x_new, dtype=np.float64) - x
    quad = (G[:p, :p] @ x - G[p, :p]) @ s / n + 0.5 * s @ (G[:p, :p] @ s) / n
    pen = 0.0
    for g, (a, b) in enumerate(zip(gptr[:-1], gptr[1:])):
        n0 = np.sqrt(np.dot(x[a:b], x[a:b]))
        dsq = 2.0 * np.dot(x[a:b], s[a:b]) + np.dot(s[a:b], s[a:b])
        n1 = np.sqrt(max(n0 * n0 + dsq, 0.0))
        if n0 + n1 > 0:
            pen += w2[g] * dsq / (n0 + n1)
        if d2 is not None:
            pen += 0.5 * d2[g] * dsq
    return float(quad + pen)

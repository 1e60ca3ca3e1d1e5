"""Float64 reference of one l1 step of the second-order phase (``slm_newton_step_l1``, csrc/newton_kernels.cuh;
``newton_phase(..., w1=...)`` in ``sparselm_b200/newton.py``), one column at a time, in plain numpy.

On the manifold where the signs s_j of the non-zero coordinates are fixed and no active group norm is zero,

    phi(x) = 1/(2n) x'Gx - c'x/n + sum_j w1_j s_j x_j + sum_g w_g ||x_g|| + 1/2 sum_g d_g ||x_g||^2,

a coordinate is active iff x_j != 0.  The step solves H d = -grad on the active coordinates (H as for the pure
group step: the l1 term has no curvature), finds t_cross = min{ -x_j/d_j : x_j d_j < 0 }, backtracks from
min(1, t_cross) with the kernel's difference formulas plus the l1 difference t sum_j w1_j s_j d_j, and stores
the coordinates that reach zero at the accepted t as exact zeros.  Every tried step is recorded with its
Armijo margin (as in ``newton_reference.line_search``) so that a caller can tell a decision rounding could flip.
"""

from __future__ import annotations

import numpy as np

import newton_reference as NR

ARMIJO = NR.ARMIJO
HALVINGS = NR.HALVINGS


def crossings(x, d):
    """Step length at which each coordinate of x + t d reaches zero (inf where it moves away or stays)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(x * d < 0, -x / d, np.inf)


def l1_step(G, p, n, x, w1, w2, d2, gptr):
    """One l1 Newton step of one column.  G Gram (rows/cols < p: X'X, row p: X'y), n rows of the data term,
    x [p] start point, w1 [p] l1 weights, w2 [Gn] group weights (zeros and gptr = [0, p] for Lasso), d2 [Gn] or
    None, gptr [Gn+1].  Returns a dict: act, on, kk, H, grad, gs, d, ok, dec, t_cross, accepted, t (0 when not
    accepted), x_new, zeroed (coordinates set to exactly 0 by the step), trials."""
    gptr = np.asarray(gptr, dtype=np.int64)
    gid = NR.group_ids(gptr)
    Gn = len(gptr) - 1
    x = np.asarray(x, dtype=np.float64)
    w1 = np.asarray(w1, dtype=np.float64)
    w2 = np.asarray(w2, dtype=np.float64)
    nrm = np.sqrt(np.array([np.dot(x[gptr[g]:gptr[g + 1]], x[gptr[g]:gptr[g + 1]]) for g in range(Gn)]))
    on = (nrm > 0)[gid] & (x != 0)
    act = np.flatnonzero(on)
    safe = np.where(nrm > 0, nrm, 1.0)
    u = np.where(on, x / safe[gid], 0.0)
    kk = np.where(on, w2[gid] / safe[gid], 0.0)
    dp = np.where(on, 0.0 if d2 is None else np.asarray(d2)[gid], 0.0)
    gs = np.where(on, (G[:p, :p] @ x - G[p, :p]) / n, 0.0)
    s = np.sign(x)
    grad = np.where(on, gs + (kk + dp) * x + w1 * s, 0.0)
    H = NR.compact_hessian(G, n, act, gid, u, kk, dp)
    d = np.zeros(p)
    ok = True
    if len(act):
        try:
            np.linalg.cholesky(H)
            d[act] = -np.linalg.solve(H, grad[act])
        except np.linalg.LinAlgError:
            ok = False
    # the kernel's sums
    g1 = np.array([np.dot(x[gptr[g]:gptr[g + 1]], d[gptr[g]:gptr[g + 1]]) for g in range(Gn)])
    g2 = np.array([np.dot(d[gptr[g]:gptr[g + 1]], d[gptr[g]:gptr[g + 1]]) for g in range(Gn)])
    q1 = float(gs @ d)
    gd = float(grad @ d)
    r1 = float(np.sum(dp * x * d))
    r2 = float(np.sum(dp * d * d))
    ud = np.array([np.dot(u[gptr[g]:gptr[g + 1]], d[gptr[g]:gptr[g + 1]]) for g in range(Gn)])
    kkg = np.array([kk[gptr[g]:gptr[g + 1]][on[gptr[g]:gptr[g + 1]]].max(initial=0.0) for g in range(Gn)])
    cdd = float(np.sum((kk + dp) * d * d) - np.sum(kkg * ud * ud))
    l1d = float(np.sum(np.where(on, w1 * s * d, 0.0)))
    dec = -gd
    q2 = dec - cdd
    cross = crossings(x, d)
    t_cross = float(cross.min(initial=np.inf))
    usable = ok and dec > 0.0 and np.isfinite(dec)
    t, accepted, trials = min(1.0, t_cross), False, []
    if usable:
        for _ in range(HALVINGS):
            dsq = 2.0 * t * g1 + t * t * g2
            nn = np.sqrt(np.maximum(nrm * nrm + dsq, 0.0))
            terms = w2 * dsq / (nn + safe)
            dphi = t * q1 + 0.5 * t * t * q2 + t * r1 + 0.5 * t * t * r2 + float(np.sum(terms)) + t * l1d
            thr = ARMIJO * t * gd
            size = (abs(t * q1) + 0.5 * t * t * (abs(dec) + abs(cdd)) + abs(t * r1) + 0.5 * t * t * abs(r2)
                    + float(np.sum(np.abs(terms))) + abs(t * l1d) + abs(thr))
            trials.append((t, dphi, thr, size))
            if dphi <= thr:
                accepted = True
                break
            t *= 0.5
    ts = t if accepted else 0.0
    if accepted:
        zeroed = np.flatnonzero(cross <= ts)
        x_new = x + ts * d
        x_new[zeroed] = 0.0
    else:
        zeroed = np.zeros(0, dtype=np.int64)
        x_new = x.copy()
    return dict(act=act, on=on, kk=kk, H=H, grad=grad, gs=gs, d=d, ok=ok, dec=dec, t_cross=t_cross,
                accepted=accepted, t=ts, x_new=x_new, zeroed=zeroed, trials=trials)


def objective_change(G, p, n, x, x_new, w1, w2, d2, gptr):
    """phi(x_new) - phi(x) with the l1 term, formed without cancellation where it matters (s = x_new - x)."""
    x = np.asarray(x, dtype=np.float64)
    x_new = np.asarray(x_new, dtype=np.float64)
    return NR.objective_change(G, p, n, x, x_new, w2, d2, gptr) + float(np.sum(w1 * (np.abs(x_new) - np.abs(x))))

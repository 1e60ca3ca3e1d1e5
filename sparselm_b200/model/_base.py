"""Base class of the engine-backed estimators.

Mirrors the reference's ``CVXRegressor`` (src/sparselm/model/_base.py:69-519):
same constructor arguments, ``fit(X, y, sample_weight=None) -> self``, ``coef_``
/ ``intercept_`` / ``predict`` / ``score``, and the same order of operations in
``fit`` (validate -> preprocess -> hyper-parameter validation -> solve -> set
intercept, _base.py:173-202).  What differs is the solve seam: instead of
building a cvxpy problem (``generate_problem``, _base.py:414-467) and calling
``problem.solve`` (_base.py:512-519) the estimator describes its penalty as a
``ProblemSpec`` and hands it to the CUDA engine, which works on the Gram matrix
of the (centred, weighted) design.

cvxpy-specific surface (``canonicals_``, ``add_constraints``) is not part of the
path and is not provided; ``generate_problem(X, y)`` is kept as "validate and
describe the problem" and returns the ProblemSpec.
"""

from __future__ import annotations

import warnings
from abc import ABCMeta, abstractmethod
from dataclasses import dataclass, field
from numbers import Real

import numpy as np
from sklearn.base import BaseEstimator, RegressorMixin
from sklearn.utils._param_validation import Interval
from sklearn.utils.validation import check_is_fitted, validate_data

from ..engine import PenaltyGrid, get_engine

__all__ = ["EngineRegressor", "CVXRegressor", "ProblemSpec"]


@dataclass
class ProblemSpec:
    """One penalised least-squares problem in solver feature order.

    min_b 1/(2n)||y - X b||^2 + lam1 ||b||_1 + sum_g w2_g ||b_g|| + 1/2 sum_g d2_g ||b_g||^2
    """

    p: int                               # features of X
    pe: int                              # solver features (== p unless overlap expansion)
    lam1: float = 0.0
    col_perm: np.ndarray | None = None   # solver order -> column of X (groups made contiguous)
    ext_idx: np.ndarray | None = None    # overlap: solver feature a duplicates column ext_idx[a]
    gptr: np.ndarray | None = None       # int32 (G+1,)
    gw: np.ndarray | None = None         # (G,) group weights (adaptive update needs them)
    w2: np.ndarray | None = None         # (G,)
    d2: np.ndarray | None = None         # (G,)
    adaptive: dict | None = None         # a1, a2, alpha, eps, tol, max_iter, update_function
    standardize: bool = False            # group norms ||X_g b_g|| (solved in whitened variables)
    std_delta: np.ndarray | None = None  # (G,) ridge of the standardized ridged variant (then d2 is None)
    split: bool = False                  # standardized group norms next to an l1 term: sparselm_b200/split.py
    key: tuple = field(default_factory=tuple)  # structure key: specs with equal keys can be batched

    @property
    def n_groups(self):
        return self.pe if self.gptr is None else len(self.gptr) - 1

    @property
    def strength(self):
        """Scalar penalty strength used to order the columns of a batch: weakly penalised
        problems have the densest iterates, and the row-sparse Gram apply works on chunks of
        adjacent columns, so columns of similar strength should sit together."""
        s = self.__dict__.get("_strength")
        if s is None:
            s = float(self.lam1)
            if self.w2 is not None and len(self.w2):
                s += float(self.w2.sum()) / len(self.w2)
            if self.adaptive is not None:
                s += float(self.adaptive["alpha"])
            self.__dict__["_strength"] = s
        return s


def stack_specs(specs):
    """Columns of one engine batch from specs that share their structure key."""
    s0 = specs[0]
    K = len(specs)
    lam1 = np.array([s.lam1 for s in specs], dtype=float)
    W2 = None if s0.w2 is None else np.stack([s.w2 for s in specs], axis=1)
    D2 = None if s0.d2 is None else np.stack([s.d2 for s in specs], axis=1)
    ad = None
    if s0.adaptive is not None:
        a = s0.adaptive
        ad = dict(
            a1=None if a["a1"] is None else np.array([s.adaptive["a1"] for s in specs], dtype=float),
            a2=None if a["a2"] is None else np.array([s.adaptive["a2"] for s in specs], dtype=float),
            alpha=np.array([s.adaptive["alpha"] for s in specs], dtype=float),
            gw=s0.gw, eps=a["eps"], tol=a["tol"], max_iter=a["max_iter"],
            update_function=a["update_function"],
        )
    assert W2 is None or W2.shape == (s0.n_groups, K)
    return PenaltyGrid(p=s0.pe, lam1=lam1, gptr=s0.gptr, W2=W2, D2=D2, adaptive=ad)


def group_structure(groups, p):
    """(col_perm, gptr, n_groups): labels in np.sort(np.unique()) order
    (reference _lasso.py:248), features permuted so that groups are contiguous."""
    labels = np.asarray(groups)
    _, inv = np.unique(labels, return_inverse=True)
    inv = inv.reshape(-1)
    n_groups = int(inv.max()) + 1 if len(inv) else 0
    order = np.argsort(inv, kind="stable")
    counts = np.bincount(inv, minlength=n_groups)
    gptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    col_perm = None if np.array_equal(order, np.arange(p)) else order.astype(np.int32)
    return col_perm, gptr, n_groups


class EngineRegressor(RegressorMixin, BaseEstimator, metaclass=ABCMeta):
    """Abstract sklearn-compatible regressor solved on the B200 engine.

    Args:
        fit_intercept (bool): estimate an intercept (data centred first).
        copy_X (bool): kept for API compatibility; X is never modified (it is
            copied to the device).
        warm_start (bool): kept for API compatibility (reference _base.py:132).
        solver (str | None): accepted and ignored (there is one solver: the engine).
        solver_options (dict | None): engine options: ``tol`` (relative duality
            gap, default 1e-10), ``max_iter``, ``check_every``, ``floor_rel``,
            ``device``, ``newton`` (second-order phase: None = automatic for pure
            group penalties, True / False forces it, ``"l1"`` also runs it for
            penalties with an l1 term).
    """

    _parameter_constraints: dict = {
        "fit_intercept": ["boolean"],
        "copy_X": ["boolean"],
        "warm_start": ["boolean"],
        "solver": [str, None],
        "solver_options": [dict, None],
    }

    def __init__(self, fit_intercept=False, copy_X=True, warm_start=False, solver=None, solver_options=None):
        self.fit_intercept = fit_intercept
        self.copy_X = copy_X
        self.warm_start = warm_start
        self.solver = solver
        self.solver_options = solver_options

    @classmethod
    def _get_param_names(cls):
        # sklearn re-derives this from inspect.signature on every get_params / set_params /
        # _validate_params call; a grid search re-parametrises one estimator per candidate
        names = cls.__dict__.get("_param_names_cache")
        if names is None:
            names = super()._get_param_names()
            cls._param_names_cache = names
        return names

    # ---- hooks --------------------------------------------------------------
    @abstractmethod
    def _problem_spec(self, n_features: int) -> ProblemSpec:
        """Describe the penalty for the current hyper-parameters."""

    def _validate_hyperparams(self, X, y) -> None:
        """Reference: CVXRegressor._validate_params(X, y) (_base.py:229-245)."""
        only = self.__dict__.get("_validate_only")
        if only:
            # a grid search re-parametrises ONE working estimator per candidate: every parameter was validated
            # for the first candidate, only the grid's own parameters can have changed since
            from sklearn.utils._param_validation import validate_parameter_constraints

            cons = self._parameter_constraints
            validate_parameter_constraints({k: cons[k] for k in only if k in cons},
                                           {k: getattr(self, k) for k in only if k in cons},
                                           caller_name=self.__class__.__name__)
            return
        self._validate_params()  # sklearn: checks _parameter_constraints

    def _engine_options(self):
        opts = dict(self.solver_options) if self.solver_options is not None else {}
        if not isinstance(opts, dict):
            raise TypeError("solver_options must be a dictionary")
        known = {"tol", "max_iter", "check_every", "floor_rel", "device", "newton"}
        nw = opts.get("newton")
        if not (nw is None or isinstance(nw, (bool, np.bool_)) or (isinstance(nw, str) and nw == "l1")):
            raise ValueError(f"solver_options['newton'] must be None, True, False or 'l1', got {nw!r}")
        return {k: v for k, v in opts.items() if k in known}

    # ---- sklearn API ---------------------------------------------------------
    def fit(self, X, y, sample_weight=None):
        """Fit the linear model coefficients on the GPU engine."""
        # finiteness is checked on the device (FoldData.check_finite, raised at the first host sync
        # of the solve) instead of a host pass over X: 50 ms for the 640 MB of a 20000 x 4000 design
        X, y = validate_data(self, X, y, accept_sparse=False, y_numeric=True, multi_output=False,
                             dtype=np.float64, ensure_all_finite=False)
        self._validate_hyperparams(X, y)
        opts = self._engine_options()
        spec = self._problem_spec(X.shape[1])
        engine = get_engine(opts.pop("device", None))
        sw = None
        if sample_weight is not None:
            from sklearn.utils.validation import _check_sample_weight

            sw = _check_sample_weight(sample_weight, X, dtype=np.float64)
        fd = engine.prepare(X, y, None, self.fit_intercept, sw, col_perm=spec.col_perm)
        self._fit_prepared(engine, fd, spec, opts)
        return self

    def _fit_prepared(self, engine, fd, spec, opts, B0=None):
        """Solve on an already prepared (device-resident) design.  B0: optional start point
        (device tensor [pe], solver feature order), e.g. the CV solution of the same
        candidate on one training fold."""
        out = solve_specs(engine, fd, [spec], use_full=True, B0=B0, **opts)
        coef = out["coef"][0, :, 0].cpu().numpy()
        self.coef_ = _to_original_order(coef, spec)
        if self.fit_intercept:
            self.intercept_ = float(out["intercept"][0, 0].item())
        else:
            self.intercept_ = 0.0
        if spec.adaptive is not None:
            self.n_iter_ = int(out["n_pass"][0, 0])
        self.solver_info_ = {
            "gap": float(out["gap"][0, 0]), "objective": float(out["primal"][0, 0]),
            "iterations": int(out["n_iter"][0, 0]), "status": int(out["status"][0, 0]),
        }
        if self.solver_info_["status"] != 0:
            from sklearn.exceptions import ConvergenceWarning

            warnings.warn(
                f"{type(self).__name__}: the engine stopped with status {self.solver_info_['status']} "
                f"(gap {self.solver_info_['gap']:.3e}); raise solver_options['max_iter']",
                ConvergenceWarning,
            )
        return self

    def predict(self, X):
        check_is_fitted(self, "coef_")
        X = validate_data(self, X, accept_sparse=False, reset=False, dtype=np.float64)
        return X @ self.coef_ + self.intercept_

    def generate_problem(self, X, y, preprocess_data=True, sample_weight=None):
        """Validate hyper-parameters against (X, y) and return the problem description
        (the reference builds its cvxpy problem here, _base.py:414-467)."""
        X = np.asarray(X)
        self._validate_hyperparams(X, np.asarray(y))
        self.problem_spec_ = self._problem_spec(X.shape[1])
        return self.problem_spec_

    def __sklearn_tags__(self):
        tags = super().__sklearn_tags__()
        tags.target_tags.required = True
        return tags


# historical name of the base class in the reference
CVXRegressor = EngineRegressor


def _to_original_order(coef_solver, spec: ProblemSpec):
    if spec.col_perm is None:
        return np.ascontiguousarray(coef_solver)
    out = np.empty_like(coef_solver)
    out[spec.col_perm] = coef_solver
    return out


def _empty_like_grid(s0):
    """A zero-column PenaltyGrid with the structure of spec s0 (rank owns no column of a fold)."""
    G = s0.n_groups
    ad = None
    if s0.adaptive is not None:
        a = s0.adaptive
        z = np.zeros(0)
        ad = dict(a1=None if a["a1"] is None else z, a2=None if a["a2"] is None else z, alpha=z, gw=s0.gw,
                  eps=a["eps"], tol=a["tol"], max_iter=a["max_iter"], update_function=a["update_function"])
    return PenaltyGrid(p=s0.pe, lam1=np.zeros(0), gptr=s0.gptr, W2=None if s0.w2 is None else np.zeros((G, 0)),
                       D2=None if s0.d2 is None else np.zeros((G, 0)), adaptive=ad)


SMALL_P = 160  # designs up to this many (expanded) features iterate inside one fused kernel


def solve_specs(engine, fd, specs, use_full=False, tol=1e-10, max_iter=None, check_every=10,
                floor_rel=1e-14, B0=None, newton=None):
    """Solve problems (equal structure keys) on every training Gram of `fd` (or on its
    full Gram when use_full) as one engine batch.  `specs` is either one list (the same
    K problems on every fold) or a list of per-fold lists (sharded grids).

    Returns device tensors in the column order of fd.Xa: coef [F, p, ldz], intercept
    [F, ldz], and numpy [F, ldz] gap / primal / n_iter / status / n_pass.
    """
    torch = engine.torch
    p = fd.p
    G = fd.G_full[None] if use_full else fd.G_train
    F = G.shape[0]
    keys = ["full"] if use_full else list(range(F))
    n_obs = np.array([fd.n_obs(k) for k in keys])
    fold_specs = specs if (len(specs) and isinstance(specs[0], (list, tuple))) else [specs] * F
    assert len(fold_specs) == F
    s0 = next(fs[0] for fs in fold_specs if len(fs))
    memo = {}  # an unsharded search solves the same candidate list on every fold
    grids = []
    for fs in fold_specs:
        if id(fs) not in memo:
            memo[id(fs)] = stack_specs(fs) if len(fs) else _empty_like_grid(s0)
        grids.append(memo[id(fs)])
    Ks = [g.K for g in grids]
    used = [i for i in range(F) if Ks[i] > 0]
    if s0.split:
        # SparseGroupLasso(standardize=True): l1 on b next to ||X_g b_g|| group norms -- method of
        # multipliers around the engine's solves (sparselm_b200/split.py)
        from ..split import solve_split

        res = solve_split(engine, fd, G, keys, n_obs, fold_specs, tol=tol, max_iter=max_iter, check_every=check_every,
                          floor_rel=floor_rel)
        fd.check_finite()
        coef = res["B"]
        if fd.fit_intercept:
            icpt = torch.stack([engine.intercepts(G[f], p, coef[f], Ks[f]) for f in range(F)])
        else:
            icpt = torch.zeros((F, res["ldz"]), dtype=torch.float64, device=engine.device)
        res.update(coef=coef, intercept=icpt)
        return res
    wctx = None
    if s0.ext_idx is not None:  # overlap: solve on the duplicated-column Gram (_lasso.py:461)
        idx_dev = engine.to_device(np.asarray(s0.ext_idx, dtype=np.int32))
        Gs = engine.gram_gather(G, p, idx_dev, s0.pe)
    else:
        Gs = G
    if s0.standardize:
        # group norms ||X_g b_g|| (_lasso.py:249-252) / ||sqrtm(X_g^T X_g + sqrt(delta_g) I) b_g||
        # (:776-789): solve in the whitened variables gamma_g = R_g b_g, ridge folded into the Gram
        gptr = np.arange(s0.pe + 1) if s0.gptr is None else s0.gptr
        dl = s0.std_delta
        gscale = None
        if fd.extra.get("weighted"):  # weights normalised to sum to the row count (_base.py:214)
            rows = np.array([float(fd.n) if k == "full" else float(fd.n_train[k]) for k in keys])
            gscale = rows / n_obs
        Gs, wctx = engine.whiten(Gs, s0.pe, gptr, n_obs, shift=None if dl is None else np.sqrt(dl), ridge=dl,
                                 gscale=gscale)
    # step sizes stay on the device: nothing before the solver's first convergence check
    # synchronises the host, so packing, Gram build and power iterations are enqueued back to back
    if Gs is not G:
        L = engine.lipschitz_device(Gs, s0.pe).clamp_min(1e-300) * engine.to_device(engine.LIPSCHITZ_MARGIN / n_obs)
    else:
        L = fd.lipschitz_dev(engine, keys, used)
    B_start = None
    if B0 is not None and s0.adaptive is None and not s0.standardize:
        ldz0 = max(8, (max(Ks) + 7) // 8 * 8)
        if B0.dim() == 3:  # a start point per (fold, column), solver feature order
            assert tuple(B0.shape) == (F, s0.pe, ldz0), (tuple(B0.shape), (F, s0.pe, ldz0))
            B_start = B0
        else:
            B_start = torch.zeros((F, s0.pe, ldz0), dtype=torch.float64, device=engine.device)
            B_start[0, :, 0] = B0
    if max_iter is None:
        # fused small-design iterations cost ~0.3 us each: ill-conditioned small problems (p > n,
        # vanishing penalties) get the iterations plain accelerated proximal gradient needs
        max_iter = 1000000 if s0.pe <= SMALL_P else 20000
    res = engine.solve(Gs, s0.pe, n_obs, L, grids, B0=B_start, tol=tol, max_iter=max_iter,
                       check_every=check_every, floor_rel=floor_rel, newton=newton)
    fd.check_finite()  # the solve synchronised: the deferred input validation is free here
    B = res["B"]
    ldz = res["ldz"]
    if wctx is not None:  # back to the caller's variables: b_g = R_g^{-1} gamma_g
        B = torch.stack([engine.unwhiten(B[f], wctx, f, s0.pe, Ks[f]) for f in range(F)])
    if s0.ext_idx is not None:  # fold back (_lasso.py:492-501)
        idx = np.asarray(s0.ext_idx)
        order = np.argsort(idx, kind="stable").astype(np.int32)
        inv_ptr = np.concatenate([[0], np.cumsum(np.bincount(idx, minlength=p))]).astype(np.int32)
        ip, ii = engine.to_device(inv_ptr), engine.to_device(order)
        coef = torch.stack([engine.fold_back(B[f], ip, ii, p, Ks[f]) for f in range(F)])
    else:
        coef = B
    if fd.fit_intercept:
        icpt = torch.stack([engine.intercepts(G[f], p, coef[f], Ks[f]) for f in range(F)])
    else:
        icpt = torch.zeros((F, ldz), dtype=torch.float64, device=engine.device)
    res.update(coef=coef, intercept=icpt)
    return res

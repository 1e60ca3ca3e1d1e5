"""Stability selection (Meinshausen & Buehlmann 2010; complementary pairs, Shah & Samworth 2013) on the batched
engine.

How often does feature j enter the model when the fit is repeated on random halves of the rows, along a grid of
penalties?  Every (candidate, subsample) cell is a fit of one structure on its own row subset: the subsample Grams
are built 16 at a time (Engine.split_chunk), all candidates are solved on them as one batch (solve_specs), and the
coefficient tables are reduced to selection counts on the device (slm_support_counts).  Coefficients never leave the
device; per chunk only the solver's convergence info comes back.
"""

from __future__ import annotations

import math
import numbers
import warnings

import numpy as np
from sklearn.base import BaseEstimator, MetaEstimatorMixin
from sklearn.feature_selection import SelectorMixin
from sklearn.model_selection import ParameterGrid
from sklearn.utils import check_random_state
from sklearn.utils.validation import check_is_fitted, check_X_y

from .engine import get_engine
from .model._base import EngineRegressor
from .model_selection import _SolveInfo, describe_candidates, split_batches

__all__ = ["StabilitySelection", "batched_selection", "draw_subsamples", "selection_summary"]


def draw_subsamples(n, n_subsamples, sample_fraction, complementary_pairs, random_state=None):
    """Row subsets of the fits: `n_subsamples` sorted int64 arrays of floor(sample_fraction * n) distinct rows, drawn
    from check_random_state(random_state).  With complementary_pairs (sample_fraction 0.5, n_subsamples even)
    n_subsamples / 2 halves are drawn and each is followed by its complement, which has ceil(n / 2) rows."""
    if not 0.0 < sample_fraction < 1.0:
        raise ValueError(f"sample_fraction must lie in (0, 1), got {sample_fraction!r}")
    if not isinstance(n_subsamples, numbers.Integral) or n_subsamples < 1:
        raise ValueError(f"n_subsamples must be a positive integer, got {n_subsamples!r}")
    if complementary_pairs and (sample_fraction != 0.5 or n_subsamples % 2):
        raise ValueError("complementary_pairs needs sample_fraction == 0.5 and an even n_subsamples")
    m = int(math.floor(sample_fraction * n))
    if m < 2 or (complementary_pairs and n - m < 2):
        raise ValueError(f"a subsample of {n} rows at sample_fraction {sample_fraction} has fewer than two rows")
    rng = check_random_state(random_state)
    out = []
    for _ in range(n_subsamples // 2 if complementary_pairs else n_subsamples):
        rows = np.sort(rng.choice(n, m, replace=False)).astype(np.int64)
        out.append(rows)
        if complementary_pairs:
            keep = np.ones(n, dtype=bool)
            keep[rows] = False
            out.append(np.flatnonzero(keep).astype(np.int64))
    return out


def selection_summary(counts, union, threshold):
    """Stability statistics of n_sub subsample fits: counts [p, n_cand] (fits selecting feature j for candidate c),
    union [n_sub, p] (feature selected by some candidate on that subsample).  Returns (stability_scores [p, n_cand],
    scores [p], q, bound): q is the mean size of the union of the selected sets over the candidates, and bound the
    Meinshausen-Buehlmann bound on the expected number of falsely selected features, q^2 / ((2 threshold - 1) p),
    inf for threshold <= 0.5."""
    union = np.asarray(union, dtype=bool)
    n_sub, p = union.shape
    stability = np.asarray(counts, dtype=np.float64) / float(n_sub)
    q = float(union.sum(axis=1).mean())
    bound = math.inf if threshold <= 0.5 else q * q / ((2.0 * threshold - 1.0) * p)
    return stability, stability.max(axis=1), q, bound


def batched_selection(engine, X, y, subsamples, ests, specs, opts, selection_tol=1e-6, sample_weight=None):
    """Fit every (candidate, subsample) cell and count selections on the device.

    X: (n, p) float64 design; y: (n,); subsamples: row index arrays (distinct rows each); ests/specs: per candidate
    its fit_intercept and ProblemSpec (describe_candidates); opts: solver options; sample_weight: optional strictly
    positive (n,) fit weights.  Candidates of different structure keys run as separate batches.
    Returns counts [p, n_cand] (int64, original feature order: fits that select feature j for candidate c),
    union [n_sub, p] (bool: feature selected by some candidate on that subsample), info {n_iter, status, gap,
    n_pass: [n_cand, n_sub]} and n_unconverged."""
    torch = engine.torch
    yv = np.asarray(y, dtype=np.float64)
    p = X.shape[1]
    # a split whose training rows are the subsample and whose test list is empty
    splits = [(np.asarray(rows, dtype=np.int64), np.zeros(0, dtype=np.int64)) for rows in subsamples]
    n_sub, n_cand = len(splits), len(specs)
    counts = np.zeros((p, n_cand), dtype=np.int64)
    union = np.zeros((n_sub, p), dtype=bool)
    info = _SolveInfo(n_cand, n_sub)
    slot_split = np.empty(n_sub, dtype=np.int64)  # row r of a union table holds subsample slot_split[r]
    unions, perms = {}, {}
    for fkey, _, idxs, chunks in split_batches(engine, X, yv, splits, ests, specs, opts, {},
                                               sample_weight=sample_weight):
        s0 = specs[idxs[0]]
        if fkey not in unions:
            # per column order: the union of one subsample is OR-ed over the batches in Xa column order
            unions[fkey] = torch.zeros((n_sub, p), dtype=torch.uint8, device=engine.device)
            perms[fkey] = s0.col_perm
        K = len(idxs)
        cnt = torch.zeros((p, K), dtype=torch.int32, device=engine.device)
        for c0, order, _, out, _ in chunks:
            c1 = c0 + len(order)
            # the slot order of a chunk depends on the build modes only: the same for every batch
            slot_split[c0:c1] = order
            engine.support_counts(out["coef"], K, selection_tol, cnt, unions[fkey][c0:c1])
            info.record(out, order, [idxs] * len(order))
        c = cnt.cpu().numpy()  # one D2H per batch, in Xa column order
        if s0.col_perm is not None:
            c_orig = np.empty_like(c)
            c_orig[s0.col_perm] = c
            c = c_orig
        counts[:, idxs] = c
    for fkey, u in unions.items():
        u = u.cpu().numpy().astype(bool)
        if perms[fkey] is not None:
            u_orig = np.empty_like(u)
            u_orig[:, perms[fkey]] = u
            u = u_orig
        union[slot_split] |= u
    return dict(counts=counts, union=union, info=info.tables, n_unconverged=info.n_unconverged)


class StabilitySelection(SelectorMixin, MetaEstimatorMixin, BaseEstimator):
    """Stability selection of the features of an engine-backed estimator.

    Every candidate of `param_grid` is fitted on `n_subsamples` random row subsets; feature j is selected in one
    fit iff ``|b_j| > selection_tol * max_k |b_k|`` (an all-zero fit selects nothing).  A feature's stability
    score is its largest selection frequency over the candidates; ``get_support`` / ``transform`` keep the
    features whose score reaches `threshold`.

    Args:
        estimator: an engine estimator with a penalty (Lasso, the group Lassos, their adaptive variants).
        param_grid (dict | list[dict]): candidates, as in GridSearchCV.
        n_subsamples (int): number of subsamples.
        sample_fraction (float): fraction of the rows in a subsample, in (0, 1); a subsample has
            floor(sample_fraction * n) rows.
        complementary_pairs (bool): draw n_subsamples / 2 halves and pair each with its complement (needs
            sample_fraction 0.5 and an even n_subsamples; with an odd n the complement has ceil(n / 2) rows).
        threshold (float): selection frequency in (0, 1] a feature needs to be selected.
        selection_tol (float): relative size below which a coefficient counts as zero.
        random_state: seed of the subsample draws.

    Attributes:
        subsamples_ (list[ndarray]): the row indices of every subsample.
        candidates_ (list[dict]): the candidates, in ParameterGrid order.
        stability_scores_ (ndarray [p, n_candidates]): selection frequency per feature and candidate.
        scores_ (ndarray [p]): stability_scores_.max(axis=1).
        selected_size_ (float): mean over the subsamples of the size of the union of the selected sets over the
            candidates (q_Lambda).
        expected_false_positives_ (float): q_Lambda^2 / ((2 threshold - 1) p), inf for threshold <= 0.5.
        solver_info_ (dict): n_iter, status, gap, n_pass per (candidate, subsample).
        n_features_in_ (int).
    """

    def __init__(self, estimator, param_grid, *, n_subsamples=100, sample_fraction=0.5, complementary_pairs=True,
                 threshold=0.6, selection_tol=1e-6, random_state=None):
        self.estimator = estimator
        self.param_grid = param_grid
        self.n_subsamples = n_subsamples
        self.sample_fraction = sample_fraction
        self.complementary_pairs = complementary_pairs
        self.threshold = threshold
        self.selection_tol = selection_tol
        self.random_state = random_state

    def _check_params(self):
        est = self.estimator
        if not isinstance(est, EngineRegressor) or not getattr(est, "_batchable", True):
            raise ValueError(f"StabilitySelection needs a penalised engine estimator (Lasso, a group Lasso or an "
                             f"adaptive variant), got {type(est).__name__}")
        if not 0.0 < self.threshold <= 1.0:
            raise ValueError(f"threshold must lie in (0, 1], got {self.threshold!r}")
        if not (0.0 <= self.selection_tol < math.inf):
            raise ValueError(f"selection_tol must be finite and >= 0, got {self.selection_tol!r}")

    def fit(self, X, y, sample_weight=None):
        """Draw the subsamples, fit every (candidate, subsample) cell on the GPU and count the selections."""
        self._check_params()
        # finiteness is checked on the device (the Gram of all rows) instead of a host pass over X
        Xv, yv = check_X_y(X, y, dtype=np.float64, y_numeric=True, ensure_min_samples=2, ensure_all_finite=False)
        n, p = Xv.shape
        sw = None
        if sample_weight is not None:
            sw = np.asarray(sample_weight, dtype=np.float64).reshape(-1)
            if sw.shape[0] != n or not np.all(np.isfinite(sw)) or not np.all(sw > 0):
                raise ValueError("sample_weight must hold one finite, strictly positive weight per row")
        subsamples = draw_subsamples(n, self.n_subsamples, self.sample_fraction, self.complementary_pairs,
                                     self.random_state)
        candidates = list(ParameterGrid(self.param_grid))
        valid = set(self.estimator.get_params(deep=False))
        for c in candidates:
            if not set(c) <= valid:
                raise ValueError(f"invalid parameters {sorted(set(c) - valid)} for {type(self.estimator).__name__}")
        ests, specs = describe_candidates(self.estimator, candidates, Xv, yv)
        opts = self.estimator._engine_options()
        engine = get_engine(opts.pop("device", None))
        res = batched_selection(engine, Xv, yv, subsamples, ests, specs, opts, self.selection_tol, sw)
        if res["n_unconverged"]:
            from sklearn.exceptions import ConvergenceWarning

            warnings.warn(f"{res['n_unconverged']} (candidate, subsample) problems did not reach the gap tolerance",
                          ConvergenceWarning)
        self.subsamples_ = subsamples
        self.candidates_ = candidates
        self.stability_scores_, self.scores_, self.selected_size_, self.expected_false_positives_ = \
            selection_summary(res["counts"], res["union"], self.threshold)
        self.solver_info_ = res["info"]
        self.n_features_in_ = p
        return self

    def _get_support_mask(self):
        check_is_fitted(self, "scores_")
        return self.scores_ >= self.threshold

"""Hyper-parameter search: GridSearchCV with the one-standard-error rule and
LineSearchCV (reference: src/sparselm/model_selection.py).

The reference runs ``n_candidates x n_splits`` independent Python fits through
joblib (model_selection.py:304-323), each rebuilding its cvxpy problem.  Here the
whole (candidate, fold) grid of an engine-backed estimator is ONE batch on the
GPU: the per-fold Gram matrices are built once, every candidate is a column of
the batched accelerated proximal-gradient solve, and the CV scores are computed
on the device.  Anything the batched seam does not cover (foreign estimators,
fit params, exotic scorers or splitters) takes sklearn's generic per-fit path,
which still fits on the engine through ``estimator.fit``.

Splits that are not one partition of the rows into at most 15 folds (repeated, shuffled,
leave-one-out, time-series and grouped splitters) are batched too: the full Gram is built once
and the training Grams of at most 16 splits at a time are built from their rows or as a
downdate of the full Gram (``batched_cv_splits``).
"""

from __future__ import annotations

import hashlib
import numbers
import re
import time
import warnings
from copy import deepcopy

import numpy as np
from numpy.ma import MaskedArray
from scipy.stats import rankdata
from sklearn.base import clone
from sklearn.model_selection import GridSearchCV as _SkGridSearchCV
from sklearn.model_selection import ParameterGrid, check_cv
from sklearn.model_selection._search import BaseSearchCV
from sklearn.utils.validation import check_X_y

from .engine import EngineError, get_engine, split_chunks
from .model._base import EngineRegressor, solve_specs

__all__ = ["GridSearchCV", "LineSearchCV"]

# scorers that need a residual statistic beyond the two sums: the row of slm_cv_score_stats' output that holds it
_STAT_ROWS = {"neg_max_error": 2, "neg_mean_absolute_percentage_error": 3, "neg_median_absolute_error": 4}
_DEVICE_SCORERS = {None, "r2", "neg_root_mean_squared_error", "neg_mean_squared_error",
                   "neg_mean_absolute_error", "d2_absolute_error_score"} | set(_STAT_ROWS)
# scorers a sharded search leaves to sklearn's loop: a median of row-sharded residuals needs a residual exchange
_UNSHARDED_SCORERS = set(_STAT_ROWS) | {"d2_absolute_error_score"}


def _stat_mask(metrics):
    """slm_cv_score_stats bit mask of the statistics the metrics {name: scorer} need (0: the two sums suffice)."""
    return sum(1 << r for v, r in _STAT_ROWS.items() if v in set(metrics.values()))


def _abs_dev_median(v):
    """sum |v - median(v)|: the denominator of d2_absolute_error_score (np.median equals sklearn's
    _weighted_percentile(v, 1, 50, average=True))."""
    return float(np.abs(v - np.median(v)).sum()) if len(v) else 0.0


def _device_metrics(scoring):
    """`scoring` as the batched seam understands it: one device scorer name, or a dict
    {metric name: device scorer name} for sklearn's list / tuple / dict multi-metric forms;
    None when some scorer has to run on the host (callables, other metrics)."""
    if scoring is None:
        return "r2"
    if isinstance(scoring, str):
        return scoring if scoring in _DEVICE_SCORERS else None
    if isinstance(scoring, (list, tuple, set)):
        names = list(scoring)
        if not names or len(set(names)) != len(names):
            return None
        scoring = {nm: nm for nm in names}
    if isinstance(scoring, dict) and scoring and all(
            isinstance(k, str) and isinstance(v, str) and v in _DEVICE_SCORERS for k, v in scoring.items()):
        return dict(scoring)
    return None


def _select_best_index_onestd(refit, refit_metric, results):
    """One-standard-error rule (reference model_selection.py:190-223): among the
    candidates whose summed non-negative numeric hyper-parameters are at least those
    of the best-scoring candidate, take the one whose mean score is closest to
    (best mean - its std)."""
    if callable(refit):
        best_index = refit(results)
        if not isinstance(best_index, numbers.Integral):
            raise TypeError("best_index_ returned is not an integer")
        if best_index < 0 or best_index >= len(results["params"]):
            raise IndexError("best_index_ index out of range")
        return best_index
    opt_index = results[f"rank_test_{refit_metric}"].argmin()
    m = results[f"mean_test_{refit_metric}"][opt_index]
    sig = results[f"std_test_{refit_metric}"][opt_index]
    metrics = results[f"mean_test_{refit_metric}"]
    params = []
    for name in [key for key in results if re.match(r"^param_(\w+)", key)]:
        if all(isinstance(val, numbers.Number) for val in results[name]):
            pv = np.array(results[name], dtype=float)
            if np.all(pv > -1e-9):
                params.append(pv)
    params_sum = np.sum(params, axis=0)
    one_std_dists = np.abs(metrics - m + sig)
    candidates = np.arange(len(metrics))[params_sum >= params_sum[opt_index]]
    return candidates[np.argmin(one_std_dists[candidates])]


def _is_partition(splits, n):
    seen = np.zeros(n, dtype=np.int64)
    for train, test in splits:
        seen[test] += 1
        if len(train) + len(test) != n:
            return False
        mask = np.ones(n, dtype=bool)
        mask[test] = False
        if not np.array_equal(np.flatnonzero(mask), np.sort(train)):
            return False
    return bool(np.all(seen == 1))


def _split_route(splits, n, world=1):
    """How a search runs its CV splits: "partition" (one partition of the rows into 2..15 folds: the fold path
    of batched_cv), "splits" (arbitrary row sets: batched_cv_splits) or None (sklearn's per-fit loop: sharded
    searches, an empty test set, fewer than two training rows, a row repeated inside a split)."""
    if 2 <= len(splits) <= 15 and _is_partition(splits, n):
        return "partition"
    if world > 1 or not splits:
        return None
    for train, test in splits:
        tr, te = np.asarray(train), np.asarray(test)
        if len(te) == 0 or len(tr) < 2 or tr.dtype.kind not in "iu" or te.dtype.kind not in "iu":
            return None
        both = np.concatenate([tr, te])
        if both.min() < 0 or both.max() >= n or len(np.unique(both)) != len(both):
            return None
    return "splits"


def _metric(scoring, sse, sae, n_rows, sst, stats=None):
    """Score per column from residual sums (greater is better, sklearn convention).  stats: what the other
    scorers need, {"max", "mape", "median"}: per-column max |r|, sum |r| / max(|y|, eps) and median |r|;
    "sad": sum |y - median(y)| over the scored rows."""
    if scoring == "neg_median_absolute_error":
        return -stats["median"]
    if scoring == "neg_max_error":
        return -stats["max"]
    if scoring == "neg_mean_absolute_percentage_error":
        return -stats["mape"] / n_rows
    if scoring == "d2_absolute_error_score":
        # sklearn's d2_pinball_score(alpha=0.5): NaN on fewer than two rows, force-finite otherwise
        if n_rows < 2:
            from sklearn.exceptions import UndefinedMetricWarning

            warnings.warn("D^2 score is not well-defined with less than two samples.", UndefinedMetricWarning)
            return np.full(np.shape(sae), np.nan)
        sae = np.asarray(sae, dtype=np.float64)
        if stats["sad"] == 0.0:
            return np.where(sae == 0.0, 1.0, 0.0)
        return np.where(sae == 0.0, 1.0, 1.0 - sae / stats["sad"])
    if scoring == "neg_root_mean_squared_error":
        return -np.sqrt(sse / n_rows)
    if scoring == "neg_mean_squared_error":
        return -sse / n_rows
    if scoring == "neg_mean_absolute_error":
        return -sae / n_rows
    # r2 (estimator.score / "r2"), with sklearn's force_finite convention
    if sst == 0.0:
        return np.where(sse == 0.0, 1.0, 0.0)
    return 1.0 - sse / sst


def _split_metric(scoring, sse, sae, n_rows, sst, stats=None):
    """_metric of the arbitrary-split path, with sklearn's rule for r2 on fewer than two rows: NaN and an
    UndefinedMetricWarning (LeaveOneOut with scoring="r2")."""
    if scoring == "r2" and n_rows < 2:
        from sklearn.exceptions import UndefinedMetricWarning

        warnings.warn("R^2 score is not well-defined with less than two samples.", UndefinedMetricWarning)
        return np.full(np.shape(sse), np.nan)
    return _metric(scoring, sse, sae, n_rows, sst, stats)


class _WarmStarts:
    """candidate index -> device view [pe] of its solution on the first training fold that
    solved it (start point of the refit).  The views are made on demand: building one per
    (fold, candidate) eagerly costs more host time than the scoring kernels it delays."""

    def __init__(self):
        self._batches = []

    def add(self, B, idxs, mine):
        self._batches.append((B, np.asarray(idxs), [np.asarray(m) for m in mine]))

    def get(self, ci, default=None):
        for B, idxs, mine in self._batches:
            for f, m in enumerate(mine):
                pos = np.nonzero(idxs[m] == ci)[0] if len(m) else ()
                if len(pos):
                    return B[f, :, int(pos[0])]
        return default

    def __getitem__(self, ci):
        v = self.get(ci)
        if v is None:
            raise KeyError(ci)
        return v


def _fold_key(est, spec):
    return (bool(est.fit_intercept), None if spec.col_perm is None else spec.col_perm.tobytes())


def prepare_folds(engine, X, yv, test_folds, est, spec, cache=None, cache_key=None, shard=None, sample_weight=None):
    """Device-resident design + Grams for (fit_intercept, column order) of `est`/`spec`,
    through the FoldData cache of a LineSearchCV when there is one.  Only enqueues GPU
    work (H2D copies, packing, Gram build): the caller can keep working on the host.
    A sharded rank uploads only its own slice of every fold's rows (Gram build and scoring are both
    row-sharded) when the design comes from the host; a design that is already device-resident, or the
    cached one of a LineSearchCV, is kept whole."""
    ck = None
    if cache is not None and cache_key is not None:
        # keyed on the full content of the split: a shuffling splitter draws a new partition per
        # line, and two partitions can agree in fold sizes and first indices
        fold_hash = hashlib.sha1(np.concatenate([np.asarray(t, dtype=np.int64) for t in test_folds]).tobytes()).hexdigest()
        ck = (cache_key, _fold_key(est, spec), tuple(len(t) for t in test_folds), fold_hash)
        if ck in cache:
            return cache[ck]
    own_rows = (shard is not None and shard.world > 1 and cache is None
                and not (isinstance(X, engine.torch.Tensor) and X.is_cuda))
    fd = engine.prepare(X, yv, test_folds, est.fit_intercept, sample_weight, col_perm=spec.col_perm, shard=shard,
                        own_rows=own_rows)
    if ck is not None:
        cache[ck] = fd
    return fd


def _cache_key(cache, Xv, yv, sw):
    """Data part of the device-data cache key of a LineSearchCV: the identity of X (check_X_y returns the float64 design
    it was given) and the content of y and of the weights (check_X_y returns a new y object at every line)."""
    if cache is None:
        return None
    return (id(Xv), hashlib.sha1(np.ascontiguousarray(yv).tobytes()).hexdigest(),
            None if sw is None else hashlib.sha1(sw.tobytes()).hexdigest())


def prepare_split_data(engine, X, yv, splits, est, spec, cache=None, cache_key=None, sample_weight=None):
    """Device-resident design + full Gram for arbitrary splits (Engine.prepare_splits), through the FoldData
    cache of a LineSearchCV when there is one.  Only enqueues GPU work."""
    ck = None
    if cache is not None and cache_key is not None:
        # keyed on the full content of every split, training and test rows alike: repeated / shuffled splitters
        # can draw new splits per line, and rows in neither set make the test rows alone ambiguous
        h = hashlib.sha1()
        for train, test in splits:
            for a in (train, test):
                a = np.asarray(a, dtype=np.int64)
                h.update(np.int64(len(a)).tobytes())
                h.update(a.tobytes())
        ck = ("splits", cache_key, _fold_key(est, spec), len(splits), h.hexdigest())
        if ck in cache:
            return cache[ck]
    sd = engine.prepare_splits(X, yv, splits, est.fit_intercept, sample_weight, col_perm=spec.col_perm)
    if ck is not None:
        cache[ck] = sd
    return sd


def _stats_of(ext, s, sad):
    """The stats argument of _metric for split s: columns of the [3][n_cand][n_splits] statistics table (or None)."""
    d = {"sad": sad}
    if ext is not None:
        d.update(max=ext[0][:, s], mape=ext[1][:, s], median=ext[2][:, s])
    return d


def candidate_batches(specs):
    """{structure key: candidate indices}: the candidates solved as one batch, in order of increasing penalty strength
    (dense iterates first: the row-sparse apply shares one support list per chunk of adjacent columns)."""
    batches = {}
    for ci, s in enumerate(specs):
        batches.setdefault(s.key, []).append(ci)
    return {k: np.asarray(sorted(v, key=lambda ci: (specs[ci].strength, ci))) for k, v in batches.items()}


class _SolveInfo:
    """Solver info of a search's (candidate, cell) grid: the n_iter / status / gap / n_pass tables [n_cand, n_cells],
    the number of unconverged problems, the iterations run and the Newton-phase totals (engine._run_batch)."""

    def __init__(self, n_cand, n_cells):
        self.tables = dict(n_iter=np.zeros((n_cand, n_cells), dtype=int), status=np.zeros((n_cand, n_cells), dtype=int),
                           gap=np.zeros((n_cand, n_cells)), n_pass=np.zeros((n_cand, n_cells), dtype=int))
        self.n_unconverged, self.iters_run, self.newton = 0, 0, {}

    def record(self, out, cells, cands):
        """Take one solve_specs output whose slot f solved cell cells[f] for the candidates cands[f] (its first
        len(cands[f]) columns)."""
        for f, (c, ci) in enumerate(zip(cells, cands)):
            for k, t in self.tables.items():
                t[ci, c] = out[k][f, :len(ci)]
        self.n_unconverged += int(out["n_unconverged"])
        self.iters_run += int(out["iters_run"])
        for k, v in (out.get("newton") or {}).items():
            self.newton[k] = self.newton.get(k, 0) + v

    def allreduce(self, shard, device, resid):
        """The last exchange of a sharded grid: ONE sum over the ranks of the residual tables `resid` (returned), the
        info tables and n_unconverged.  iters_run and newton stay this rank's."""
        tabs = [resid] + [t.astype(np.float64) for t in self.tables.values()] + [np.array([float(self.n_unconverged)])]
        flat = shard.allreduce_sum_numpy(np.concatenate([t.ravel() for t in tabs]), device)
        o = resid.size
        resid = flat[:o].reshape(resid.shape)
        for k, t in self.tables.items():
            self.tables[k] = flat[o:o + t.size].reshape(t.shape).astype(t.dtype)
            o += t.size
        self.n_unconverged = int(round(float(flat[o])))
        return resid


def _residual_tables(n_cand, n_cells, want_train, stat_mask):
    """Zeroed residual tables of a search: [kind][row][n_cand][n_cells], kind 0 the test rows and 1 the training rows
    (only with train scores); rows Σr², Σ|r| and, when a scorer needs a statistic (stat_mask), max |r|, the
    percentage sum and median |r| (the rows of slm_cv_score_stats)."""
    return np.zeros((2 if want_train else 1, 5 if stat_mask else 2, n_cand, n_cells))


def _split_cells(yv, splits, metrics, want_train):
    """Per split (n_rows, sst, sad) of its test rows and of its training rows (None without train scores): the inputs
    of _scores.  sst and sad are 0.0 where no metric needs them (r2, d2_absolute_error_score)."""
    need_r2 = "r2" in metrics.values()
    need_d2 = "d2_absolute_error_score" in metrics.values()

    def cell(rows):
        v = yv[np.asarray(rows)]
        return (len(v), float(((v - v.mean()) ** 2).sum()) if need_r2 and len(v) else 0.0,
                _abs_dev_median(v) if need_d2 else 0.0)

    return [cell(te) for _, te in splits], [cell(tr) for tr, _ in splits] if want_train else None


def _partition_cells(yv, test_folds, metrics, want_train):
    """_split_cells of a partition: the sst of a fold's training rows is downdated from the sums over all rows,
    q_tr - s_tr^2 / n_tr."""
    need_r2 = "r2" in metrics.values()
    need_d2 = "d2_absolute_error_score" in metrics.values()
    n = len(yv)
    test_cells, train_cells = [], [] if want_train else None
    tot_sum, tot_sq = float(yv.sum()), float((yv * yv).sum())
    for t in test_folds:
        v = yv[t]
        test_cells.append((len(t), float(((v - v.mean()) ** 2).sum()) if need_r2 else 0.0,
                           _abs_dev_median(v) if need_d2 else 0.0))
        if want_train:
            ntr = n - len(t)
            s_tr, q_tr = tot_sum - float(v.sum()), tot_sq - float((v ** 2).sum())
            sad_tr = 0.0
            if need_d2:
                mask = np.ones(n, dtype=bool)
                mask[t] = False
                sad_tr = _abs_dev_median(yv[mask])
            train_cells.append((ntr, q_tr - s_tr * s_tr / ntr, sad_tr))
    return test_cells, train_cells


def _scores(scoring, metric, resid, test_cells, train_cells=None):
    """(test_scores, train_scores) of a search: per metric of `scoring` (one scorer name, or {metric name: scorer
    name}) a table [n_cand, n_cells] formed by `metric` from the residual tables (_residual_tables) and the per-cell
    (n_rows, sst, sad) of the test rows and of the training rows (None: no train scores).  `metric` is _metric on a
    partition and _split_metric on arbitrary splits: they differ in r2 on one row."""
    multi = not isinstance(scoring, str)
    metrics = dict(scoring) if multi else {"score": scoring}
    out = [None, None]
    for kind, cells in enumerate((test_cells, train_cells)[:len(resid)]):
        R = resid[kind]
        tabs = {m: np.empty(R.shape[1:]) for m in metrics}
        for c, (n_rows, sst, sad) in enumerate(cells):
            for m, scorer in metrics.items():
                tabs[m][:, c] = metric(scorer, R[0][:, c], R[1][:, c], n_rows, sst,
                                       _stats_of(R[2:] if len(R) > 2 else None, c, sad))
        out[kind] = tabs if multi else tabs["score"]
    return out


def split_batches(engine, X, yv, splits, ests, specs, opts, sds, cache=None, cache_key=None, sample_weight=None):
    """The (batch, chunk) loop of a search over arbitrary splits.  Per structure key yields (fkey, sd, idxs, chunks):
    the SplitData of the batch's (fit_intercept, column order), prepared on first use into `sds`; the batch's
    candidates (candidate_batches); and a generator that yields per chunk of at most 16 splits (c0, order, fd, out, t):
    the chunk's training Grams (Engine.split_chunk: slot j holds split order[j], c0 the chunk's first split), every
    candidate of the batch solved on them (solve_specs) and the host time the two took.  One [16, pa, pa] buffer
    serves every chunk and batch: a batch's chunks are walked before the next batch is asked for."""
    chunks = split_chunks(len(splits))
    buf = None
    for idxs in candidate_batches(specs).values():
        s0, e0 = specs[idxs[0]], ests[idxs[0]]
        fkey = _fold_key(e0, s0)
        if fkey not in sds:
            sds[fkey] = prepare_split_data(engine, X, yv, splits, e0, s0, cache, cache_key, sample_weight)
        sd = sds[fkey]
        if buf is None:
            buf = engine.torch.empty((chunks[0][1] - chunks[0][0], sd.pa, sd.pa), dtype=engine.torch.float64,
                                     device=engine.device)
        yield fkey, sd, idxs, _solved_chunks(engine, sd, [specs[ci] for ci in idxs], chunks, buf, opts)


def _solved_chunks(engine, sd, bspecs, chunks, buf, opts):
    for c0, c1 in chunks:
        t0 = time.perf_counter()
        order, fd = engine.split_chunk(sd, c0, c1, buf)
        out = solve_specs(engine, fd, bspecs, **opts)
        yield c0, order, fd, out, time.perf_counter() - t0


def batched_cv_splits(engine, X, y, splits, ests, specs, opts, scoring, return_train_score=False, cache=None,
                      cache_key=None, sds=None, sample_weight=None):
    """batched_cv for arbitrary splits (list of (train, test) index arrays, see _split_route): the training Grams of
    at most 16 splits at a time are built (Engine.split_chunk), their Lipschitz constants estimated and every
    candidate solved on them as one batch (solve_specs), then the test lists are scored (slm_cv_score_rows, or
    slm_cv_score_stats when a scorer needs a residual statistic).
    Train scores: a split built from its training rows scores that list; a downdated split scores all rows
    minus the rows outside its training set (the residual sums are additive), or, when a statistic is needed (a
    median does not downdate), the explicit list of its training rows, made for the chunk and dropped after it.
    Returns the same dict as batched_cv; its "fds" hold the refit data (SplitData.full)."""
    yv = np.asarray(y, dtype=np.float64)
    n = yv.shape[0]
    p = X.shape[1]
    n_splits, n_cand = len(splits), len(specs)
    metrics = {"score": scoring} if isinstance(scoring, str) else dict(scoring)
    want_train = bool(return_train_score)
    stat_mask = _stat_mask(metrics)
    resid = _residual_tables(n_cand, n_splits, want_train, stat_mask)
    fit_time = np.zeros(n_cand)
    score_time = np.zeros(n_cand)
    info = _SolveInfo(n_cand, n_splits)
    sds = {} if sds is None else dict(sds)
    warm = _WarmStarts()
    for _, sd, idxs, chunks in split_batches(engine, X, yv, splits, ests, specs, opts, sds, cache, cache_key,
                                             sample_weight):
        K = len(idxs)
        for c0, order, fd, out, t_solve in chunks:
            t1 = time.perf_counter()
            if c0 == 0:
                warm.add(out["B"], idxs, [np.arange(K)] * len(order))
            icpt = (lambda f: out["intercept"][f]) if sd.fit_intercept else (lambda f: None)
            rows_items, rows_where, range_items, range_where = [], [], [], []
            for f, s in enumerate(order):
                rows_items.append((sd.test_rows(s), out["coef"][f], K, icpt(f)))
                rows_where.append((0, s, 1.0))
                if want_train and stat_mask:
                    tr = sd.build_rows(s) if sd.direct[s] else engine.to_device(
                        np.sort(np.asarray(splits[s][0])).astype(np.int32))
                    rows_items.append((tr, out["coef"][f], K, icpt(f)))
                    rows_where.append((1, s, 1.0))
                elif want_train:
                    rows_items.append((sd.build_rows(s), out["coef"][f], K, icpt(f)))
                    if sd.direct[s]:
                        rows_where.append((1, s, 1.0))
                    else:
                        rows_where.append((1, s, -1.0))
                        range_items.append((0, n, out["coef"][f], K, icpt(f)))
                        range_where.append((1, s, 1.0))
            if stat_mask:
                res = engine.cv_score_stats(sd.Xa, p, rows_items, rows_scaled=sd.weighted, stats=stat_mask)
            else:
                res = engine.cv_score_rows(sd.Xa, p, rows_items, rows_scaled=sd.weighted)
            res_r = engine.cv_score_many(sd.Xa, p, range_items, rows_scaled=sd.weighted) if range_items else None
            res = res.cpu().numpy()  # one D2H each
            res_r = None if res_r is None else res_r.cpu().numpy()
            for r, wh in ((res, rows_where), (res_r, range_where)):
                for i, (kind, s, sign) in enumerate(wh):
                    resid[kind][:2, idxs, s] += sign * r[i, :2, :K]
                    if stat_mask:  # one item per split and kind: the statistics are not summed
                        resid[kind][2:, idxs, s] = r[i, 2:5, :K]
            t2 = time.perf_counter()
            info.record(out, order, [idxs] * len(order))
            fit_time[idxs] += t_solve / (K * n_splits)
            score_time[idxs] += (t2 - t1) / (K * n_splits)
    test_scores, train_scores = _scores(scoring, _split_metric, resid, *_split_cells(yv, splits, metrics, want_train))
    return dict(test_scores=test_scores, train_scores=train_scores, fit_time=fit_time, score_time=score_time,
                info=info.tables, fds={k: v.full for k, v in sds.items()}, n_unconverged=info.n_unconverged,
                iters_run=info.iters_run, warm=warm, newton=info.newton)


def batched_cv(engine, X, y, test_folds, ests, specs, opts, scoring, return_train_score=False, cache=None,
               cache_key=None, shard=None, fds=None, sample_weight=None):
    """Solve every (candidate, fold) problem as device batches and score them.

    X: (n, p) numpy array or torch tensor (host, pinned or already on the device);
    y: (n,) numpy array; test_folds: list of index arrays partitioning the rows;
    ests/specs: one configured estimator and its ProblemSpec per candidate.
    shard: optional parallel.GridShard -- this rank builds the Gram of its rows, solves
    its share of the (fold, candidate) grid, and the score tables are summed over ranks.
    sample_weight: optional (n,) strictly positive fit weights, split per fold like the
    reference's fit_params (model_selection.py:266); the scores stay unweighted.
    Returns test_scores [n_cand, n_splits] (+ train scores, timings, solver info and
    the device-resident FoldData objects keyed by (fit_intercept, column order)).
    """
    n, p = X.shape
    n_splits, n_cand = len(test_folds), len(specs)
    yv = np.asarray(y, dtype=np.float64)
    # one scorer name, or {metric name: scorer name}: every device scorer derives from the same
    # two residual sums, so a multi-metric search costs nothing extra on the GPU
    metrics = {"score": scoring} if isinstance(scoring, str) else dict(scoring)
    sharded = shard is not None and shard.world > 1
    want_train = bool(return_train_score)
    stat_mask = _stat_mask(metrics)
    if sharded and (stat_mask or "d2_absolute_error_score" in metrics.values()):
        raise ValueError("a sharded search scores the residual sums only: statistics and d2 need one rank's residuals")
    # residual sums per (candidate, fold) over the test rows (and over the training rows when train scores are asked
    # for).  A sharded search fills in the sums of ITS rows of every fold (scoring is row-sharded like the Gram build)
    # and the tables are summed over the ranks; the metrics are formed from the complete sums afterwards.
    resid = _residual_tables(n_cand, n_splits, want_train, stat_mask)
    fit_time = np.zeros(n_cand)
    score_time = np.zeros(n_cand)
    info = _SolveInfo(n_cand, n_splits)
    # with a statistic, the training rows of fold f are scored as one row list [0, r0_f) + [r1_f, n) of the packed
    # design, made once per call
    train_lists = {}

    fds = {} if fds is None else dict(fds)  # may arrive pre-populated (prepare started early)
    if n_cand and _fold_key(ests[0], specs[0]) not in fds:
        # enqueue the GPU side of the preparation (H2D, packing, Gram build) before the host-side grouping and
        # ordering of the candidates below: that Python work then runs while the GPU is busy
        fds[_fold_key(ests[0], specs[0])] = prepare_folds(engine, X, yv, test_folds, ests[0], specs[0], cache, cache_key,
                                                         shard, sample_weight)
    warm = _WarmStarts()  # candidate -> device view [pe] of its solution on some training fold (refit start)
    for idxs in candidate_batches(specs).values():
        s0, e0 = specs[idxs[0]], ests[idxs[0]]
        fkey = _fold_key(e0, s0)
        K = len(idxs)
        if sharded:
            from .parallel import assign_columns

            owner = assign_columns(n_splits, K, shard.world)  # owner[f][k]: rank that solves column k of fold f
            mine = [np.flatnonzero(owner[f] == shard.rank) for f in range(n_splits)]
        else:
            owner = None
            mine = [np.arange(K)] * n_splits
        if fkey not in fds:
            fds[fkey] = prepare_folds(engine, X, yv, test_folds, e0, s0, cache, cache_key, shard, sample_weight)
        fd = fds[fkey]
        t0 = time.perf_counter()
        out = solve_specs(engine, fd, [[specs[idxs[k]] for k in mine[f]] for f in range(n_splits)], **opts)
        t1 = time.perf_counter()
        warm.add(out["B"], idxs, mine)
        wtd = bool(fd.extra.get("weighted"))
        if not fd.extra.get("partial_folds"):
            # every row is resident: each rank scores the columns it solved on whole folds (a sharded grid then
            # needs no exchange of coefficients; the partial tables are summed with the info tables below).
            # All (fold, row range) problems go through one batched scoring launch.
            icpt = (lambda f: out["intercept"][f]) if fd.fit_intercept else (lambda f: None)
            items, where, titems, twhere = [], [], [], []
            for f in range(n_splits):
                kf = len(mine[f])
                if kf == 0:
                    continue
                ci = idxs[mine[f]]
                items.append((fd.row_ptr[f], fd.row_ptr[f + 1], out["coef"][f], kf, icpt(f)))
                where.append((0, f, ci))
                if want_train and stat_mask:
                    if f not in train_lists:
                        train_lists[f] = engine.to_device(np.concatenate(
                            [np.arange(0, fd.row_ptr[f]), np.arange(fd.row_ptr[f + 1], n)]).astype(np.int32))
                    titems.append((train_lists[f], out["coef"][f], kf, icpt(f)))
                    twhere.append((1, f, ci))
                elif want_train:
                    for r0, r1 in ((0, fd.row_ptr[f]), (fd.row_ptr[f + 1], n)):
                        if r1 > r0:
                            items.append((r0, r1, out["coef"][f], kf, icpt(f)))
                            where.append((1, f, ci))
            if stat_mask:
                for it, wh in ((items, where), (titems, twhere)):
                    if it:
                        res = engine.cv_score_stats(fd.Xa, p, it, rows_scaled=wtd, stats=stat_mask).cpu().numpy()
                        for i, (kind, f, ci) in enumerate(wh):
                            resid[kind][:, ci, f] = res[i][:, :len(ci)]
            elif items:
                res = engine.cv_score_many(fd.Xa, p, items, rows_scaled=wtd).cpu().numpy()  # one D2H
                for i, (kind, f, ci) in enumerate(where):
                    resid[kind][:, ci, f] += res[i][:, :len(ci)]
        else:
            _sharded_residual_sums(engine, shard, fd, out, owner, mine, idxs, resid, wtd)
        t2 = time.perf_counter()
        info.record(out, range(n_splits), [idxs[m] for m in mine])
        fit_time[idxs] = (t1 - t0) / (K * n_splits)
        score_time[idxs] = (t2 - t1) / (K * n_splits)
    if sharded:
        resid = info.allreduce(shard, engine.device, resid)
    test_scores, train_scores = _scores(scoring, _metric, resid, *_partition_cells(yv, test_folds, metrics, want_train))
    return dict(test_scores=test_scores, train_scores=train_scores, fit_time=fit_time, score_time=score_time,
                info=info.tables, fds=fds, n_unconverged=info.n_unconverged, iters_run=info.iters_run, warm=warm,
                newton=info.newton)


def _sharded_residual_sums(engine, shard, fd, out, owner, mine, idxs, resid, wtd):
    """Row-sharded scoring of a sharded grid (north_star: "NCCL all-gather of CV scores and
    coefficients").  Every rank publishes the coefficients (+ intercepts) of the columns it solved,
    ONE all-gather makes all K x n_splits solutions resident everywhere (C3: 10 MB per rank), and each
    rank forms the residual sums of ITS slice of every fold's rows -- the slice it uploaded for the
    Gram build, so a host-resident design crosses the bus once, 1/world per rank.  Adds this rank's
    partial sums of the batch's candidates `idxs` into the residual tables `resid` (test rows, and the
    training rows when resid has them)."""
    import ctypes

    from .parallel import gather_layout, scoring_plan

    torch = engine.torch
    W = shard.world
    p, n_splits = fd.p, len(mine)
    # send layout: [p + 1][ldg], the columns this rank solved, fold after fold (only what was solved travels: C3 on
    # 8 ranks, 2.6 MB per rank)
    kfr, pad, off, ldg = gather_layout(owner, W)
    send = torch.zeros((p + 1, ldg), dtype=torch.float64, device=engine.device)
    for f in range(n_splits):
        kf = len(mine[f])
        if kf:
            o = int(off[shard.rank, f])
            send[:p, o:o + kf] = out["coef"][f][:, :kf]
            if fd.fit_intercept:
                send[p, o:o + kf] = out["intercept"][f][:kf]
    recv = torch.empty((W,) + tuple(send.shape), dtype=torch.float64, device=engine.device)
    comm = shard.comm_ptr(engine.device)
    if comm is not None:
        engine._ck(engine.lib.slm_gather_results(engine.h, ctypes.c_void_p(comm), engine._ptr(send), engine._ptr(recv),
                                                 send.numel(), engine.stream), "slm_gather_results")
    else:
        shard.all_gather_(send, recv)
    # every (fold, solving rank) group against this rank's slice of the fold's rows -- and, for train scores,
    # against its slices of the other folds -- as ONE batched scoring launch
    plan = scoring_plan(owner, shard.fold_row_ranges(fd.row_ptr), W, len(resid) > 1)
    items = []
    for lo, hi, r, f, kind, cols in plan:
        o, kf = int(off[r, f]), len(cols)
        items.append((lo, hi, recv[r, :p, o:o + int(pad[r, f])], kf, recv[r, p, o:o + kf] if fd.fit_intercept else None))
    if items:
        res = engine.cv_score_many(fd.Xa, p, items, rows_scaled=wtd).cpu().numpy()  # one D2H
        for i, (lo, hi, r, f, kind, cols) in enumerate(plan):
            resid[kind][:, idxs[cols], f] += res[i][:, :len(cols)]


def describe_candidates(est, candidates, X, y, on_first=None):
    """(ests, specs) of the candidates (dicts of parameters of `est`) on the design X, y: per candidate a namespace
    holding its fit_intercept and its ProblemSpec.  on_first(ests[0], specs[0]) runs once the first candidate is
    described, before the others (GridSearchCV enqueues its device preparation there)."""
    from types import SimpleNamespace

    p = X.shape[1]
    ests, specs = [], []
    # one working estimator re-parametrised per candidate (cloning 100 estimators and
    # re-deriving their group structure costs more host time than the GPU solve)
    work = clone(est)
    for ci, c in enumerate(candidates):
        work.set_params(**c)
        if ci == 1:
            # from the second candidate on only the grid's own parameters are re-validated, and the
            # group structure memoised for the first candidate is reused without re-hashing `groups`
            # (the working estimator is private to this loop)
            work.__dict__["_validate_only"] = set().union(*[set(cc) for cc in candidates])
            work.__dict__["_groups_frozen"] = True
        with warnings.catch_warnings():
            if ci > 0:  # structural warnings (e.g. groups=None) are emitted once
                warnings.simplefilter("ignore", UserWarning)
            work._validate_hyperparams(X, y)
        ests.append(SimpleNamespace(fit_intercept=bool(work.fit_intercept)))
        specs.append(work._problem_spec(p))
        if ci == 0 and on_first is not None:
            on_first(ests[0], specs[0])
    return ests, specs


class GridSearchCV(_SkGridSearchCV):
    """Exhaustive search over a parameter grid, batched on the GPU for engine-backed
    estimators.  Same constructor as the reference (model_selection.py:160-187):
    sklearn's GridSearchCV plus ``opt_selection_method`` in {"max_score",
    "one_std_score"} and default scoring "neg_root_mean_squared_error"; fitted
    attributes ``best_params_``, ``best_score_``, ``best_score_std_``,
    ``best_estimator_``, ``cv_results_`` (:376-422).
    """

    def __init__(self, estimator, param_grid, *, opt_selection_method="max_score",
                 scoring="neg_root_mean_squared_error", n_jobs=None, refit=True, cv=None, verbose=0,
                 pre_dispatch="2*n_jobs", error_score=np.nan, return_train_score=False):
        super().__init__(estimator=estimator, param_grid=param_grid, scoring=scoring, n_jobs=n_jobs,
                         refit=refit, cv=cv, verbose=verbose, pre_dispatch=pre_dispatch,
                         error_score=error_score, return_train_score=return_train_score)
        self.opt_selection_method = opt_selection_method

    # sklearn calls self._select_best_index(self.refit, refit_metric, results)
    def _select_best_index(self, refit, refit_metric, results):
        if self.opt_selection_method == "max_score":
            return _SkGridSearchCV._select_best_index(refit, refit_metric, results)
        if self.opt_selection_method == "one_std_score":
            return _select_best_index_onestd(refit, refit_metric, results)
        raise NotImplementedError(f"Method {self.opt_selection_method} not implemented!")

    _select_best_index_onestd = staticmethod(_select_best_index_onestd)

    # ------------------------------------------------------------------ #
    def fit(self, X, y=None, **params):
        """Run the search.  Engine-backed estimators with batchable grids are solved as
        one device batch; everything else goes through sklearn's per-fit loop."""
        plan = self._batch_plan(X, y, params)
        if plan is None:
            super().fit(X, y, **params)
            if hasattr(self, "best_index_") and not callable(self.refit):
                self.best_score_std_ = self.cv_results_["std_test_score"][self.best_index_] \
                    if "std_test_score" in self.cv_results_ else None
            self.batched_ = False
            return self
        return self._fit_batched(plan)

    # ------------------------------------------------------------------ #
    def _batch_plan(self, X, y, params):
        est = self.estimator
        if not isinstance(est, EngineRegressor) or y is None or not getattr(est, "_batchable", True):
            return None
        # fit params: only sample_weight is understood by the batched seam (strictly positive:
        # the unweighted CV scores are recovered from the sqrt(sw)-scaled rows); groups only reach the splitter
        sw = groups = None
        for k, v in params.items():
            if v is None:
                continue
            if k == "groups":
                groups = v
            elif k == "sample_weight":
                sw = v
            else:
                return None
        metrics = _device_metrics(self.scoring)
        if metrics is None:
            return None
        shard = getattr(self, "_shard", None)
        if shard is not None and shard.world > 1 and _UNSHARDED_SCORERS & set(
                [metrics] if isinstance(metrics, str) else metrics.values()):
            return None  # DESIGN section 7: statistics of row-sharded residuals are not formed
        if callable(self.refit) or hasattr(X, "columns"):
            return None
        if not isinstance(_device_metrics(self.scoring), str) and self.refit is not False and (
                not isinstance(self.refit, str) or self.refit not in _device_metrics(self.scoring)):
            return None  # sklearn's own loop raises its multi-metric refit error
        if self.opt_selection_method not in ("max_score", "one_std_score"):
            raise NotImplementedError(f"Method {self.opt_selection_method} not implemented!")
        try:
            # finiteness is checked on the device (engine.prepare) instead of a host pass over X
            Xv, yv = check_X_y(X, y, dtype=np.float64, y_numeric=True, ensure_min_samples=2,
                               ensure_all_finite=False)
        except Exception:
            return None
        n, p = Xv.shape
        if sw is not None:
            try:
                sw = np.asarray(sw, dtype=np.float64).reshape(-1)
            except Exception:
                return None
            if sw.shape[0] != n or not np.all(np.isfinite(sw)) or not np.all(sw > 0):
                return None
        cv = check_cv(self.cv, yv, classifier=False)
        try:
            splits = list(cv.split(Xv, yv, groups))
        except Exception:
            return None  # sklearn's loop raises the splitter's own error
        route = _split_route(splits, n, 1 if shard is None else shard.world)
        if route is None:
            return None
        candidates = list(ParameterGrid(self.param_grid))
        valid = set(est.get_params(deep=False))
        if any(not set(c) <= valid for c in candidates):
            return None
        pre_fds = {}
        cache = getattr(self, "_fd_cache", None)
        cache_key = _cache_key(cache, Xv, yv, sw)

        def start_prepare(e0, s0):
            # the design of the first candidate starts its way to the device (H2D, packing,
            # Gram build are only enqueued) while the host describes the other candidates
            opts0 = est._engine_options()
            engine = get_engine(opts0.pop("device", None))
            if route == "splits":
                pre_fds[_fold_key(e0, s0)] = prepare_split_data(engine, Xv, yv, splits, e0, s0, cache, cache_key, sw)
            else:
                pre_fds[_fold_key(e0, s0)] = prepare_folds(engine, Xv, yv, [np.asarray(test) for _, test in splits],
                                                           e0, s0, cache, cache_key, shard, sw)

        try:
            ests, specs = describe_candidates(est, candidates, Xv, yv, on_first=start_prepare)
        except (NotImplementedError, EngineError):
            raise
        except Exception:
            return None  # sklearn's loop applies error_score semantics per candidate
        return dict(X=Xv, y=yv, n=n, p=p, splits=splits, candidates=candidates, ests=ests, specs=specs,
                    fds=pre_fds, sample_weight=sw, route=route, cache_key=cache_key)

    def _fit_batched(self, plan):
        Xv, yv, n, p = plan["X"], plan["y"], plan["n"], plan["p"]
        splits, candidates, specs, ests = plan["splits"], plan["candidates"], plan["specs"], plan["ests"]
        n_splits, n_cand = len(splits), len(candidates)
        base = self.estimator
        opts = base._engine_options()
        engine = get_engine(opts.pop("device", None))
        scoring = _device_metrics(self.scoring)
        multi = not isinstance(scoring, str)
        test_folds = [np.asarray(test) for _, test in splits]
        cache, cache_key = getattr(self, "_fd_cache", None), plan["cache_key"]
        sw = plan.get("sample_weight")
        if plan["route"] == "splits":
            res = batched_cv_splits(engine, Xv, yv, splits, ests, specs, opts, scoring,
                                    return_train_score=self.return_train_score, cache=cache, cache_key=cache_key,
                                    sds=plan.get("fds"), sample_weight=sw)
        else:
            res = batched_cv(engine, Xv, yv, test_folds, ests, specs, opts, scoring,
                             return_train_score=self.return_train_score, cache=cache, cache_key=cache_key,
                             shard=getattr(self, "_shard", None), fds=plan.get("fds"), sample_weight=sw)
        test_scores, train_scores = res["test_scores"], res["train_scores"]
        fit_time, score_time, info, fds = res["fit_time"], res["score_time"], res["info"], res["fds"]
        if res["n_unconverged"]:
            from sklearn.exceptions import ConvergenceWarning

            warnings.warn(f"{res['n_unconverged']} (candidate, fold) problems did not reach the gap tolerance",
                          ConvergenceWarning)

        # ---- cv_results_ in sklearn's layout ------------------------------------------
        results = {}

        def _store(name, arr, splits_=False, rank=False):
            if splits_:
                for i in range(n_splits):
                    results[f"split{i}_{name}"] = arr[:, i]
            mean = arr.mean(axis=1)
            results[f"mean_{name}"] = mean
            results[f"std_{name}"] = np.sqrt(((arr - mean[:, None]) ** 2).mean(axis=1))
            if rank:
                if np.isnan(mean).all():
                    ranks = np.ones_like(mean, dtype=np.int32)
                else:
                    m = np.nan_to_num(mean, nan=np.nanmin(mean) - 1)
                    ranks = rankdata(-m, method="min").astype(np.int32, copy=False)
                results[f"rank_{name}"] = ranks

        _store("fit_time", np.tile(fit_time[:, None], (1, n_splits)))
        _store("score_time", np.tile(score_time[:, None], (1, n_splits)))
        names = sorted({k for c in candidates for k in c})
        for name in names:
            vals = [c.get(name, None) for c in candidates]
            try:
                arr = np.array(vals)
                if arr.ndim != 1 or arr.dtype.kind not in "fiub":
                    raise ValueError
                ma = MaskedArray(arr, mask=[name not in c for c in candidates])
            except Exception:
                ma = MaskedArray(np.empty(n_cand, dtype=object), mask=[name not in c for c in candidates])
                for i, v in enumerate(vals):
                    ma[i] = v
            results[f"param_{name}"] = ma
        results["params"] = candidates
        for m in (scoring if multi else ["score"]):
            _store(f"test_{m}", test_scores[m] if multi else test_scores, splits_=True, rank=True)
            if train_scores is not None:
                _store(f"train_{m}", train_scores[m] if multi else train_scores, splits_=True)

        self.multimetric_ = multi
        refit_metric = self.refit if multi else "score"
        if self.refit or not self.multimetric_:
            self.best_index_ = int(self._select_best_index(self.refit, refit_metric, results))
            self.best_score_ = results[f"mean_test_{refit_metric}"][self.best_index_]
            self.best_score_std_ = results[f"std_test_{refit_metric}"][self.best_index_]
            self.best_params_ = results["params"][self.best_index_]
        if self.refit:
            bi = self.best_index_
            self.best_estimator_ = clone(base).set_params(**clone(self.best_params_, safe=False))
            spec = specs[bi]
            fkey = _fold_key(ests[bi], spec)
            t0 = time.time()
            self.best_estimator_.n_features_in_ = p
            self.best_estimator_._fit_prepared(engine, fds[fkey], spec, dict(opts), B0=res["warm"].get(bi))
            self.refit_time_ = time.time() - t0
        from sklearn.metrics import check_scoring, get_scorer

        self.scorer_ = {m: get_scorer(v) for m, v in scoring.items()} if multi else \
            check_scoring(base, scoring=self.scoring)
        self.cv_results_ = results
        self.n_splits_ = n_splits
        self.solver_info_ = info
        self.batched_ = True
        return self


class LineSearchCV(BaseSearchCV):
    """Coordinate-wise line search over several hyper-parameters
    (reference model_selection.py:427-703): ``n_iter`` successive 1-D grid searches,
    parameter ``i % n_params`` swept while the others stay at their last best value
    (initially the first value of their grid).

    Args:
        estimator: estimator object.
        param_grid (list[tuple[str, list]]): ordered (name, values) pairs.
        opt_selection_method (str | list[str] | None): selection rule per parameter.
        n_iter (int | None): number of line searches; default ``2 * n_params``.
        (remaining arguments as GridSearchCV)
    """

    def __init__(self, estimator, param_grid, *, opt_selection_method=None, n_iter=None,
                 scoring="neg_root_mean_squared_error", n_jobs=None, refit=True, cv=None, verbose=0,
                 pre_dispatch="2*n_jobs", error_score=np.nan, return_train_score=False):
        super().__init__(estimator=estimator, scoring=scoring, n_jobs=n_jobs, refit=refit, cv=cv, verbose=verbose,
                         pre_dispatch=pre_dispatch, error_score=error_score, return_train_score=return_train_score)
        self.param_grid = param_grid
        self.opt_selection_method = opt_selection_method
        self.n_iter = n_iter

    def fit(self, X, y=None, *, groups=None, **fit_params):
        grid = self.param_grid
        if not (isinstance(grid, (list, tuple)) and len(grid) > 0 and isinstance(grid[0], (tuple, list))
                and isinstance(grid[0][0], str)):
            raise ValueError("Parameter grid is not given in the correct format!")
        n_params = len(grid)
        if self.opt_selection_method is None:
            methods = ["max_score"] * n_params
        elif isinstance(self.opt_selection_method, str):
            methods = [self.opt_selection_method] * n_params
        elif (isinstance(self.opt_selection_method, (list, tuple))
              and all(isinstance(m, str) for m in self.opt_selection_method)
              and len(self.opt_selection_method) == n_params):
            methods = list(self.opt_selection_method)
        else:
            raise ValueError(
                "Optimal hyperparams selection methods should be given as a single string, or as a list of "
                "strings with the same amount of parameters!")
        n_iter = self.n_iter if (self.n_iter is not None and self.n_iter > 0) else 2 * n_params

        history = []
        fd_cache = {}  # device-resident design shared by every line (same X, y, folds)
        best = None
        if isinstance(self.estimator, EngineRegressor) and y is not None and not hasattr(X, "columns"):
            # one float64 conversion for all lines: the FoldData cache recognises the design by identity
            try:
                X, y = check_X_y(X, y, dtype=np.float64, y_numeric=True, ensure_min_samples=2, ensure_all_finite=False)
            except Exception:
                pass  # the first GridSearchCV raises the proper error
        for i in range(n_iter):
            pid = i % n_params
            last = [values[0] for _, values in grid] if best is None else [best[name] for name, _ in grid]
            line = {name: (values if j == pid else [last[j]]) for j, (name, values) in enumerate(grid)}
            gs = GridSearchCV(estimator=self.estimator, param_grid=line, opt_selection_method=methods[pid],
                              scoring=self.scoring, n_jobs=self.n_jobs, refit=self.refit, cv=self.cv,
                              verbose=self.verbose, pre_dispatch=self.pre_dispatch, error_score=self.error_score,
                              return_train_score=self.return_train_score)
            gs._fd_cache = fd_cache
            if getattr(self, "_shard", None) is not None:
                gs._shard = self._shard
            if groups is not None:
                fit_params = dict(fit_params, groups=groups)
            gs.fit(X, y, **fit_params)
            best = deepcopy(gs.best_params_)
            history.append(gs)
        for attr in [v for v in vars(history[-1]) if v.endswith("_") and not v.startswith("__")]:
            setattr(self, attr, getattr(history[-1], attr))
        self.history_ = history
        return self

    def _run_search(self, evaluate_candidates):
        """Unused: the search is driven by ``fit``."""
        return

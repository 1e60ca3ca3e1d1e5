"""Host driver of the CUDA engine: owns device memory (torch tensors), streams and
the call sequence into the C ABI (include/sparselm_b200.h).

PyTorch is plumbing here (allocation, H2D/D2H, streams, torch.distributed);
every arithmetic step of the hot path is a kernel of libsparselm_b200.so.  There
is no CPU fallback: constructing an Engine without a CUDA device raises.
"""

from __future__ import annotations

import ctypes
import os
import sys
from dataclasses import dataclass, field

import numpy as np

from . import _lib

__all__ = ["Engine", "PenaltyGrid", "FoldData", "SplitData", "EngineError", "get_engine", "plan_splits", "split_chunks"]


class EngineError(RuntimeError):
    pass


def _round_up(x, m):
    return (x + m - 1) // m * m


@dataclass
class PenaltyGrid:
    """K penalised problems sharing one design (columns of the batch).

    penalty_k(b) = sum_j w1_jk |b_j| + sum_g W2[g,k] ||b_g|| + 1/2 sum_g D2[g,k] ||b_g||^2
    in *solver feature order* (groups contiguous: gptr[g]..gptr[g+1]).
    """

    p: int
    lam1: np.ndarray                      # (K,) l1 weight per column (w1_jk = lam1_k)
    gptr: np.ndarray | None = None        # int32 (G+1,), None => singleton groups
    W2: np.ndarray | None = None          # (G, K)
    D2: np.ndarray | None = None          # (G, K)
    # adaptive re-weighting (None => single pass)
    adaptive: dict | None = None
    # keys: a1 (K,)|None, a2 (K,)|None, alpha (K,), gw (G,)|None, eps, tol, max_iter,
    #       update_function (callable|None)

    @property
    def K(self):
        return int(len(self.lam1))

    @property
    def n_groups(self):
        return self.p if self.gptr is None else int(len(self.gptr) - 1)


@dataclass
class FoldData:
    """Device-resident problem data of one CV search (or one plain fit)."""

    n: int
    p: int
    pa: int
    Xa: object                 # torch [n, pa] augmented design, rows sorted by fold
    row_ptr: np.ndarray        # int64 (F+1,) test-fold row ranges in Xa
    G_train: object            # torch [F, pa, pa] training Grams (centred if fit_intercept)
    G_full: object             # torch [pa, pa] Gram of all rows (centred if fit_intercept)
    n_train: np.ndarray        # (F,)
    fit_intercept: bool
    row_perm: np.ndarray | None = None
    extra: dict = field(default_factory=dict)
    _lam: dict = field(default_factory=dict)   # fold index (or "full") -> lambda_max estimate
    _lam_dev: dict = field(default_factory=dict)  # same, as 0-d device tensors (no host sync)
    G_all: object = None       # torch [F+1, pa, pa]: G_train followed by G_full (same storage)
    _finite: object = None     # device flag of the deferred input check (None once checked)

    def check_finite(self):
        """Deferred input validation (sklearn's ensure_all_finite without a host pass over
        X): the column sums / sum(y) / n row of the full Gram is non-finite iff X, y or the
        weights hold a NaN or an infinity.  Evaluated at the first host sync that follows."""
        if self._finite is not None:
            ok = bool(self._finite.item())
            self._finite = None
            if not ok:
                raise ValueError("Input X, y or sample_weight contains NaN or infinity.")

    @property
    def n_folds(self):
        return len(self.n_train)

    def n_obs(self, which):
        """n of the 1/(2n) data term: rows of the training set (sum of weights if weighted)."""
        if which == "full":
            return float(self.extra.get("n_obs_full", float(self.n)))
        return float(self.extra.get("n_obs_train", self.n_train)[which])

    def lipschitz(self, engine, which):
        """L = LIPSCHITZ_MARGIN x (power-iteration lower bound of lambda_max(G)) / n for the training Gram of fold
        `which` (or "full"), computed on first use (a sharded rank only pays for the Grams it iterates on).  The
        margin covers lambda_max on most spectra, not all (DESIGN section 2 item 3)."""
        keys = list(which) if isinstance(which, (list, tuple, np.ndarray)) else [which]
        missing = [k for k in keys if k not in self._lam]
        if missing:
            ints = sorted(k for k in missing if k != "full")
            # contiguous runs of folds go through one batched power iteration
            runs, start = [], None
            for i, k in enumerate(ints):
                if start is None:
                    start = prev = k
                elif k == prev + 1:
                    prev = k
                else:
                    runs.append((start, prev))
                    start = prev = k
            if start is not None:
                runs.append((start, prev))
            F = self.n_folds
            for a, b in runs:
                if b == F - 1 and self.G_all is not None and "full" not in self._lam:
                    # the full-data Gram (refit) rides along in the same batched power iteration
                    lam = engine.lipschitz(self.G_all[a:F + 1], self.p)
                    self._lam["full"] = float(lam[-1])
                    if "full" in missing:
                        missing.remove("full")
                else:
                    lam = engine.lipschitz(self.G_train[a:b + 1], self.p)
                for j, k in enumerate(range(a, b + 1)):
                    self._lam[k] = float(lam[j])
            if "full" in missing:
                self._lam["full"] = float(engine.lipschitz(self.G_full[None], self.p)[0])
        out = np.array([max(self._lam[k], 1e-300) * engine.LIPSCHITZ_MARGIN / self.n_obs(k) for k in keys])
        return out if isinstance(which, (list, tuple, np.ndarray)) else float(out[0])

    def lipschitz_dev(self, engine, keys, used):
        """Device tensor [len(keys)] of L (as `lipschitz`) for the Grams `keys`
        (training folds or "full"); entries of keys not listed in `used` are 1.  Nothing
        here synchronises the host: the power iterations are only enqueued and their
        results stay on the device (cached per Gram for later searches on the same data)."""
        torch = engine.torch
        need = [keys[i] for i in used if keys[i] not in self._lam_dev]
        ints = sorted(k for k in need if k != "full")
        F = self.n_folds
        runs, start = [], None
        for k in ints:
            if start is None:
                start = prev = k
            elif k == prev + 1:
                prev = k
            else:
                runs.append((start, prev))
                start = prev = k
        if start is not None:
            runs.append((start, prev))
        want_full = "full" in need
        for a, b in runs:
            if b == F - 1 and self.G_all is not None and "full" not in self._lam_dev:
                lam = engine.lipschitz_device(self.G_all[a:F + 1], self.p)  # the refit Gram rides along
                self._lam_dev["full"] = lam[-1]
                want_full = False
            else:
                lam = engine.lipschitz_device(self.G_train[a:b + 1], self.p)
            for j, k in enumerate(range(a, b + 1)):
                self._lam_dev[k] = lam[j]
        if want_full:
            self._lam_dev["full"] = engine.lipschitz_device(self.G_full[None], self.p)[0]
        scale = np.ones(len(keys))
        parts = []
        one = None
        for i, k in enumerate(keys):
            if i in used:
                parts.append(self._lam_dev[k])
                scale[i] = engine.LIPSCHITZ_MARGIN / self.n_obs(k)
            else:
                if one is None:
                    one = torch.ones((), dtype=torch.float64, device=engine.device)
                parts.append(one)
        return torch.stack(parts).clamp_min(1e-300) * engine.to_device(scale)


@dataclass
class SplitData:
    """Device-resident problem data of a CV search whose splits are arbitrary row sets (not one
    partition of the rows): repeated / shuffled splits, leave-one-out, time-series and grouped splits.

    The training Grams are not kept: Engine.split_chunk builds those of at most SLM_MAX_FOLDS splits at
    a time, so memory stays O(SLM_MAX_FOLDS pa^2) whatever the number of splits.  Split s is built
    either directly from its training rows (direct[s]) or as a downdate of the full Gram by the rows
    outside its training set (test rows and rows in neither set), whichever list is shorter; only
    that list is stored, in one CSR array per mode (splits in order)."""

    n: int
    p: int
    pa: int
    Xa: object                 # torch [n, pa] augmented design, original row order
    G_raw: object              # torch [pa, pa] uncentred Gram of all rows
    full: FoldData             # refit data: G_full = the full Gram, centred if fit_intercept
    direct: np.ndarray         # bool (S,): build split s from its training rows (else downdate)
    direct_ptr: np.ndarray     # int64 CSR offsets into direct_dev, over the direct splits in order
    direct_dev: object         # torch int32: training rows of the direct splits
    out_ptr: np.ndarray        # int64 CSR offsets into out_dev, over the downdate splits in order
    out_dev: object            # torch int32: rows outside the training set of the downdate splits
    test_ptr: np.ndarray       # int64 (S+1,) CSR offsets into test_dev
    test_dev: object           # torch int32: test rows of every split
    n_obs: np.ndarray          # (S,) n of the 1/(2n) data term: training rows, or sum of their weights
    n_train: np.ndarray        # (S,) training rows
    fit_intercept: bool
    weighted: bool

    @property
    def n_splits(self):
        return len(self.direct)

    def test_rows(self, s):
        """Device int32 view of the test rows of split s."""
        return self.test_dev[int(self.test_ptr[s]):int(self.test_ptr[s + 1])]

    def build_rows(self, s):
        """Device int32 view of the list split s is built from: its training rows (direct) or the rows
        outside its training set (downdate)."""
        j = int(np.count_nonzero(self.direct[:s]))
        if self.direct[s]:
            return self.direct_dev[int(self.direct_ptr[j]):int(self.direct_ptr[j + 1])]
        k = s - j
        return self.out_dev[int(self.out_ptr[k]):int(self.out_ptr[k + 1])]


def split_chunks(n_splits):
    """[s0, s1) ranges of at most SLM_MAX_FOLDS splits: the unit of the Gram build and of the solve."""
    return [(s0, min(n_splits, s0 + _lib.SLM_MAX_FOLDS)) for s0 in range(0, n_splits, _lib.SLM_MAX_FOLDS)]


def plan_splits(splits, n, sample_weight=None):
    """Host side of Engine.prepare_splits: per split its build mode and the one row list that mode
    needs, the test lists and n_obs.  splits: (train, test) index arrays, each without repeated rows.
    Returns a dict of numpy arrays (CSR lists as int32 values and int64 offsets)."""
    direct, dl, ol, tl, n_obs, n_train = [], [], [], [], [], []
    for train, test in splits:
        tr = np.sort(np.asarray(train, dtype=np.int64))
        te = np.sort(np.asarray(test, dtype=np.int64))
        if len(tr) and (tr[0] < 0 or tr[-1] >= n) or len(te) and (te[0] < 0 or te[-1] >= n):
            raise ValueError("split indices out of range")
        if np.any(np.diff(tr) == 0) or np.any(np.diff(te) == 0):
            raise ValueError("a split repeats a row")
        d = len(tr) <= n - len(tr)  # the training rows are at most as many as the rows outside them
        direct.append(d)
        if d:
            dl.append(tr)
        else:
            keep = np.ones(n, dtype=bool)
            keep[tr] = False
            ol.append(np.flatnonzero(keep))
        tl.append(te)
        n_train.append(float(len(tr)))
        n_obs.append(float(len(tr)) if sample_weight is None else float(np.asarray(sample_weight, dtype=np.float64)[tr].sum()))

    def csr(lists):
        ptr = np.concatenate([[0], np.cumsum([len(v) for v in lists])]).astype(np.int64)
        vals = np.concatenate(lists).astype(np.int32) if lists else np.zeros(0, dtype=np.int32)
        return ptr, vals

    dptr, dvals = csr(dl)
    optr, ovals = csr(ol)
    tptr, tvals = csr(tl)
    return dict(direct=np.array(direct, dtype=bool), direct_ptr=dptr, direct_rows=dvals, out_ptr=optr, out_rows=ovals,
                test_ptr=tptr, test_rows=tvals, n_obs=np.array(n_obs), n_train=np.array(n_train))


class Engine:
    # 12 block power iterations reach >= 0.93 lambda_max on flat (Marchenko-Pastur) spectra;
    # the margin turns the lower bound into a safe step size (tests/test_gpu_engine.py)
    LIPSCHITZ_ITERS = 12
    PIPELINE_BLOCK_BYTES = 64 << 20  # rows of a host design travel and enter the Gram in blocks of this size
    LIPSCHITZ_MARGIN = 1.10
    # second-order phase (_run_batch): iterations before the first Newton phase / between two phases
    # (measured on BASELINE configs[3], profiles/r02o_newton_tuning.txt: 500/200 469 ms, 300/200 430 ms, 300/100 422 ms,
    # 200/100 457 ms per search)
    NEWTON_FIRST = 300
    NEWTON_LATER = 100
    # an l1 phase that removed coordinates from a column's support counts as progress, not as one of the three failed
    # phases after which the column stays first-order: a truncated step drops about one coordinate, so a support with
    # many spurious coordinates needs several phases (profiles/r03_newton_l1_probe.jsonl: with / without this rule)
    NEWTON_L1_SHRINK_IS_PROGRESS = True

    def __init__(self, device: int | None = None):
        import torch

        if not torch.cuda.is_available():
            raise EngineError(
                "sparselm_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback"
            )
        self.torch = torch
        self.lib = _lib.load()
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        h = ctypes.c_void_p()
        rc = self.lib.slm_create(self.device_index, ctypes.byref(h))
        if rc != 0:
            raise EngineError(f"slm_create failed with code {rc}")
        self.h = h
        self.sm_count = self.lib.slm_sm_count(self.h)

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.slm_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ---- helpers ---------------------------------------------------------
    def _ck(self, rc, what):
        if rc != 0:
            msg = self.lib.slm_last_error(self.h)
            raise EngineError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    @property
    def stream(self):
        return ctypes.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    @staticmethod
    def _ptr(t):
        return ctypes.c_void_p(0 if t is None else t.data_ptr())

    def to_device(self, a, dtype=None):
        """numpy / torch (cpu, pinned or cuda) -> contiguous cuda tensor."""
        torch = self.torch
        if isinstance(a, torch.Tensor):
            t = a
        else:
            t = torch.from_numpy(np.ascontiguousarray(a))
            if t.numel() * t.element_size() <= (8 << 20):
                # small host arrays (penalty tables, y, index lists) are staged through torch's
                # cached pinned pool so that the upload is asynchronous: a pageable H2D copy
                # would stall the host until the GPU has drained the stream
                if dtype is not None and t.dtype != dtype:
                    t = t.to(dtype)
                t = t.pin_memory()
        if dtype is not None and t.dtype != dtype:
            t = t.to(dtype)
        if t.device != self.device:
            t = t.to(self.device, non_blocking=True)
        return t.contiguous()

    def set_option(self, name, value):
        """Engine switch by name ("coop", "tma", "fused_prox", "force_apply_shape", "force_sparse_shape",
        "force_syrk_shape", "force_score_shape").  The force_* options pin a tile of the GEMM menus:
        -1 = automatic, an id past the menu raises EngineError."""
        self._ck(self.lib.slm_set_option(self.h, name.encode(), int(value)), "slm_set_option")

    def launch_count(self):
        return int(self.lib.slm_launch_count(self.h))

    def tma_launch_count(self):
        """TMA-fed GEMM launches (gemm_f64_tma_kernel) among them."""
        return int(self.lib.slm_tma_launch_count(self.h))

    def tma_probe(self, A, col0, row0, rows4):
        """Raw shared-memory images of one tiled box load and one 4-row gather (diagnostic)."""
        torch = self.torch
        out = torch.empty(320, dtype=torch.float64, device=self.device)
        r4 = (ctypes.c_int32 * 4)(*[int(r) for r in rows4])
        self._ck(self.lib.slm_tma_probe(self.h, self._ptr(A), A.shape[0], A.shape[1], int(col0), int(row0), r4,
                                        self._ptr(out), self.stream), "slm_tma_probe")
        return out

    def timing_enable(self, on=True):
        self.lib.slm_timing_enable(self.h, 1 if on else 0)

    def timing_reset(self):
        self.lib.slm_timing_reset(self.h)

    def timing_read(self):
        names = ["gram_build", "gram_apply", "prox", "gap", "score", "lipschitz_apply"]
        out = {}
        for i, nm in enumerate(names):
            ms, n, fl = ctypes.c_double(), ctypes.c_int64(), ctypes.c_double()
            self.lib.slm_timing_read(self.h, i, ctypes.byref(ms), ctypes.byref(n), ctypes.byref(fl))
            out[nm] = {"ms": ms.value, "launches": n.value, "flops": fl.value}
        return out

    # ---- K1: pack + Gram ---------------------------------------------------
    def padded_cols(self, p):
        return int(self.lib.slm_padded_cols(p))

    def pack(self, X, y, sample_weight=None, col_perm=None, row_perm=None):
        torch = self.torch
        Xd = self.to_device(X, torch.float64)
        yd = self.to_device(y, torch.float64).reshape(-1)
        n, p = Xd.shape
        pa = self.padded_cols(p)
        Xa = torch.empty((n, pa), dtype=torch.float64, device=self.device)
        sw = None if sample_weight is None else self.to_device(sample_weight, torch.float64)
        cp = None if col_perm is None else self.to_device(np.asarray(col_perm, dtype=np.int32))
        rp = None if row_perm is None else self.to_device(np.asarray(row_perm, dtype=np.int64))
        self._ck(self.lib.slm_pack_design(self.h, self._ptr(Xd), Xd.stride(0), self._ptr(yd), self._ptr(sw),
                                          self._ptr(cp), self._ptr(rp), n, p, self._ptr(Xa), pa, self.stream),
                 "slm_pack_design")
        return Xa

    def gram_blocks(self, Xa, row_ptr, extra=0, zero=False):
        """[F(+extra), pa, pa]: block f = Xa[rows_f]^T Xa[rows_f]; `extra` spare slots.
        Empty row ranges leave their block untouched (zero=True pre-clears the array)."""
        torch = self.torch
        row_ptr = np.ascontiguousarray(row_ptr, dtype=np.int64)
        F = len(row_ptr) - 1
        pa = Xa.shape[1]
        alloc = torch.zeros if zero else torch.empty
        G = alloc((F + extra, pa, pa), dtype=torch.float64, device=self.device)
        self._ck(self.lib.slm_gram_blocks(self.h, self._ptr(Xa), pa,
                                          row_ptr.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), F,
                                          self._ptr(G), self.stream), "slm_gram_blocks")
        return G

    def gram_complement(self, Gblk, F=None, out=None):
        """In place: blocks -> complements (training Grams); returns the total."""
        torch = self.torch
        pa = Gblk.shape[-1]
        F = Gblk.shape[0] if F is None else F
        Gtot = torch.empty((pa, pa), dtype=torch.float64, device=self.device) if out is None else out
        self._ck(self.lib.slm_gram_complement(self.h, self._ptr(Gblk), F, pa, self._ptr(Gtot), self.stream),
                 "slm_gram_complement")
        return Gtot

    def gram_center(self, G, p):
        pa = G.shape[-1]
        Gs = G.reshape(-1, pa, pa)
        for f in range(Gs.shape[0]):
            self._ck(self.lib.slm_gram_center(self.h, self._ptr(Gs[f]), pa, p, self.stream), "slm_gram_center")

    def gram_gather(self, G, p, idx_dev, pe):
        torch = self.torch
        pa = G.shape[-1]
        pae = self.padded_cols(pe)
        Gs = G.reshape(-1, pa, pa)
        out = torch.empty((Gs.shape[0], pae, pae), dtype=torch.float64, device=self.device)
        for f in range(Gs.shape[0]):
            self._ck(self.lib.slm_gram_gather(self.h, self._ptr(Gs[f]), pa, p, self._ptr(idx_dev), pe,
                                              self._ptr(out[f]), pae, self.stream), "slm_gram_gather")
        return out

    def lipschitz(self, G, p, iters=None):
        """lambda_max of each Gram's leading p x p block (lower bound, no margin)."""
        torch = self.torch
        pa = G.shape[-1]
        Gs = G.reshape(-1, pa, pa)
        F = Gs.shape[0]
        out = np.zeros(F)
        iters = self.LIPSCHITZ_ITERS if iters is None else iters
        for f0 in range(0, F, _lib.SLM_MAX_FOLDS):
            nf = min(F - f0, _lib.SLM_MAX_FOLDS)
            nbytes = self.lib.slm_lipschitz_workspace(p, nf)
            work = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            lam = (ctypes.c_double * nf)()
            self._ck(self.lib.slm_lipschitz(self.h, self._ptr(Gs[f0]), pa * pa, pa, p, nf, iters,
                                            self._ptr(work), lam, self.stream), "slm_lipschitz")
            out[f0:f0 + nf] = np.frombuffer(lam, dtype=np.float64, count=nf)
        return out

    def lipschitz_device(self, G, p, iters=None):
        """Same estimate, left on the device ([F] tensor) without synchronising the host."""
        torch = self.torch
        pa = G.shape[-1]
        Gs = G.reshape(-1, pa, pa)
        F = Gs.shape[0]
        out = torch.empty(F, dtype=torch.float64, device=self.device)
        iters = self.LIPSCHITZ_ITERS if iters is None else iters
        for f0 in range(0, F, _lib.SLM_MAX_FOLDS):
            nf = min(F - f0, _lib.SLM_MAX_FOLDS)
            nbytes = self.lib.slm_lipschitz_workspace(p, nf)
            work = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
            self._ck(self.lib.slm_lipschitz_dev(self.h, self._ptr(Gs[f0]), pa * pa, pa, p, nf, iters,
                                                self._ptr(work), ctypes.c_void_p(out.data_ptr() + 8 * f0),
                                                self.stream), "slm_lipschitz_dev")
        return out

    def gram_apply(self, G, p, K, Z):
        """GZ_f = G_f Z_f (tests / roofline)."""
        torch = self.torch
        pa = G.shape[-1]
        Gs = G.reshape(-1, pa, pa)
        F = Gs.shape[0]
        ldz = Z.shape[-1]
        GZ = torch.zeros_like(Z)
        Karr = (ctypes.c_int32 * F)(*[int(k) for k in K])
        self._ck(self.lib.slm_gram_apply(self.h, self._ptr(Gs), pa * pa, pa, p, F, Karr, self._ptr(Z), ldz,
                                         self._ptr(GZ), self.stream), "slm_gram_apply")
        return GZ

    def gram_cg(self, G, p, tol=1e-13, max_iter=None, shift=None):
        """Least-squares coefficients of ONE Gram G [pa, pa]: conjugate gradients on
        (G + diag(shift)) b = c (c = row p), products on the tensor-core apply.  Returns
        (X8, iters, relres): X8 is [p, 8] with the solution in column 0."""
        torch = self.torch
        pa = G.shape[-1]
        if max_iter is None:
            max_iter = 10 * int(p) + 100
        nbytes = self.lib.slm_gram_cg_workspace(p)
        work = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        X8 = torch.empty((p, 8), dtype=torch.float64, device=self.device)
        iters, rel = ctypes.c_int32(0), ctypes.c_double(0.0)
        self._ck(self.lib.slm_gram_cg(self.h, self._ptr(G), pa, p, self._ptr(shift), float(tol), int(max_iter),
                                      self._ptr(work), nbytes,
                                      self._ptr(X8), ctypes.byref(iters), ctypes.byref(rel), self.stream),
                 "slm_gram_cg")
        return X8, int(iters.value), float(rel.value)

    def gram_apply_rowsparse(self, G, p, K, Z, chunk_w=32):
        """The same product through the solver's row-sparse path (support lists per chunk of
        `chunk_w` columns are built on the device from Z)."""
        torch = self.torch
        pa = G.shape[-1]
        Gs = G.reshape(-1, pa, pa)
        F = Gs.shape[0]
        ldz = Z.shape[-1]
        GZ = torch.zeros_like(Z)
        Karr = (ctypes.c_int32 * F)(*[int(k) for k in K])
        nbytes = self.lib.slm_rowsparse_workspace(p, ldz, F)
        work = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._ck(self.lib.slm_gram_apply_rowsparse(self.h, self._ptr(Gs), pa * pa, pa, p, F, Karr, self._ptr(Z), ldz,
                                                   self._ptr(GZ), int(chunk_w), self._ptr(work), nbytes,
                                                   self.stream), "slm_gram_apply_rowsparse")
        return GZ

    def apply_stats(self):
        """(executed, dense-equivalent) flops of the solver's Gram applies since timing_reset."""
        ex, de = ctypes.c_double(), ctypes.c_double()
        self.lib.slm_apply_stats(self.h, ctypes.byref(ex), ctypes.byref(de))
        return ex.value, de.value

    # ---- data preparation for a CV search / a plain fit --------------------
    def prepare(self, X, y, test_folds=None, fit_intercept=False, sample_weight=None, col_perm=None, shard=None,
                own_rows=False):
        """Pack the design, build per-fold training Grams + the full Gram.

        test_folds: list of index arrays forming a partition of range(n) (the CV
        test sets), or None for a single fit on all rows.
        own_rows: (sharded searches on a host-resident X) bring only this rank's slice of
        every test fold's rows to the device, the rows its share of the Gram build and of the
        scoring needs.  False = every row.
        """
        if isinstance(X, self.torch.Tensor):
            n, p = X.shape
        else:
            X = np.asarray(X)
            n, p = X.shape
        row_perm = None
        if test_folds is None:
            row_ptr = np.array([0, n], dtype=np.int64)
        else:
            sizes = [len(t) for t in test_folds]
            row_ptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
            perm = np.concatenate([np.asarray(t, dtype=np.int64) for t in test_folds])
            ident = np.arange(n)
            if len(perm) != n:
                raise ValueError("test_folds must partition the rows")
            if not np.array_equal(perm, ident):  # KFold without shuffling is the identity: no sort needed
                if not np.array_equal(np.sort(perm), ident):
                    raise ValueError("test_folds must partition the rows")
                row_perm = perm
        sw = None
        if sample_weight is not None:
            sw = np.asarray(sample_weight, dtype=np.float64)
        F = len(row_ptr) - 1
        sharded = shard is not None and shard.world > 1
        on_host = not (isinstance(X, self.torch.Tensor) and X.is_cuda)
        # rows of every test fold whose Gram block this rank builds (all of them unless sharded)
        fold_rows = shard.fold_row_ranges(row_ptr) if sharded else \
            [(int(row_ptr[f]), int(row_ptr[f + 1])) for f in range(F)]
        partial = False  # did the prepare routine leave the rows of other ranks unpacked?
        self._complemented = False  # set by the sharded reduce when it already produced training Grams + total
        if on_host and row_perm is None and n >= 4096:
            Xa, allG, partial = self._prepare_pipelined(X, y, sw, col_perm, row_ptr, fold_rows,
                                                        shard if sharded else None, own_rows and sharded)
        elif sharded:
            Xa, allG, partial = self._prepare_sharded(X, y, sw, col_perm, row_perm, row_ptr, fold_rows, shard,
                                                      own_rows)
        else:
            Xa = self.pack(X, y, sw, col_perm, row_perm)
            allG = self.gram_blocks(Xa, row_ptr, extra=1 if F > 1 else 0)
        pa = Xa.shape[1]
        if F > 1:
            G_train, G_full = allG[:F], allG[F]
            if not self._complemented:
                self.gram_complement(allG, F, out=G_full)  # blocks -> training Grams
            n_train = (n - np.diff(row_ptr)).astype(np.float64)
        else:
            G_full = allG[0]
            G_train = allG[:0]
            n_train = np.zeros(0)
        extra = {}
        if sw is not None:
            # reference: weights are rescaled to sum to n (_base.py:214), i.e. the data term is
            # 1/(2 sum(sw)) sum_i sw_i r_i^2 -- the "n" of a weighted problem is sum(sw) of its rows
            swp = sw if row_perm is None else sw[row_perm]
            tot = float(sw.sum())
            extra["n_obs_full"] = tot
            if F > 1:
                extra["n_obs_train"] = tot - np.add.reduceat(swp, row_ptr[:-1])
            extra["weighted"] = True
        if fit_intercept:
            self.gram_center(G_full, p)
            if F > 1:
                self.gram_center(G_train, p)
        if partial:
            # only this rank's slice of every fold's rows reached the device
            extra["partial_folds"] = True
        finite = self.torch.isfinite(G_full[p + 1]).all()  # checked at the next host sync
        return FoldData(n=n, p=p, pa=pa, Xa=Xa, row_ptr=row_ptr, G_train=G_train, G_full=G_full,
                        n_train=n_train, fit_intercept=bool(fit_intercept), row_perm=row_perm, extra=extra,
                        G_all=allG if F > 1 else None, _finite=finite)

    def prepare_splits(self, X, y, splits, fit_intercept=False, sample_weight=None, col_perm=None):
        """Pack the design in its original row order and build the full Gram, for a CV search over
        arbitrary splits (list of (train, test) index arrays, no row repeated inside a split).  The
        training Grams are built chunk by chunk later (split_chunk).  Returns a SplitData."""
        torch = self.torch
        if isinstance(X, torch.Tensor):
            n, p = X.shape
        else:
            X = np.asarray(X)
            n, p = X.shape
        sw = None if sample_weight is None else np.asarray(sample_weight, dtype=np.float64)
        plan = plan_splits(splits, n, sw)
        row_ptr = np.array([0, n], dtype=np.int64)
        if not (isinstance(X, torch.Tensor) and X.is_cuda) and n >= 4096:
            Xa, allG, _ = self._prepare_pipelined(X, y, sw, col_perm, row_ptr, [(0, n)])
        else:
            Xa = self.pack(X, y, sw, col_perm)
            allG = self.gram_blocks(Xa, row_ptr)
        G_raw = allG[0]
        G_full = G_raw
        if fit_intercept:
            G_full = G_raw.clone()
            self.gram_center(G_full, p)
        extra = {"n_obs_full": float(sw.sum()), "weighted": True} if sw is not None else {}
        finite = torch.isfinite(G_raw[p + 1]).all()  # checked at the next host sync
        full = FoldData(n=n, p=p, pa=Xa.shape[1], Xa=Xa, row_ptr=row_ptr, G_train=allG[:0], G_full=G_full,
                        n_train=np.zeros(0), fit_intercept=bool(fit_intercept), extra=extra, _finite=finite)
        dev = lambda a: self.to_device(a) if len(a) else torch.zeros(1, dtype=torch.int32, device=self.device)  # noqa: E731
        return SplitData(n=n, p=p, pa=Xa.shape[1], Xa=Xa, G_raw=G_raw, full=full, direct=plan["direct"],
                         direct_ptr=plan["direct_ptr"], direct_dev=dev(plan["direct_rows"]), out_ptr=plan["out_ptr"],
                         out_dev=dev(plan["out_rows"]), test_ptr=plan["test_ptr"], test_dev=dev(plan["test_rows"]),
                         n_obs=plan["n_obs"], n_train=plan["n_train"], fit_intercept=bool(fit_intercept),
                         weighted=sw is not None)

    def split_chunk(self, sd, s0, s1, buf):
        """Training Grams of splits s0..s1-1 of `sd` (at most SLM_MAX_FOLDS) in buf [>= s1-s0, pa, pa],
        centred if fit_intercept.  The direct splits take the first slots, the downdate splits the
        others.  Returns (order, fd): order[j] = split in slot j; fd a FoldData whose G_train are those
        slots (solve_specs, scoring and the refit take it as they take a partition's)."""
        c = s1 - s0
        assert 0 < c <= min(_lib.SLM_MAX_FOLDS, buf.shape[0])
        d = sd.direct[s0:s1]
        order = np.concatenate([s0 + np.flatnonzero(d), s0 + np.flatnonzero(~d)])
        a = int(d.sum())
        j0 = int(sd.direct[:s0].sum())  # direct splits before the chunk = its first entry of the direct CSR
        k0 = s0 - j0
        G = buf[:c]
        if a:
            self.gram_rows_update(sd.Xa, sd.direct_ptr[j0:j0 + a + 1], sd.direct_dev, G[:a])
        if a < c:
            G[a:].copy_(sd.G_raw.expand(c - a, sd.pa, sd.pa))
            self.gram_rows_update(sd.Xa, sd.out_ptr[k0:k0 + c - a + 1], sd.out_dev, G[a:], accumulate=True, negate=True)
        if sd.fit_intercept:
            self.gram_center(G, sd.p)
        extra = dict(sd.full.extra)
        extra["n_obs_train"] = sd.n_obs[order]
        fd = FoldData(n=sd.n, p=sd.p, pa=sd.pa, Xa=sd.Xa, row_ptr=None, G_train=G, G_full=sd.full.G_full,
                      n_train=sd.n_train[order], fit_intercept=sd.fit_intercept, extra=extra, _finite=sd.full._finite)
        return order, fd

    def gram_rows_update(self, Xa, row_ptr, rows_dev, G, accumulate=False, negate=False):
        """G[s] (+|-)= Xa[rows_s]^T Xa[rows_s] for every s (slm_gram_rows_update): rows_s =
        rows_dev[row_ptr[s]:row_ptr[s+1]] (device int32, ascending; row_ptr a host array of absolute
        offsets); accumulate=False overwrites G[s]; an empty list leaves G[s] untouched."""
        row_ptr = np.ascontiguousarray(row_ptr, dtype=np.int64)
        S = len(row_ptr) - 1
        pa = Xa.shape[1]
        Gs = G.reshape(-1, pa, pa)
        assert Gs.shape[0] >= S and Gs.stride(0) == pa * pa and Gs.is_contiguous()
        self._ck(self.lib.slm_gram_rows_update(self.h, self._ptr(Xa), Xa.shape[0], pa, S,
                                               row_ptr.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                               self._ptr(rows_dev), self._ptr(Gs), pa * pa, int(bool(accumulate)),
                                               int(bool(negate)), self.stream), "slm_gram_rows_update")
        return G

    def _gram_block_into(self, Xa, lo, hi, out, accumulate=False):
        """out (+)= Xa[lo:hi]^T Xa[lo:hi] (out untouched when the range is empty)."""
        if hi <= lo:
            return
        if accumulate:
            self._ck(self.lib.slm_gram_block_add(self.h, self._ptr(Xa), Xa.shape[1], int(lo), int(hi),
                                                 ctypes.c_void_p(out.data_ptr()), self.stream), "slm_gram_block_add")
            return
        ptr = np.array([lo, hi], dtype=np.int64)
        self._ck(self.lib.slm_gram_blocks(self.h, self._ptr(Xa), Xa.shape[1],
                                          ptr.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), 1,
                                          ctypes.c_void_p(out.data_ptr()), self.stream), "slm_gram_blocks")

    def _prepare_sharded(self, X, y, sw, col_perm, row_perm, row_ptr, fold_rows, shard, own_rows=False):
        """Row-sharded Gram build (SURVEY 8e): this rank contributes, for every test fold, the
        Gram of its own 1/world slice of that fold's rows; the blocks are then summed over the
        ranks.  With `own_rows` only this rank's slices are packed (everything otherwise)."""
        torch = self.torch
        F = len(row_ptr) - 1
        partial = own_rows and row_perm is None and F > 1
        if not partial:
            Xa = self.pack(X, y, sw, col_perm, row_perm)
        else:
            Xd = self.to_device(X, torch.float64)
            yd = self.to_device(y, torch.float64).reshape(-1)
            swd = None if sw is None else self.to_device(sw, torch.float64)
            cp = None if col_perm is None else self.to_device(np.asarray(col_perm, dtype=np.int32))
            n, p = Xd.shape
            Xa = torch.empty((n, self.padded_cols(p)), dtype=torch.float64, device=self.device)
            for a, b in fold_rows:
                self._pack_rows(Xd, yd, swd, cp, a, b, Xa)
        pa = Xa.shape[1]
        allG = torch.zeros((F + (1 if F > 1 else 0), pa, pa), dtype=torch.float64, device=self.device)
        for f, (lo, hi) in enumerate(fold_rows):
            self._gram_block_into(Xa, lo, hi, allG[f])
        self._complemented = self._allreduce_grams(allG, F, shard)
        return Xa, allG, partial

    def _allreduce_grams(self, allG, F, shard):
        """Sum the partial Gram blocks allG[:F] over the ranks: upper triangles packed into one buffer,
        ONE NCCL all-reduce.  For F > 1 the reduced buffer is unpacked straight into the F training
        Grams + the total (allG[:F+1], slm_tri_complement) and True is returned: the caller skips its own
        complement pass.  The collective runs on the caller's NCCL communicator inside the engine
        (slm_gram_allreduce) when the process group exposes it, through torch.distributed otherwise.
        (Measured on B200/NVLink: NCCL's bandwidth is bound by the CTAs it gets and the FP64 build
        wants every SM, so overlapping the two only slows both; half the bytes in one full-speed
        collective after the builds is faster at every rank count.)"""
        torch = self.torch
        pa = allG.shape[-1]
        nb = max(F, 1)
        tri = int(self.lib.slm_tri_size(pa))
        buf = torch.empty((nb, tri), dtype=torch.float64, device=self.device)
        comm = shard.comm_ptr(self.device)
        if F > 1 and comm is not None:
            self._ck(self.lib.slm_gram_allreduce(self.h, ctypes.c_void_p(comm), self._ptr(allG), pa * pa, pa, F,
                                                 self._ptr(buf), self.stream), "slm_gram_allreduce")
            return True
        self._ck(self.lib.slm_tri_pack(self.h, self._ptr(allG), pa * pa, pa, nb, self._ptr(buf), self.stream),
                 "slm_tri_pack")
        shard.allreduce_sum_(buf)
        if F > 1:
            self._ck(self.lib.slm_tri_complement(self.h, self._ptr(buf), pa, F, self._ptr(allG), pa * pa, self.stream),
                     "slm_tri_complement")
            return True
        self._ck(self.lib.slm_tri_unpack(self.h, self._ptr(buf), pa, nb, self._ptr(allG), pa * pa, self.stream),
                 "slm_tri_unpack")
        return False

    def _pack_rows(self, Xd, yd, swd, cp, a, b, Xa):
        """Xa[a:b] = [X | y | 1 | 0] of the device-resident rows a..b (identity row order)."""
        if b <= a:
            return
        pa = Xa.shape[1]
        self._ck(self.lib.slm_pack_design(self.h, ctypes.c_void_p(Xd.data_ptr() + 8 * a * Xd.stride(0)), Xd.stride(0),
                                          ctypes.c_void_p(yd.data_ptr() + 8 * a),
                                          ctypes.c_void_p(0 if swd is None else swd.data_ptr() + 8 * a),
                                          self._ptr(cp), ctypes.c_void_p(0), b - a, Xd.shape[1],
                                          ctypes.c_void_p(Xa.data_ptr() + 8 * a * pa), pa, self.stream),
                 "slm_pack_design")

    def _prepare_pipelined(self, X, y, sw, col_perm, row_ptr, fold_rows, shard=None, own_rows=False):
        """Host-resident X: the rows of one test fold at a time are copied to the device on a
        copy stream while the previous fold is packed and its Gram block is built, so the
        H2D transfer hides behind the FP64 tensor work (needs pinned memory to be truly
        asynchronous; pageable arrays still overlap chunk by chunk).  fold_rows[f] = the rows
        of fold f whose Gram this rank builds; with `shard` the blocks are then summed over the
        ranks (one all-reduce of the packed upper triangles); with `own_rows` (F > 1) only those
        rows travel."""
        torch = self.torch
        Xt = X if isinstance(X, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(X, dtype=np.float64))
        if Xt.dtype != torch.float64:
            Xt = Xt.to(torch.float64)
        n, p = Xt.shape
        pa = self.padded_cols(p)
        F = len(row_ptr) - 1
        dev = self.device
        yd = self.to_device(y, torch.float64).reshape(-1)
        swd = None if sw is None else self.to_device(sw, torch.float64)
        cp = None if col_perm is None else self.to_device(np.asarray(col_perm, dtype=np.int32))
        Xa = torch.empty((n, pa), dtype=torch.float64, device=dev)
        alloc = torch.zeros if shard is not None else torch.empty
        allG = alloc((F + (1 if F > 1 else 0), pa, pa), dtype=torch.float64, device=dev)

        # row blocks: the test folds, split further so that a block stays <= PIPELINE_BLOCK_BYTES;
        # the Gram of a fold (of the whole design for a plain fit) is accumulated block by block,
        # so only the last block's product is exposed after the last byte has crossed the bus
        blocks = []
        max_rows = max(1024, self.PIPELINE_BLOCK_BYTES // (8 * p))
        for f in range(F):
            a, b = int(row_ptr[f]), int(row_ptr[f + 1])
            if F > 1 and own_rows:
                a, b = fold_rows[f]  # only this rank's slice of the fold travels
                if b <= a:
                    if shard is not None:
                        blocks.append((a, a))  # nothing to build, but the collective still runs
                    continue
            nb = max(1, -(-(b - a) // max_rows))
            edges = np.linspace(a, b, nb + 1).astype(np.int64)
            blocks += [(int(edges[i]), int(edges[i + 1])) for i in range(nb) if edges[i + 1] > edges[i] or b == a]
        if not hasattr(self, "_copy_stream"):
            self._copy_stream = torch.cuda.Stream(device=dev)
        cur = torch.cuda.current_stream(dev)
        self._copy_stream.wait_stream(cur)
        staged = []
        started = set()  # Grams that already hold their first block
        for a, b in blocks:
            with torch.cuda.stream(self._copy_stream):
                blk = Xt[a:b].to(dev, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
            staged.append((a, b, blk, ev))
        for a, b, blk, ev in staged:
            cur.wait_event(ev)
            blk.record_stream(cur)
            self._ck(self.lib.slm_pack_design(self.h, self._ptr(blk), blk.stride(0), ctypes.c_void_p(yd.data_ptr() + 8 * a),
                                              ctypes.c_void_p(0 if swd is None else swd.data_ptr() + 8 * a),
                                              self._ptr(cp), ctypes.c_void_p(0), b - a, p,
                                              ctypes.c_void_p(Xa.data_ptr() + 8 * a * pa), pa, self.stream),
                     "slm_pack_design")
            # the Gram of the block's test fold (F > 1) / of the design (F == 1) takes the block as
            # soon as its rows are packed
            f = int(np.searchsorted(row_ptr, a, side="right") - 1) if F > 1 else 0
            lo, hi = max(a, fold_rows[f][0]), min(b, fold_rows[f][1])
            if hi > lo:
                self._gram_block_into(Xa, lo, hi, allG[f], accumulate=f in started)
                started.add(f)
        if shard is not None:
            self._complemented = self._allreduce_grams(allG, F, shard)
        return Xa, allG, bool(F > 1 and own_rows)

    # ---- K5-K8: batched solve ------------------------------------------------
    def solve(self, G, p, n_obs, lipschitz, grids, B0=None, tol=1e-10, floor_rel=1e-14, max_iter=20000,
              check_every=10, newton=None, W1_init=None):
        """Solve grids[f] (a PenaltyGrid) on Gram G[f] for every f, as one batch.

        newton: pure group penalties only (no l1 term) -- columns that have not converged after a
        first stretch of NEWTON_FIRST iterations get a lock-step Newton phase on their active groups
        (sparselm_b200/newton.py) between further stretches.  None (default) = on for
        160 < p <= 2048: below, the fused small-design kernel iterates at ~0.3 us per iteration;
        above, one p x p factorisation per column and step costs more than the iterations it saves
        unless the problem is known to be ill-conditioned (then pass True).  "l1": the same phase for
        every penalty, including those with an l1 term (Lasso, SparseGroupLasso and their adaptive
        variants: Newton steps on the manifold of fixed signs); for a pure group penalty the same as True.

        W1_init: optional device tensor [F, p, ldz] of per-coordinate l1 weights (instead of the
        per-column lam1; sparselm_b200/split.py).

        Returns dict with B (torch [F,p,ldz]), and numpy [F][K_f] arrays gap, primal,
        n_iter, status, n_pass.
        """
        torch = self.torch
        pa = G.shape[-1]
        Gs = G.reshape(-1, pa, pa)
        F = Gs.shape[0]
        if F > _lib.SLM_MAX_FOLDS:
            raise ValueError(f"at most {_lib.SLM_MAX_FOLDS} Grams per batch")
        assert len(grids) == F
        g0 = grids[0]
        Ks = [g.K for g in grids]
        ldz = max(8, _round_up(max(Ks), 8))
        Gn = g0.n_groups
        gptr_dev = None if g0.gptr is None else self.to_device(np.asarray(g0.gptr, dtype=np.int32))
        dev = self.device

        def stack_cols(rows, getter):
            out = np.zeros((F, rows, ldz))
            for f, g in enumerate(grids):
                v = getter(g)
                out[f, :, : g.K] = v
            return out

        lam1 = self.to_device(stack_cols(1, lambda g: np.asarray(g.lam1, dtype=float)[None, :]).reshape(F, ldz))
        use_W2 = any(g.W2 is not None for g in grids)
        use_D2 = any(g.D2 is not None for g in grids)
        W2 = self.to_device(stack_cols(Gn, lambda g: g.W2 if g.W2 is not None else 0.0)) if use_W2 else None
        D2 = self.to_device(stack_cols(Gn, lambda g: g.D2 if g.D2 is not None else 0.0)) if use_D2 else None
        W1 = None

        B = torch.zeros((F, p, ldz), dtype=torch.float64, device=dev)
        if B0 is not None:
            B.copy_(B0)
        nbytes = self.lib.slm_solve_workspace(p, ldz, F, Gn)
        work = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        # per-column results share one buffer so that they come back in a single D2H copy
        ncol = F * ldz
        rbuf = torch.zeros(24 * ncol, dtype=torch.uint8, device=dev)
        gap = rbuf[: 8 * ncol].view(torch.float64).view(F, ldz)
        primal = rbuf[8 * ncol: 16 * ncol].view(torch.float64).view(F, ldz)
        n_iter = rbuf[16 * ncol: 20 * ncol].view(torch.int32).view(F, ldz)
        status = rbuf[20 * ncol:].view(torch.int32).view(F, ldz)
        status.fill_(-1)

        bt = _lib.SlmBatch()
        bt.n_folds, bt.n_groups, bt.p, bt.pa, bt.ldz = F, Gn, p, pa, ldz
        bt.G_dev, bt.g_stride = Gs.data_ptr(), pa * pa
        bt.gptr_dev = 0 if gptr_dev is None else gptr_dev.data_ptr()
        bt.max_group = 0 if g0.gptr is None else int(np.diff(np.asarray(g0.gptr)).max(initial=0))
        lips_dev = lipschitz if isinstance(lipschitz, torch.Tensor) else None
        bt.lipschitz_dev = 0 if lips_dev is None else lips_dev.data_ptr()
        for f in range(F):
            bt.K[f] = Ks[f]
            bt.n_obs[f] = float(n_obs[f])
            bt.lipschitz[f] = 1.0 if lips_dev is not None else float(lipschitz[f])
        bt.lam1_dev = lam1.data_ptr()
        bt.W2_dev = 0 if W2 is None else W2.data_ptr()
        bt.D2_dev = 0 if D2 is None else D2.data_ptr()
        bt.B_dev = B.data_ptr()
        bt.work_dev, bt.work_bytes = work.data_ptr(), nbytes
        bt.tol, bt.floor_rel, bt.max_iter, bt.check_every = tol, floor_rel, int(max_iter), int(check_every)
        bt.gap_dev, bt.primal_dev = gap.data_ptr(), primal.data_ptr()
        bt.n_iter_dev, bt.status_dev = n_iter.data_ptr(), status.data_ptr()

        ad = g0.adaptive
        # columns without any l1 / group penalty (alpha = 0 is valid in the reference, _lasso.py:77-79):
        # the duality-gap test of the proximal iterations degenerates there, so they are solved as
        # (ridged) least squares by conjugate gradients on the same Gram and frozen in the batch
        unpen = None if W1_init is not None else \
            self._solve_unpenalised(Gs, p, n_obs, grids, g0, B, rbuf, F, ldz, ncol, tol)
        nctx = None
        if newton is None:
            newton = 160 < p <= 2048
        if newton and (W2 is not None or (ad is not None and ad.get("a2") is not None)):
            no_l1 = not np.any(np.concatenate([np.asarray(g.lam1, dtype=float).ravel() for g in grids]) != 0.0)
            if no_l1 and (ad is None or ad.get("a1") is None) and g0.gptr is not None:
                gid = torch.from_numpy(np.repeat(np.arange(Gn), np.diff(np.asarray(g0.gptr))).astype(np.int64)).to(dev)
                nctx = dict(Gs=Gs, B=B, gid=gid, gid32=gid.to(torch.int32), gptr_dev=gptr_dev,
                            n_obs=[float(v) for v in n_obs], Ks=Ks, status=status, n_iter=n_iter,
                            primal=primal, get_W2=lambda: W2, D2=D2, p=p, ldz=ldz, F=F, tol=tol, floor_rel=floor_rel,
                            stats={"phases": 0, "factorizations": 0, "newton_columns": 0, "ms": 0.0})
        has_l1 = W1_init is not None or (ad is not None and ad.get("a1") is not None) or bool(np.any(np.concatenate(
            [np.asarray(g.lam1, dtype=float).ravel() for g in grids]) != 0.0))
        if nctx is None and isinstance(newton, str) and newton == "l1" and has_l1 and (g0.gptr is not None or (W2 is None and D2 is None)):
            if g0.gptr is None:  # no group table (Lasso): one group of all p coordinates with zero weight
                ngptr = np.array([0, p], dtype=np.int64)
                zero_w2 = torch.zeros((F, 1, ldz), dtype=torch.float64, device=dev)
                get_W2 = lambda: zero_w2  # noqa: E731
            else:
                ngptr = np.asarray(g0.gptr, dtype=np.int64)
                get_W2 = lambda: W2 if W2 is not None else torch.zeros((F, Gn, ldz), dtype=torch.float64, device=dev)  # noqa: E731
            lam1_full = lam1[:, None, :].expand(F, p, ldz)  # the per-column l1 weight, broadcast (no copy)
            # the l1 weights the iterations use: W1_init, else lam1 until the adaptive passes allocate W1
            get_W1 = lambda: W1 if W1 is not None else (W1_init if W1_init is not None and ad is None else lam1_full)  # noqa: E731
            gid = torch.from_numpy(np.repeat(np.arange(len(ngptr) - 1), np.diff(ngptr)).astype(np.int64)).to(dev)
            nctx = dict(Gs=Gs, B=B, gid=gid, gid32=gid.to(torch.int32),
                        gptr_dev=self.to_device(ngptr.astype(np.int32)), n_obs=[float(v) for v in n_obs], Ks=Ks,
                        status=status, n_iter=n_iter, primal=primal, get_W2=get_W2, get_W1=get_W1, D2=D2, p=p,
                        ldz=ldz, F=F, tol=tol, floor_rel=floor_rel,
                        stats={"phases": 0, "factorizations": 0, "newton_columns": 0, "ms": 0.0})
        n_pass = np.ones((F, ldz), dtype=np.int64)
        total_iters = 0
        if ad is None:
            bt.W1_dev, bt.skip_dev = (0 if W1_init is None else W1_init.data_ptr()), 0
            skip0 = None
            if unpen is not None:
                skip0 = torch.from_numpy(unpen.astype(np.int32)).to(dev)
                bt.skip_dev = skip0.data_ptr()
            total_iters = self._run_batch(bt, nctx, base_skip=skip0)
        else:
            max_pass = int(ad["max_iter"])
            use_w1 = ad.get("a1") is not None
            use_w2 = ad.get("a2") is not None
            if use_w2 and W2 is None:
                W2 = torch.zeros((F, Gn, ldz), dtype=torch.float64, device=dev)
                bt.W2_dev = W2.data_ptr()

            def colvec(key):
                out = np.zeros((F, ldz))
                for f, g in enumerate(grids):
                    v = g.adaptive.get(key)
                    if v is not None:
                        out[f, : g.K] = v
                return self.to_device(out)

            a1 = colvec("a1") if use_w1 else None
            a2 = colvec("a2") if use_w2 else None
            alpha = colvec("alpha")
            gw = None if ad.get("gw") is None else self.to_device(np.asarray(ad["gw"], dtype=float))
            dnorm = torch.zeros((F, ldz), dtype=torch.float64, device=dev)
            skip = torch.zeros((F, ldz), dtype=torch.int32, device=dev)
            n_pass[:] = 0
            conv = np.zeros((F, ldz), dtype=bool)
            for f in range(F):
                conv[f, Ks[f]:] = True
            if unpen is not None:  # alpha = 0: the weights stay zero, the reference stops after one solve
                conv |= unpen
                n_pass[unpen] = 1
                skip.copy_(torch.from_numpy(conv.astype(np.int32)))
            for ps in range(max_pass):
                bt.W1_dev = 0 if W1 is None else W1.data_ptr()
                bt.skip_dev = skip.data_ptr()
                total_iters += self._run_batch(bt, nctx, base_skip=skip)
                n_pass[~conv] = ps + 1
                if use_w1 and W1 is None:  # previous l1 weights were lam1 (broadcast)
                    W1 = lam1[:, None, :].expand(F, p, ldz).contiguous()
                if ad.get("update_function") is not None:
                    self._host_update(ad, grids, B, W1, W2, dnorm, a1, a2, gptr_dev, gw, p, ldz, Ks)
                else:
                    for f in range(F):
                        self._ck(self.lib.slm_adaptive_update(
                            self.h, self._ptr(B[f]), p, ldz, Ks[f], Gn, self._ptr(gptr_dev), self._ptr(gw),
                            self._ptr(None if a1 is None else a1[f]), self._ptr(None if a2 is None else a2[f]),
                            self._ptr(alpha[f]), float(ad["eps"]), self._ptr(None if W1 is None else W1[f]),
                            self._ptr(None if not use_w2 else W2[f]), self._ptr(dnorm[f]), self.stream),
                            "slm_adaptive_update")
                dn = dnorm.cpu().numpy()
                conv |= dn <= float(ad["tol"])  # _adaptive_lasso.py:189-194
                if conv.all():
                    break
                skip.copy_(torch.from_numpy(conv.astype(np.int32)))

        rh = rbuf.cpu().numpy()
        res = {
            "B": B, "ldz": ldz, "K": Ks,
            "gap": rh[: 8 * ncol].view(np.float64).reshape(F, ldz),
            "primal": rh[8 * ncol: 16 * ncol].view(np.float64).reshape(F, ldz),
            "n_iter": rh[16 * ncol: 20 * ncol].view(np.int32).reshape(F, ldz),
            "status": rh[20 * ncol:].view(np.int32).reshape(F, ldz),
            "n_pass": n_pass, "iters_run": int(total_iters), "n_unconverged": int(bt.n_unconverged),
            "W1": W1, "W2": W2, "newton": None if nctx is None else nctx["stats"],
        }
        return res

    def _solve_unpenalised(self, Gs, p, n_obs, grids, g0, B, rbuf, F, ldz, ncol, tol):
        """Conjugate gradients for the columns whose penalty has no l1 / group part; fills B and the
        result buffer (gap 0, status, iterations) and returns their [F, ldz] mask (None: there are none)."""
        torch = self.torch
        mask = np.zeros((F, ldz), dtype=bool)
        for f, g in enumerate(grids):
            if g.K == 0:
                continue
            z = np.asarray(g.lam1, dtype=float) == 0.0
            if g.W2 is not None:
                z &= ~np.any(np.asarray(g.W2) != 0.0, axis=0)
            if g.adaptive is not None:
                z &= np.asarray(g.adaptive["alpha"], dtype=float) == 0.0
            mask[f, : g.K] = z
        if not mask.any():
            return None
        gptr = np.arange(p + 1) if g0.gptr is None else np.asarray(g0.gptr)
        sizes = np.diff(gptr)
        gap = rbuf[: 8 * ncol].view(torch.float64).view(F, ldz)
        primal = rbuf[8 * ncol: 16 * ncol].view(torch.float64).view(F, ldz)
        n_iter = rbuf[16 * ncol: 20 * ncol].view(torch.int32).view(F, ldz)
        status = rbuf[20 * ncol:].view(torch.int32).view(F, ldz)
        for f, g in enumerate(grids):
            done = {}
            for k in np.flatnonzero(mask[f]):
                d2 = None if g.D2 is None else np.asarray(g.D2)[:, k]
                key = None if d2 is None or not np.any(d2) else d2.tobytes()
                if key not in done:
                    shift = None if key is None else self.to_device(np.repeat(float(n_obs[f]) * d2, sizes))
                    X8, iters, rel = self.gram_cg(Gs[f], p, tol=min(1e-13, 1e-3 * tol), shift=shift)
                    b = X8[:, 0]
                    cvec = Gs[f][p, :p]
                    obj = (Gs[f][p, p] - (cvec * b).sum()) / (2.0 * float(n_obs[f]))  # = 1/(2n)||y - Xb||^2 + ridge at the optimum
                    done[key] = (b, iters, int(rel > 1e-9), obj)
                b, iters, st, obj = done[key]
                B[f, :, k] = b
                n_iter[f, k] = iters
                status[f, k] = st
                primal[f, k] = obj
                gap[f, k] = 0.0
        return mask

    def _run_batch(self, bt, nctx, base_skip=None):
        """One slm_solve_batch call -- or, with a Newton context, stretches of iterations with a
        lock-step Newton phase (newton.newton_phase) on the still unconverged columns in between.
        Converged columns are frozen through skip_dev; iteration counts are accumulated over the
        stretches.  Convergence is only ever decided by the engine's own certificate."""
        if nctx is None:
            self._ck(self.lib.slm_solve_batch(self.h, ctypes.byref(bt), self.stream), "slm_solve_batch")
            return bt.iters_run
        from .newton import newton_phase, newton_phase_device

        torch = self.torch
        F, ldz, p, Ks = nctx["F"], nctx["ldz"], nctx["p"], nctx["Ks"]
        B, Gs, status, n_iter = nctx["B"], nctx["Gs"], nctx["status"], nctx["n_iter"]
        budget, first, later, max_phases = int(bt.max_iter), self.NEWTON_FIRST, self.NEWTON_LATER, 12
        skip_ph = torch.zeros((F, ldz), dtype=torch.int32, device=self.device)
        if base_skip is not None:
            skip_ph.copy_(base_skip)
        for f in range(F):
            skip_ph[f, Ks[f]:] = 1
        base = skip_ph.cpu().numpy() != 0
        frozen = base.copy()
        acc = np.zeros((F, ldz), dtype=np.int64)
        fails = np.zeros((F, ldz), dtype=np.int64)  # Newton phases a column went through without finishing
        orig_skip = bt.skip_dev
        bt.skip_dev = skip_ph.data_ptr()
        total = 0
        try:
            last = False
            for ph in range(max_phases):
                last = last or ph == max_phases - 1
                bt.max_iter = max(1, budget - total) if last else max(1, min(first if ph == 0 else later, budget - total))
                self._ck(self.lib.slm_solve_batch(self.h, ctypes.byref(bt), self.stream), "slm_solve_batch")
                total += bt.iters_run
                st = status.cpu().numpy()
                acc[~frozen] += n_iter.cpu().numpy()[~frozen]
                slow = ~frozen & (st == 1)
                if not slow.any() or total >= budget or last:
                    break
                frozen |= ~slow
                skip_ph.copy_(torch.from_numpy(frozen.astype(np.int32)))
                # a column that three Newton phases did not finish (l1: nor shrink its support) stays with the
                # iterations (bounded extra cost on problems the phase does not help); with no candidate left the
                # next stretch runs to max_iter
                fi, ki = np.nonzero(slow & (fails < 3))
                if len(fi) == 0:
                    last = True
                    continue
                W2, D2 = nctx["get_W2"](), nctx["D2"]
                W1 = nctx["get_W1"]() if "get_W1" in nctx else None
                prim = nctx["primal"].cpu().numpy()
                floor = max(nctx["floor_rel"], 4e-15 / nctx["tol"])
                yty = Gs[:, p, p].cpu().numpy()
                scale = np.array([max(abs(prim[f, k]), floor * yty[f] / (2.0 * nctx["n_obs"][f])) for f, k in zip(fi, ki)])
                # chunks of columns: one [k, p, p] FP64 Hessian / factor at most ~16 GB
                chunk = max(1, int(16e9 // (32.0 * p * p)))
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                for c0 in range(0, len(fi), chunk):
                    fc = torch.from_numpy(fi[c0:c0 + chunk].astype(np.int64)).to(self.device)
                    kc = torch.from_numpy(ki[c0:c0 + chunk].astype(np.int64)).to(self.device)
                    X = B[fc, :, kc]
                    w2 = W2[fc, :, kc]
                    d2 = None if D2 is None else D2[fc, :, kc]
                    w1 = None if W1 is None else W1[fc, :, kc]
                    nn = torch.tensor([nctx["n_obs"][f] for f in fi[c0:c0 + chunk]], dtype=torch.float64, device=self.device)
                    sc = torch.from_numpy(scale[c0:c0 + chunk]).to(self.device)
                    if "gptr_dev" in nctx and os.environ.get("SLM_NEWTON_TORCH", "0") != "1":
                        Xn, info = newton_phase_device(self, Gs, fc, nn, X, w2, d2, nctx["gptr_dev"], nctx["gid32"], sc,
                                                       nctx["tol"], w1=w1)
                    else:  # SLM_NEWTON_TORCH=1: the torch / cuSOLVER model of the same iteration (A/B runs)
                        Xn, info = newton_phase(Gs, fc, nn, X, w2, d2, nctx["gid"], sc, nctx["tol"], w1=w1)
                    B[fc, :, kc] = Xn
                    nf = ~info["finished"]
                    if w1 is not None and self.NEWTON_L1_SHRINK_IS_PROGRESS:
                        nf &= (Xn != 0).sum(1) >= (X != 0).sum(1)
                    nf = nf.cpu().numpy()
                    fails[fi[c0:c0 + chunk][nf], ki[c0:c0 + chunk][nf]] += 1
                    nctx["stats"]["factorizations"] += int(info["factorizations"])
                ev1.record()
                ev1.synchronize()
                nctx["stats"]["ms"] += ev0.elapsed_time(ev1)
                nctx["stats"]["phases"] += 1
                nctx["stats"]["newton_columns"] += len(fi)
        finally:
            bt.skip_dev = orig_skip
            bt.max_iter = budget
        if os.environ.get("SLM_TRACE"):
            print(f"[slm newton] iterations {total} stats {nctx['stats']} unconverged {int(bt.n_unconverged)}", file=sys.stderr)
        keep = n_iter.cpu().numpy()
        keep[~base] = np.minimum(acc[~base], np.iinfo(np.int32).max)
        n_iter.copy_(torch.from_numpy(keep.astype(np.int32)))
        return total

    def _host_update(self, ad, grids, B, W1, W2, dnorm, a1, a2, gptr_dev, gw, p, ldz, Ks):
        """User-supplied update_function (arbitrary Python, _adaptive_lasso.py:116-118,
        177-182): evaluated on the host between passes."""
        torch = self.torch
        fn = ad["update_function"]
        Bh = B.cpu().numpy()
        F = Bh.shape[0]
        g0 = grids[0]
        gptr = np.arange(p + 1) if g0.gptr is None else np.asarray(g0.gptr)
        gwh = np.ones(len(gptr) - 1) if ad.get("gw") is None else np.asarray(ad["gw"], dtype=float)
        dn = np.zeros((F, ldz))
        W1h = None if W1 is None else W1.cpu().numpy()
        W2h = None if (W2 is None or a2 is None) else W2.cpu().numpy()
        for f, g in enumerate(grids):
            for k in range(Ks[f]):
                acc = 0.0
                b = Bh[f, :, k]
                if W1h is not None and a1 is not None:
                    wn = float(g.adaptive["a1"][k]) * np.asarray(fn(b, ad["eps"]), dtype=float)
                    acc += float(((wn - W1h[f, :, k]) ** 2).sum())
                    W1h[f, :, k] = wn
                if W2h is not None:
                    norms = np.sqrt(np.add.reduceat(b * b, gptr[:-1]))
                    wn = (float(g.adaptive["a2"][k]) * gwh) * np.asarray(fn(norms, ad["eps"]), dtype=float)
                    acc += float(((wn - W2h[f, :, k]) ** 2).sum())
                    W2h[f, :, k] = wn
                dn[f, k] = np.sqrt(acc)
        if W1h is not None and a1 is not None:
            W1.copy_(torch.from_numpy(W1h))
        if W2h is not None:
            W2.copy_(torch.from_numpy(W2h))
        dnorm.copy_(torch.from_numpy(dn))

    # ---- standardize=True: per-group whitening -------------------------------------
    def whiten(self, G, p, gptr, n_obs, shift=None, ridge=None, gscale=None):
        """Whitened copies of the Grams G [F, pa, pa] for the group structure gptr:
        Gw_f = W_f^T G_f W_f (+ n_f ridge_g W_g^T W_g on the diagonal blocks), W_f =
        blockdiag(R_g^{-1}), R_g^T R_g = gscale_f G_f[g, g] (+ shift_g I).  gscale_f (default 1) is
        rows / sum(sample_weight) of Gram f: the reference forms its standardized norms on rows
        scaled by weights *normalised to sum to the number of rows* (_base.py:214), the engine's
        Gram carries the raw weights.  Returns (Gw, ctx) where ctx
        carries the device-resident factors for `unwhiten`.  Raises ValueError if some
        group's columns are linearly dependent on the rows of a Gram (its block is not
        positive definite): ||X_g b_g|| is then only a semi-norm."""
        torch = self.torch
        pa = G.shape[-1]
        Gs = G.reshape(-1, pa, pa)
        F = Gs.shape[0]
        gptr = np.asarray(gptr, dtype=np.int64)
        Gn = len(gptr) - 1
        sizes = np.diff(gptr)
        wptr = np.concatenate([[0], np.cumsum(sizes * sizes)]).astype(np.int64)
        wtot = int(wptr[-1])
        gptr_dev = self.to_device(gptr.astype(np.int32))
        wptr_dev = self.to_device(wptr)
        shift_dev = None if shift is None else self.to_device(np.asarray(shift, dtype=np.float64))
        ridge_dev = None if ridge is None else self.to_device(np.asarray(ridge, dtype=np.float64))
        W = torch.empty((F, max(wtot, 1)), dtype=torch.float64, device=self.device)
        scratch = torch.empty(max(wtot, 1), dtype=torch.float64, device=self.device)
        info = torch.zeros(1, dtype=torch.int32, device=self.device)
        tmp = torch.empty((pa, pa), dtype=torch.float64, device=self.device)
        Gw = torch.empty_like(Gs)
        for f in range(F):
            kf = 1.0 if gscale is None else float(gscale[f])
            # R^T R = k G_gg + s I = k (G_gg + (s/k) I): factor the bracket, then W = R^{-1} = W' / sqrt(k)
            sh = shift_dev if (shift_dev is None or kf == 1.0) else shift_dev / kf
            self._ck(self.lib.slm_group_whiten_factors(self.h, self._ptr(Gs[f]), pa, p, self._ptr(gptr_dev),
                                                       self._ptr(wptr_dev), Gn, self._ptr(sh), self._ptr(W[f]),
                                                       self._ptr(scratch), self._ptr(info), self.stream),
                     "slm_group_whiten_factors")
            if kf != 1.0:
                W[f].mul_(1.0 / np.sqrt(kf))
            self._ck(self.lib.slm_gram_whiten(self.h, self._ptr(Gs[f]), pa, p, self._ptr(gptr_dev),
                                              self._ptr(wptr_dev), Gn, self._ptr(W[f]), self._ptr(ridge_dev),
                                              float(n_obs[f]), self._ptr(tmp), self._ptr(Gw[f]), self.stream),
                     "slm_gram_whiten")
        bad = int(info.item())
        if bad:
            raise ValueError(
                f"standardize=True: {bad} (group, training set) blocks X_g^T X_g are not positive definite "
                "(linearly dependent columns inside a group, or fewer rows than the group has features)")
        return Gw, dict(W=W, gptr_dev=gptr_dev, wptr_dev=wptr_dev, Gn=Gn)

    def unwhiten(self, Bg, wctx, f, p, K):
        """Coefficients of Gram f back in the caller's variables: b_g = W_g gamma_g."""
        out = self.torch.zeros_like(Bg)
        self._ck(self.lib.slm_coef_unwhiten(self.h, self._ptr(Bg), p, Bg.shape[-1], int(K), self._ptr(wctx["gptr_dev"]),
                                            self._ptr(wctx["wptr_dev"]), wctx["Gn"], self._ptr(wctx["W"][f]),
                                            self._ptr(out), self.stream), "slm_coef_unwhiten")
        return out

    # ---- K9 / K10 ---------------------------------------------------------------
    def fold_back(self, Bext, inv_ptr_dev, inv_idx_dev, p, K):
        torch = self.torch
        ldz = Bext.shape[-1]
        coef = torch.zeros((p, ldz), dtype=torch.float64, device=self.device)
        self._ck(self.lib.slm_fold_back(self.h, self._ptr(Bext), self._ptr(inv_ptr_dev), self._ptr(inv_idx_dev),
                                        p, ldz, K, self._ptr(coef), self.stream), "slm_fold_back")
        return coef

    def support_counts(self, coef, K, rel_tol, counts, union):
        """Selection counts of the [F, p, ldz] coefficient table `coef` (slm_support_counts): counts [p, K] int32
        += fits that select (j, k); union [F, p] uint8 |= some candidate of fit f selects j.  Selected:
        |b_j| > rel_tol * max_j' |b_j'| within one fit.  Both accumulate in place on the device."""
        torch = self.torch
        F, p, ldz = coef.shape
        assert coef.dtype == torch.float64 and coef.is_contiguous()
        assert counts.dtype == torch.int32 and counts.is_contiguous() and tuple(counts.shape) == (p, K)
        assert union.dtype == torch.uint8 and union.is_contiguous() and tuple(union.shape) == (F, p)
        self._ck(self.lib.slm_support_counts(self.h, self._ptr(coef), F, p, ldz, int(K), float(rel_tol),
                                             self._ptr(counts), self._ptr(union), self.stream), "slm_support_counts")

    def group_support_counts(self, coef, K, rel_tol, gptr_dev, counts, union):
        """support_counts per group (slm_group_support_counts): group g holds rows gptr_dev[g] .. gptr_dev[g+1]-1 of
        `coef` (device int32 [G+1]) and is selected in a fit iff one of its features is.  counts [G, K] int32 +=
        fits that select (g, k); union [F, G] uint8 |= some candidate of fit f selects g."""
        torch = self.torch
        F, p, ldz = coef.shape
        G = gptr_dev.shape[0] - 1
        assert coef.dtype == torch.float64 and coef.is_contiguous()
        assert gptr_dev.dtype == torch.int32 and gptr_dev.is_contiguous() and gptr_dev.is_cuda
        assert counts.dtype == torch.int32 and counts.is_contiguous() and tuple(counts.shape) == (G, K)
        assert union.dtype == torch.uint8 and union.is_contiguous() and tuple(union.shape) == (F, G)
        self._ck(self.lib.slm_group_support_counts(self.h, self._ptr(coef), F, p, ldz, int(K), float(rel_tol),
                                                   self._ptr(gptr_dev), G, self._ptr(counts), self._ptr(union),
                                                   self.stream), "slm_group_support_counts")

    def gram_scale(self, G, p, weights, slots):
        """G[s] *= outer(d, d) in place (slm_gram_scale) for the Grams G [S, pa, pa]: d = weights[slots[s]] (device
        float64 [n_rows, p], the Grams' column order) on the p feature rows and columns, 1 elsewhere."""
        torch = self.torch
        pa = G.shape[-1]
        Gs = G.reshape(-1, pa, pa)
        S = Gs.shape[0]
        slots = np.ascontiguousarray(slots, dtype=np.int64)
        assert Gs.dtype == torch.float64 and Gs.is_contiguous() and len(slots) == S
        assert weights.dtype == torch.float64 and weights.is_contiguous() and weights.shape[1] == p
        self._ck(self.lib.slm_gram_scale(self.h, self._ptr(Gs), pa * pa, pa, int(p), S, self._ptr(weights),
                                         weights.shape[0], slots.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)),
                                         self.stream), "slm_gram_scale")
        return G

    def intercepts(self, G, p, B, K):
        torch = self.torch
        ldz = B.shape[-1]
        out = torch.zeros(ldz, dtype=torch.float64, device=self.device)
        self._ck(self.lib.slm_intercepts(self.h, self._ptr(G), G.shape[-1], p, self._ptr(B), ldz, K,
                                         self._ptr(out), self.stream), "slm_intercepts")
        return out

    def cv_score(self, Xa, p, r0, r1, B, K, intercept=None, rows_scaled=False):
        """(sse[K], sae[K]) of the rows [r0, r1) of Xa for the K columns of B (unweighted
        residuals; rows_scaled: Xa was packed with sample weights)."""
        torch = self.torch
        ldz = B.shape[-1]
        m = int(r1 - r0)
        yhat = torch.empty((m + 256, ldz), dtype=torch.float64, device=self.device)
        out = torch.zeros((2, ldz), dtype=torch.float64, device=self.device)
        self._ck(self.lib.slm_cv_score(self.h, self._ptr(Xa), Xa.shape[1], p, int(r0), int(r1), self._ptr(B), ldz,
                                       K, self._ptr(intercept), 1 if rows_scaled else 0, self._ptr(yhat),
                                       self._ptr(out), self.stream),
                 "slm_cv_score")
        return out


    def cv_score_many(self, Xa, p, items, rows_scaled=False):
        """Residual sums of several (row range, coefficient block) pairs in ONE tensor-core launch.
        items: list of (r0, r1, B, K, intercept) with B a device view [p, >= K] whose row stride is even and
        whose first element is 16-byte aligned (a column slice of a wider table is fine), intercept a device
        view [K] or None.  Returns a device tensor [len(items), 2, ldo] (sse, sae in the first K entries)."""
        return self._cv_score(Xa, p, items, rows_scaled, None)[0]

    def cv_score_rows(self, Xa, p, items, rows_scaled=False):
        """cv_score_many over row lists: items are (rows, B, K, intercept) with rows a device int32 view of the
        rows of Xa to score.  Returns a device tensor [len(items), 2, ldo] (sse, sae in the first K entries)."""
        return self._cv_score(Xa, p, items, rows_scaled, None)[0]

    def cv_score_stats(self, Xa, p, items, rows_scaled=False, stats=0, return_residuals=False):
        """cv_score_many (items (r0, r1, B, K, intercept)) or cv_score_rows (items (rows, B, K, intercept)) with the
        residual statistics of the `stats` bit mask (_lib.SLM_STAT_MAX | SLM_STAT_MAPE | SLM_STAT_MEDIAN).
        Returns a device tensor [len(items), 5, ldo]: sse, sae, max |r|, sum |r| / max(|y|, eps), median |r| in
        the first K entries (rows whose bit is not set are zero); with return_residuals also, per item, the
        device view [m, ldo] of the residuals that were reduced (first K columns)."""
        out, res = self._cv_score(Xa, p, items, rows_scaled, int(stats))
        return (out, res) if return_residuals else out

    def _cv_score(self, Xa, p, items, rows_scaled, stats):
        """One call of slm_cv_score_many / _rows (stats None) or slm_cv_score_stats: range items are 5-tuples,
        row-list items 4-tuples.  Returns (out [len(items), 2 or 5, ldo], per-item [m, ldo] scratch views)."""
        torch = self.torch
        n = len(items)
        ranges = n > 0 and len(items[0]) == 5
        ldo = max([max(8, _round_up(int(it[-2]), 8)) for it in items], default=8)
        nrow = 2 if stats is None else 5
        # one leading dimension for every problem: slot i of the result is a plain [nrow, ldo] block
        out = torch.zeros((max(n, 1), nrow, ldo), dtype=torch.float64, device=self.device)
        if n == 0:
            return out, []
        rows = [max(0, int(it[1]) - int(it[0])) if ranges else int(it[0].numel()) for it in items]
        offs = np.concatenate([[0], np.cumsum([(m + 256) * ldo for m in rows])]).astype(np.int64)
        yhat = torch.empty(int(offs[-1]), dtype=torch.float64, device=self.device)
        i64, i32, vp = ctypes.c_int64 * n, ctypes.c_int32 * n, ctypes.c_void_p * n
        B, K, ic = ([it[j] for it in items] for j in (-3, -2, -1))
        Bp = vp(*[b.data_ptr() for b in B])
        ldb = i64(*[int(b.stride(0)) for b in B])
        Kc = i32(*[int(k) for k in K])
        icp = vp(*[(None if c is None else c.data_ptr()) for c in ic])
        yp = vp(*[yhat.data_ptr() + 8 * int(o) for o in offs[:-1]])
        ldy = i64(*([ldo] * n))
        op = vp(*[out.data_ptr() + 8 * i * nrow * ldo for i in range(n)])
        if ranges:
            r0, r1 = i64(*[int(it[0]) for it in items]), i64(*[int(it[1]) for it in items])
            rp = nr = None
        else:
            r0 = r1 = None
            rp, nr = vp(*[it[0].data_ptr() for it in items]), i64(*rows)
        sc = 1 if rows_scaled else 0
        if stats is not None:
            self._ck(self.lib.slm_cv_score_stats(self.h, self._ptr(Xa), Xa.shape[1], p, n, r0, r1, rp, nr, Bp, ldb,
                                                 Kc, icp, sc, stats, yp, ldy, op, self.stream), "slm_cv_score_stats")
        elif ranges:
            self._ck(self.lib.slm_cv_score_many(self.h, self._ptr(Xa), Xa.shape[1], p, n, r0, r1, Bp, ldb, Kc, icp, sc,
                                                yp, ldy, op, self.stream), "slm_cv_score_many")
        else:
            self._ck(self.lib.slm_cv_score_rows(self.h, self._ptr(Xa), Xa.shape[1], p, n, rp, nr, Bp, ldb, Kc, icp, sc,
                                                yp, ldy, op, self.stream), "slm_cv_score_rows")
        return out, [yhat[int(o):int(o) + m * ldo].view(m, ldo) for o, m in zip(offs[:-1], rows)]


_engines: dict = {}


def get_engine(device: int | None = None) -> Engine:
    """Process-wide engine per device (one handle per (process, device))."""
    import torch

    if not torch.cuda.is_available():
        raise EngineError("sparselm_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    idx = torch.cuda.current_device() if device is None else int(device)
    if idx not in _engines:
        _engines[idx] = Engine(idx)
    return _engines[idx]

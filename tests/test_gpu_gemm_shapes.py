"""Every tile shape of the FP64 GEMM menus (csrc/engine.cu), on every operand feed, against exact float64
references.

The automatic tile choice (pick_shape) only reaches a few shapes of each menu at the sizes the other tests use,
so every (menu, shape id, feed) combination is pinned here with the force_*_shape options and run at sizes aimed
at that shape's edges: M / K tails around the tile and the 16- / 32-row k-slab, N tails around the tile width, a
fold with K = 0 inside a batch, one tile cut over many CTAs, and tile counts one below, at and one above a whole
wave (sm_count x MINB) of the stream-K scheduler.  MINB is what the tile is built for; where the measured
occupancy of a shape is lower, its wave-edge cases land off the edge but remain valid tests.

Two data regimes per case:
  * integers in [-4, 4]: every partial sum is exact in float64 whatever the summation order, so the result must
    equal numpy's bit for bit -- one lost, doubled or misplaced term anywhere (one k-slab of one split tile) fails;
  * standard normal data, within the elementwise DGEMM bound 2 (k + 2) eps (|A| |B|)_ij (small integers are also
    exact in FP32 / TF32; only real-valued data exposes a reduced-precision path), run twice: the fixed-order
    stream-K fix-up promises bitwise-equal results.

Sentinels: NaN fills everything the contraction must not read (Gram rows and columns p..pa-1, Z / B columns >= K,
design rows outside the block), so a kernel that multiplies data it should have masked by zero fails; every output
is pre-filled with a NaN payload, and everything outside the region a call may write must keep those bits (stray
stores), while the region it must write has to be overwritten (missing tiles).
"""

import ctypes
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
NAN_BITS = 0x7FF8DEADBEEF0A5A  # quiet NaN with a payload no arithmetic produces
GUARD = 64  # doubles of NaN guard before and after every output (keeps 16-byte alignment)

# (BM, BN, MINB) of every menu entry, only used to aim the sizes at a shape's edges
APPLY_MENU = [(128, 128, 1), (128, 104, 1), (128, 104, 1), (128, 56, 2), (128, 128, 1), (128, 64, 2), (64, 104, 2),
              (128, 32, 2), (128, 16, 2), (128, 8, 2), (128, 24, 2), (128, 40, 2), (128, 48, 2), (128, 72, 1),
              (128, 80, 1), (128, 88, 1), (128, 96, 1)]
SPARSE_MENU = [(128, 8, 3), (128, 16, 3), (128, 24, 3), (128, 32, 3), (128, 40, 3), (128, 48, 3), (128, 56, 2),
               (128, 64, 2), (128, 72, 1), (128, 88, 1), (128, 104, 1), (128, 128, 1), (128, 104, 1), (128, 64, 2)]
SYRK_MENU = [(128, 128, 1)] * 4  # ids 0-1: 32-deep slabs (TMA-capable), 2-3: 16-deep (cp.async only)
SCORE_MENU = [(128, 128, 1), (128, 64, 2), (128, 32, 2), (128, 16, 2), (128, 8, 2)]

# "tma" option masks: bit 0 Gram build, bit 1 dense apply, bit 2 row-sparse apply on TMA; bit 3 wide bands for the
# gather kernels, bit 4 for the tiled kernels
CP_ASYNC, TMA_BOXES, TMA_WIDE_TILED, TMA_WIDE_GATHER = 0, 7, 7 + 16, 7 + 8
FEED_NAME = {CP_ASYNC: "cp_async", TMA_BOXES: "tma_boxes", TMA_WIDE_TILED: "tma_wide", TMA_WIDE_GATHER: "tma_wide"}


def _cases(menu, feeds_of):
    return [pytest.param(sid, feed, id=f"s{sid:02d}-{FEED_NAME[feed]}") for sid in range(len(menu))
            for feed in feeds_of(sid)]


APPLY_CASES = _cases(APPLY_MENU, lambda sid: (CP_ASYNC, TMA_BOXES, TMA_WIDE_TILED))
SPARSE_CASES = _cases(SPARSE_MENU,
                      lambda sid: (CP_ASYNC, TMA_BOXES, TMA_WIDE_GATHER) if SPARSE_MENU[sid][1] > 16 else (CP_ASYNC,))
SYRK_CASES = _cases(SYRK_MENU, lambda sid: (CP_ASYNC, TMA_BOXES, TMA_WIDE_TILED) if sid <= 1 else (CP_ASYNC,))


@pytest.fixture(scope="module")
def eng(engine):
    yield engine
    for opt in ("force_apply_shape", "force_sparse_shape", "force_syrk_shape", "force_score_shape"):
        engine.set_option(opt, -1)
    engine.set_option("tma", 15)  # the engine default


def _round_up(x, m):
    return (x + m - 1) // m * m


# ---- device buffers with NaN guards -------------------------------------------------------------------------
class Out:
    """A NaN-filled device buffer: `size` doubles between two guards of GUARD doubles."""

    def __init__(self, eng, size):
        import torch

        self.size = int(size)
        self.buf = torch.full((self.size + 2 * GUARD,), NAN_BITS, dtype=torch.int64, device=eng.device)
        self.t = self.buf[GUARD:GUARD + self.size].view(torch.float64)

    @property
    def ptr(self):
        return ctypes.c_void_p(self.t.data_ptr())

    def fetch(self):
        """(values [size], NaN-bits-kept mask [size]); asserts that both guards kept their bits."""
        bits = self.buf.cpu().numpy()
        assert (bits[:GUARD] == NAN_BITS).all() and (bits[GUARD + self.size:] == NAN_BITS).all(), \
            "a store landed outside the output"
        inner = bits[GUARD:GUARD + self.size]
        return inner.view(np.float64).copy(), inner == NAN_BITS


def _dev(eng, a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a)).to(eng.device)


def _check(got, kept, must, free, want, bound=None, what=""):
    """got / kept: arrays of one output's values and NaN-bits mask; must: bool mask of the entries the call has to
    write (compared with want, exactly or within bound); free: entries that may hold anything; every other entry
    must have kept its NaN bits."""
    untouched = ~(must | free)
    assert kept[untouched].all(), f"{what}: {int((~kept[untouched]).sum())} stray stores"
    g, w = got[must], want[must]
    assert np.isfinite(g).all(), f"{what}: {int((~np.isfinite(g)).sum())} entries not written or not finite"
    if bound is None:
        bad = g != w
        assert not bad.any(), f"{what}: {int(bad.sum())} of {g.size} entries differ (max {np.abs(g - w).max():.3g})"
    else:
        bad = np.abs(g - w) > bound[must]
        assert not bad.any(), f"{what}: {int(bad.sum())} of {g.size} entries outside the DGEMM bound"


def _ints(rng, shape):
    return rng.integers(-4, 5, size=shape).astype(np.float64)


def _tma_check(eng, before, eligible, what):
    assert (eng.tma_launch_count() > before) == eligible, f"{what}: TMA kernel {'not ' if eligible else ''}launched"


# ---- menu sizes and the option range check ---------------------------------------------------------------------
def _menu_size(eng, opt):
    from sparselm_b200.engine import EngineError

    n = 0
    while n < 64:
        try:
            eng.set_option(opt, n)
        except EngineError:
            break
        n += 1
    eng.set_option(opt, -1)
    return n


def test_menu_sizes_and_out_of_range_ids(eng):
    from sparselm_b200.engine import EngineError

    sizes = {opt: _menu_size(eng, opt) for opt in ("force_apply_shape", "force_sparse_shape", "force_syrk_shape",
                                                   "force_score_shape")}
    # a menu change has to update the mirrors above (and so the test ids) on purpose
    assert sizes == {"force_apply_shape": len(APPLY_MENU), "force_sparse_shape": len(SPARSE_MENU),
                     "force_syrk_shape": len(SYRK_MENU), "force_score_shape": len(SCORE_MENU)}
    assert (len(APPLY_MENU), len(SPARSE_MENU), len(SYRK_MENU), len(SCORE_MENU)) == (17, 14, 4, 5)
    for opt, n in sizes.items():
        for bad in (-2, n, n + 1, 1 << 20):
            with pytest.raises(EngineError, match=opt):
                eng.set_option(opt, bad)
        eng.set_option(opt, -1)


# ---- dense Gram apply: GZ_f = G_f Z_f ----------------------------------------------------------------------------
def _sym_gram(rng, F, p, pa, ints):
    A = _ints(rng, (F, p, p)) if ints else rng.standard_normal((F, p, p))
    G = np.full((F, pa, pa), np.nan)
    G[:, :p, :p] = np.triu(A) + np.triu(A, 1).transpose(0, 2, 1)  # symmetric, entries in [-4, 4] for integers
    return G


def _wave_ks(T, BN, folds=16):
    """per-fold K of a batch of `folds` folds with T tiles of width BN in total (one tile row): each K ends 3 columns
    short of its last tile, so that the tail is odd and the tile count is exact."""
    c = [T // folds + (1 if f < T % folds else 0) for f in range(folds)]
    return tuple(ci * BN - 3 if ci > 0 else 0 for ci in c)


def _apply_sizes(BM, BN, MINB, sms):
    """(p, Ks) of one shape's cases."""
    tails = (1, 0, 7, 8, BN, BN + 1)  # a fold with K = 0 inside the batch
    cases = [(BM - 1, tails), (BM, tails), (BM + 1, tails),  # M tails; also p % 16 == 15 / 0 / 1 (last slab 15 / 16 / 1)
             (13, (5, BN + 1)),                             # p < 16: a single, partial slab
             (BM - 3, (BN - 1,)), (BM, (BN,))]              # one tile cut over every slab's CTA (stream-K fix-up chain)
    wave = sms * MINB
    cases += [(BM - 9, _wave_ks(T, BN)) for T in (wave - 1, wave, wave + 1)]
    return cases


@functools.lru_cache(maxsize=24)
def _apply_data(p, Ks, ints):
    F = len(Ks)
    pa = _round_up(p + 2, 8)
    ldz = _round_up(max(max(Ks), 1), 8) + 8  # a column block beyond every fold's N
    rng = np.random.default_rng([p, F, ldz, int(ints)])
    G = _sym_gram(rng, F, p, pa, ints)
    Z = _ints(rng, (F, p, ldz)) if ints else rng.standard_normal((F, p, ldz))
    for f, k in enumerate(Ks):
        Z[f, :, k:] = np.nan  # columns >= K are not part of the product
    ref = [G[f, :p, :p] @ Z[f, :, :Ks[f]] for f in range(F)]
    bound = None if ints else [2 * (p + 2) * EPS * (np.abs(G[f, :p, :p]) @ np.abs(Z[f, :, :Ks[f]])) for f in range(F)]
    return G, Z, ldz, ref, bound


def _apply_expect(p, Ks, ldz, ref, bound):
    """(want, must, free, bound) over the flat [F][p][ldz] output."""
    F = len(Ks)
    want = np.zeros((F, p, ldz))
    must = np.zeros((F, p, ldz), bool)
    free = np.zeros((F, p, ldz), bool)
    bnd = np.zeros((F, p, ldz))
    for f, k in enumerate(Ks):
        if k == 0:
            continue  # no tile: the fold's output is untouched
        N = min(_round_up(k, 8), ldz)
        want[f, :, :k] = ref[f]
        must[f, :, :k] = True
        free[f, :, k:N] = True
        if bound is not None:
            bnd[f, :, :k] = bound[f]
    return want.ravel(), must.ravel(), free.ravel(), (bnd.ravel() if bound is not None else None)


def _run_apply(eng, G, p, Ks, Z, ldz):
    F = len(Ks)
    pa = G.shape[1]
    Gd, Zd = _dev(eng, G), _dev(eng, Z)
    out = Out(eng, F * p * ldz)
    Karr = (ctypes.c_int32 * F)(*Ks)
    eng._ck(eng.lib.slm_gram_apply(eng.h, eng._ptr(Gd), pa * pa, pa, p, F, Karr, eng._ptr(Zd), ldz, out.ptr,
                                   eng.stream), "slm_gram_apply")
    return out.fetch()


@pytest.mark.parametrize("sid,feed", APPLY_CASES)
def test_apply_shape(eng, sid, feed):
    BM, BN, MINB = APPLY_MENU[sid]
    eng.set_option("tma", feed)
    eng.set_option("force_apply_shape", sid)
    try:
        for p, Ks in _apply_sizes(BM, BN, MINB, eng.sm_count):
            what = f"apply shape {sid} feed {feed} p={p} Ks={Ks[:8]}"
            for ints in (True, False):
                G, Z, ldz, ref, bound = _apply_data(p, Ks, ints)
                want, must, free, bnd = _apply_expect(p, Ks, ldz, ref, bound)
                t0 = eng.tma_launch_count()
                got, kept = _run_apply(eng, G, p, Ks, Z, ldz)
                _tma_check(eng, t0, feed != CP_ASYNC, what)
                _check(got, kept, must, free, want, bnd, what + (" integers" if ints else " normal"))
                if not ints:
                    again, _ = _run_apply(eng, G, p, Ks, Z, ldz)
                    assert np.array_equal(got[must], again[must]), what + ": not bitwise reproducible"
    finally:
        eng.set_option("force_apply_shape", -1)
        eng.set_option("tma", 15)


# ---- row-sparse Gram apply -------------------------------------------------------------------------------------------
def _sparse_sizes(BN):
    """(p, Ks, chunk_w) of one shape's cases."""
    return [(129, (136, 130), 8),            # 34 chunk problems: a second launch
            (127, (40, 0, 17), 16),          # a fold with K = 0
            (128, (BN, BN + 1), 32),
            (143, (1, 7, 8), 64),
            (145, (BN + 1, 200), 128),
            (13, (13, 5), 8)]                # p < 16


@functools.lru_cache(maxsize=32)
def _sparse_data(p, Ks, chunk_w, ints):
    F = len(Ks)
    pa = _round_up(p + 2, 8)
    ldz = _round_up(max(Ks), 8) + 8
    rng = np.random.default_rng([p, F, ldz, chunk_w, int(ints)])
    G = _sym_gram(rng, F, p, pa, ints)
    Z = np.zeros((F, p, ldz))
    # support lengths per chunk: around the 4-row gather (padded with the last row) and the 16-row slab, p - 1, p
    lens = [min(p, L) for L in (0, 1, 3, 4, 5, 15, 16, 17)] + [p - 1, p]
    t = 0
    for f, k in enumerate(Ks):
        for c0 in range(0, k, chunk_w):
            c1 = min(k, c0 + chunk_w)
            L = lens[(t + f) % len(lens)]
            t += 1
            if L == 0:
                continue
            rows = [0, p - 1][:L] if L <= 2 else [0, p - 1] + list(rng.choice(np.arange(1, p - 1), L - 2,
                                                                             replace=False))
            rows = np.unique(rows)
            vals = _ints(rng, (len(rows), c1 - c0)) if ints else rng.standard_normal((len(rows), c1 - c0))
            vals[:, 0] = np.where(vals[:, 0] == 0, 3.0, vals[:, 0])  # every listed row is in the chunk's support
            Z[f, rows, c0:c1] = vals
        Z[f, :, k:] = np.nan
    ref = [G[f, :p, :p] @ Z[f, :, :Ks[f]] for f in range(F)]
    bound = None if ints else [2 * (p + 2) * EPS * (np.abs(G[f, :p, :p]) @ np.abs(Z[f, :, :Ks[f]])) for f in range(F)]
    return G, Z, ldz, ref, bound


def _run_sparse(eng, G, p, Ks, Z, ldz, chunk_w):
    import torch

    F = len(Ks)
    pa = G.shape[1]
    Gd, Zd = _dev(eng, G), _dev(eng, Z)
    out = Out(eng, F * p * ldz)
    Karr = (ctypes.c_int32 * F)(*Ks)
    nbytes = eng.lib.slm_rowsparse_workspace(p, ldz, F)
    work = torch.empty(nbytes, dtype=torch.uint8, device=eng.device)
    eng._ck(eng.lib.slm_gram_apply_rowsparse(eng.h, eng._ptr(Gd), pa * pa, pa, p, F, Karr, eng._ptr(Zd), ldz, out.ptr,
                                             chunk_w, eng._ptr(work), nbytes, eng.stream), "slm_gram_apply_rowsparse")
    return out.fetch()


@pytest.mark.parametrize("sid,feed", SPARSE_CASES)
def test_rowsparse_apply_shape(eng, sid, feed):
    BM, BN, MINB = SPARSE_MENU[sid]
    eng.set_option("tma", feed)
    eng.set_option("force_sparse_shape", sid)
    try:
        for p, Ks, chunk_w in _sparse_sizes(BN):
            what = f"row-sparse shape {sid} feed {feed} p={p} Ks={Ks} chunk_w={chunk_w}"
            for ints in (True, False):
                G, Z, ldz, ref, bound = _sparse_data(p, Ks, chunk_w, ints)
                want, must, free, bnd = _apply_expect(p, Ks, ldz, ref, bound)
                t0 = eng.tma_launch_count()
                got, kept = _run_sparse(eng, G, p, Ks, Z, ldz, chunk_w)
                _tma_check(eng, t0, feed != CP_ASYNC and BN > 16, what)
                _check(got, kept, must, free, want, bnd, what + (" integers" if ints else " normal"))
                if not ints:
                    again, _ = _run_sparse(eng, G, p, Ks, Z, ldz, chunk_w)
                    assert np.array_equal(got[must], again[must]), what + ": not bitwise reproducible"
    finally:
        eng.set_option("force_sparse_shape", -1)
        eng.set_option("tma", 15)


# ---- Gram build: G_f = Xa_f^T Xa_f (upper tiles + mirror) --------------------------------------------------------
BLOCK_ROWS = (0, 1, 15, 16, 17, 31, 32, 33, 50)  # around the 16- and 32-row slabs; 0 = untouched block


@functools.lru_cache(maxsize=16)
def _syrk_data(pa, kind, ints):
    """kind "blocks": 40 blocks (two launches) after 5 NaN rows; "add": one block [r0, r1) inside NaN rows, added to
    an integer matrix; "long": one block of 20 000 rows (hundreds of 32-row slabs over every CTA)."""
    rng = np.random.default_rng([pa, len(kind), int(ints)])
    if kind == "blocks":
        sizes = [BLOCK_ROWS[i % len(BLOCK_ROWS)] for i in range(40)]
        row_ptr = np.concatenate([[5], 5 + np.cumsum(sizes)]).astype(np.int64)
    elif kind == "add":
        row_ptr = np.array([37, 37 + 301], dtype=np.int64)
    else:
        row_ptr = np.array([0, 20000], dtype=np.int64)
    n = int(row_ptr[-1]) + 7
    Xa = np.full((n, pa), np.nan)
    r0, r1 = int(row_ptr[0]), int(row_ptr[-1])
    Xa[r0:r1] = _ints(rng, (r1 - r0, pa)) if ints else rng.standard_normal((r1 - r0, pa))
    blocks = [Xa[row_ptr[f]:row_ptr[f + 1]] for f in range(len(row_ptr) - 1)]
    ref = [b.T @ b for b in blocks]
    bound = None if ints else [2 * (len(b) + 2) * EPS * (np.abs(b).T @ np.abs(b)) for b in blocks]
    G0 = None
    if kind == "add":  # a Gram to add to: symmetric, like the sums of earlier blocks
        G0 = _ints(rng, (pa, pa))
        G0 = np.triu(G0) + np.triu(G0, 1).T
    return Xa, row_ptr, ref, bound, G0


def _run_syrk(eng, Xa, row_ptr, G0):
    import torch

    pa = Xa.shape[1]
    Xd = _dev(eng, Xa)
    F = len(row_ptr) - 1
    out = Out(eng, F * pa * pa)
    if G0 is None:
        rp = np.ascontiguousarray(row_ptr, dtype=np.int64)
        eng._ck(eng.lib.slm_gram_blocks(eng.h, eng._ptr(Xd), pa, rp.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), F,
                                        out.ptr, eng.stream), "slm_gram_blocks")
    else:
        out.t.copy_(torch.from_numpy(G0.ravel()))
        eng._ck(eng.lib.slm_gram_block_add(eng.h, eng._ptr(Xd), pa, int(row_ptr[0]), int(row_ptr[1]), out.ptr,
                                           eng.stream), "slm_gram_block_add")
    return out.fetch()


@pytest.mark.parametrize("sid,feed", SYRK_CASES)
def test_gram_build_shape(eng, sid, feed):
    eng.set_option("tma", feed)
    eng.set_option("force_syrk_shape", sid)
    try:
        for pa, kind in [(8, "blocks"), (128, "blocks"), (136, "blocks"), (8, "add"), (128, "add"), (136, "add"),
                         (8, "long")]:
            what = f"Gram build shape {sid} feed {feed} pa={pa} {kind}"
            for ints in (True, False):
                Xa, row_ptr, ref, bound, G0 = _syrk_data(pa, kind, ints)
                F = len(row_ptr) - 1
                want = np.zeros((F, pa, pa))
                must = np.zeros((F, pa, pa), bool)
                bnd = np.zeros((F, pa, pa))
                for f in range(F):
                    if row_ptr[f + 1] > row_ptr[f]:  # an empty block leaves its Gram untouched
                        want[f] = ref[f] + (G0 if G0 is not None else 0.0)
                        must[f] = True
                        if bound is not None:
                            bnd[f] = bound[f] + (2 * EPS * np.abs(G0) if G0 is not None else 0.0)
                t0 = eng.tma_launch_count()
                got, kept = _run_syrk(eng, Xa, row_ptr, G0)
                _tma_check(eng, t0, feed != CP_ASYNC and sid <= 1, what)
                _check(got, kept, must.ravel(), np.zeros(must.size, bool), want.ravel(),
                       None if ints else bnd.ravel(), what + (" integers" if ints else " normal"))
                Gs = got.reshape(F, pa, pa)
                for f in range(F):
                    if must[f, 0, 0]:
                        assert np.array_equal(Gs[f], Gs[f].T), f"{what}: block {f} mirror differs from its upper tiles"
                if not ints:
                    again, _ = _run_syrk(eng, Xa, row_ptr, G0)
                    assert np.array_equal(got[must.ravel()], again[must.ravel()]), what + ": not bitwise reproducible"
    finally:
        eng.set_option("force_syrk_shape", -1)
        eng.set_option("tma", 15)


# ---- CV scoring: Yhat = Xa[rows, :p] B, residual sums and statistics -----------------------------------------------
SCORE_M = (1, 127, 128, 129, 1000)
N_XA = 1300


@functools.lru_cache(maxsize=16)
def _score_data(p, BN, ints):
    """Xa [N_XA][lda] (packed padding finite: y, ones, zeros) and 40 problems (two launches): every m of SCORE_M x
    every K of (1, 8, BN, BN + 1), twice with other rows; ldb = K + 1 for odd K (B rows end before the rounded-up N),
    B columns >= K NaN."""
    lda = _round_up(p + 2, 8)
    rng = np.random.default_rng([p, BN, int(ints)])
    Xa = np.zeros((N_XA, lda))
    Xa[:, :p + 1] = _ints(rng, (N_XA, p + 1)) if ints else rng.standard_normal((N_XA, p + 1))
    Xa[:, p + 1] = 1.0
    probs = []
    for rep in range(2):
        for m in SCORE_M:
            for K in (1, 8, BN, BN + 1):
                ldb = K + 1 if K % 2 else K + 8
                B = np.full((p, ldb), np.nan)
                B[:, :K] = _ints(rng, (p, K)) if ints else rng.standard_normal((p, K))
                r0 = int(rng.integers(0, N_XA - m + 1))
                rows = rng.permutation(N_XA)[:m]
                if m >= 2:
                    rows[:2] = [N_XA - 1, 0]
                probs.append(dict(m=m, K=K, ldb=ldb, B=B, r0=r0, rows=rows.astype(np.int32)))
    for pr in probs:
        for form, idx in (("range", np.arange(pr["r0"], pr["r0"] + pr["m"])), ("rows", pr["rows"])):
            A = Xa[idx]
            pred = A[:, :p] @ pr["B"][:, :pr["K"]]
            res = A[:, p:p + 1] - pred
            pr["ref_" + form] = dict(pred=pred, res=res, sse=(res * res).sum(0), sae=np.abs(res).sum(0),
                            amax=np.abs(res).max(0), med=np.median(np.abs(res), axis=0),
                            bound=None if ints else 2 * (p + 2) * EPS * (np.abs(A[:, :p]) @ np.abs(pr["B"][:, :pr["K"]])))
    return Xa, probs


def _run_score(eng, Xa, p, probs, form, stats):
    """one slm_cv_score_many / _rows (stats None) or slm_cv_score_stats call over every problem; returns, per
    problem, (yhat values, yhat kept mask, out values, out kept mask) with yhat [(m + 256)][ldy], out [nrow][ldy]."""
    n = len(probs)
    Xd = _dev(eng, Xa)
    Bs = [_dev(eng, np.concatenate([pr["B"].ravel(), np.full(16, np.nan)])) for pr in probs]  # a tail after B
    ldy = [_round_up(pr["K"], 8) + 8 for pr in probs]
    nrow = 2 if stats is None else 5
    yh = [Out(eng, (pr["m"] + 256) * ly) for pr, ly in zip(probs, ldy)]
    outs = [Out(eng, nrow * ly) for ly in ldy]
    i64, i32, vp = ctypes.c_int64 * n, ctypes.c_int32 * n, ctypes.c_void_p * n
    Bp = vp(*[b.data_ptr() for b in Bs])
    ldb = i64(*[pr["ldb"] for pr in probs])
    Kc = i32(*[pr["K"] for pr in probs])
    yp = vp(*[o.t.data_ptr() for o in yh])
    ldyc = i64(*ldy)
    op = vp(*[o.t.data_ptr() for o in outs])
    lda = Xa.shape[1]
    if form == "range":
        r0 = i64(*[pr["r0"] for pr in probs])
        r1 = i64(*[pr["r0"] + pr["m"] for pr in probs])
        rp = nr = None
    else:
        rows_d = [_dev(eng, pr["rows"]) for pr in probs]
        rp, nr = vp(*[r.data_ptr() for r in rows_d]), i64(*[pr["m"] for pr in probs])
        r0 = r1 = None
    if stats is not None:
        eng._ck(eng.lib.slm_cv_score_stats(eng.h, eng._ptr(Xd), lda, p, n, r0, r1, rp, nr, Bp, ldb, Kc, None, 0, stats,
                                           yp, ldyc, op, eng.stream), "slm_cv_score_stats")
    elif form == "range":
        eng._ck(eng.lib.slm_cv_score_many(eng.h, eng._ptr(Xd), lda, p, n, r0, r1, Bp, ldb, Kc, None, 0, yp, ldyc, op,
                                          eng.stream), "slm_cv_score_many")
    else:
        eng._ck(eng.lib.slm_cv_score_rows(eng.h, eng._ptr(Xd), lda, p, n, rp, nr, Bp, ldb, Kc, None, 0, yp, ldyc, op,
                                          eng.stream), "slm_cv_score_rows")
    return [(*y.fetch(), *o.fetch(), ly) for y, o, ly in zip(yh, outs, ldy)]


@pytest.mark.parametrize("form", ["range", "rows"])
@pytest.mark.parametrize("sid", range(len(SCORE_MENU)), ids=lambda s: f"s{s:02d}")
def test_score_shape(eng, sid, form):
    from sparselm_b200._lib import SLM_STAT_MAX, SLM_STAT_MEDIAN

    BM, BN, MINB = SCORE_MENU[sid]
    eng.set_option("force_score_shape", sid)
    try:
        for p in (17, 47):  # last slab of 1 / 15 rows
            for ints in (True, False):
                Xa, probs = _score_data(p, BN, ints)
                for stats in ((None, SLM_STAT_MAX | SLM_STAT_MEDIAN) if ints else (None,)):
                    res = _run_score(eng, Xa, p, probs, form, stats)
                    if not ints:
                        again = _run_score(eng, Xa, p, probs, form, stats)
                        for i, ((yv, yk, *_), (yv2, *_)) in enumerate(zip(res, again)):
                            assert np.array_equal(yv, yv2, equal_nan=True), \
                                f"score shape {sid} {form} problem {i}: not bitwise reproducible"
                    for i, (pr, (yv, ykeep, ov, okeep, ldy)) in enumerate(zip(probs, res)):
                        m, K = pr["m"], pr["K"]
                        N = _round_up(K, 8)
                        ref = pr["ref_" + form]
                        what = (f"score shape {sid} {form} p={p} problem {i} m={m} K={K} ldb={pr['ldb']} "
                                f"stats={stats} {'integers' if ints else 'normal'}")
                        # yhat scratch: predictions (residuals with stats) in [0, m) x [0, K), partial sums in rows
                        # [m, m + 256) x [0, K); columns [K, N) free; columns >= N untouched
                        Y = np.zeros((m + 256, ldy))
                        must = np.zeros((m + 256, ldy), bool)
                        free = np.zeros((m + 256, ldy), bool)
                        Y[:m, :K] = ref["pred"] if stats is None else ref["res"]
                        must[:m, :K] = True
                        free[:, K:N] = True
                        free[m:, :K] = True
                        bnd = None
                        if ref["bound"] is not None:
                            bnd = np.zeros((m + 256, ldy))
                            bnd[:m, :K] = ref["bound"]
                        _check(yv, ykeep, must.ravel(), free.ravel(), Y.ravel(), None if bnd is None else bnd.ravel(),
                               what + " yhat")
                        if not ints:
                            continue
                        nrow = 2 if stats is None else 5
                        O = np.zeros((nrow, ldy))
                        omust = np.zeros((nrow, ldy), bool)
                        O[0, :K], O[1, :K] = ref["sse"], ref["sae"]
                        omust[:2, :K] = True
                        if stats is not None:
                            O[2, :K], O[4, :K] = ref["amax"], ref["med"]
                            omust[[2, 4], :K] = True
                        _check(ov, okeep, omust.ravel(), np.zeros(omust.size, bool), O.ravel(), None, what + " out")
    finally:
        eng.set_option("force_score_shape", -1)

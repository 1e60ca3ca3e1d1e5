"""The kernels before and after the solver loop, through the C entry points, against float64 references at their
edges (references: tests/aux_reference.py).

Every number a fit returns passes through these kernels: the design packing, the fold complements of the Gram
blocks (single-GPU and row-sharded forms), centring, the overlap gather and fold-back, intercepts, the adaptive
reweighting, the Lipschitz power iteration, the standardize=True whitening and the conjugate gradients of the
unpenalised columns.  The sizes sit on each kernel's own boundaries: the 65 535-row grid chunks of the pack, the
256-wide column blocks of the triangle, centring and gather kernels, the 64 group lanes and 4-column blocks of the
adaptive kernel, the 128 row lanes of the power iteration, the 256 threads of the group Cholesky and the 1024-thread
stride of CG.

Outputs start as a NaN payload (or, for in-place kernels, as values that must survive), inside NaN guards, and the
Python wrappers, which zero-fill their outputs, are bypassed: a missing store fails as a NaN, a stray store as changed
bits.  Kernels whose arithmetic is copies, single roundings or ordered sums without products must match a numpy
reference that does the same operations in the same order bit for bit; reductions over products (which nvcc may
contract into FMAs) must stay within the standard bound gamma_k * sum |terms|.
"""

import ctypes
import math

import numpy as np
import pytest

import aux_reference as A

pytestmark = pytest.mark.gpu

NAN_BITS = 0x7FF8DEADBEEF0A5A  # quiet NaN with a payload no arithmetic produces
GUARD = 64  # doubles of NaN guard before and after every output
U = A.U


def _nan(shape):
    return np.full(shape, NAN_BITS, dtype=np.int64).view(np.float64)


def _round_up(x, m):
    return (x + m - 1) // m * m


class Buf:
    """`size` doubles on the device between two NaN guards, filled with the NaN payload or with `init`."""

    def __init__(self, eng, size, init=None):
        import torch

        self.size = int(size)
        self.buf = torch.full((self.size + 2 * GUARD,), NAN_BITS, dtype=torch.int64, device=eng.device)
        self.t = self.buf[GUARD:GUARD + self.size].view(torch.float64)
        if init is not None:
            self.t.copy_(torch.from_numpy(np.ascontiguousarray(init, dtype=np.float64).reshape(-1)))

    @property
    def ptr(self):
        return ctypes.c_void_p(self.t.data_ptr())

    def fetch(self):
        bits = self.buf.cpu().numpy()
        assert (bits[:GUARD] == NAN_BITS).all() and (bits[GUARD + self.size:] == NAN_BITS).all(), \
            "a store landed outside the output"
        return bits[GUARD:GUARD + self.size].view(np.float64).copy()


def _dev(eng, a, dtype=None):
    import torch

    a = np.ascontiguousarray(a if dtype is None else np.asarray(a, dtype=dtype))
    return torch.from_numpy(a).to(eng.device)


def _ok(eng, rc, what):
    assert rc == 0, f"{what} returned {rc}: {eng.lib.slm_last_error(eng.h)}"


def _bits_equal(got, want, what):
    """Bitwise equality of the whole array (NaN payloads included: untouched entries must keep theirs)."""
    g = np.asarray(got).reshape(-1).view(np.int64)
    w = np.ascontiguousarray(want, dtype=np.float64).reshape(-1).view(np.int64)
    bad = g != w
    assert not bad.any(), f"{what}: {int(bad.sum())} of {g.size} entries differ (first at {int(np.argmax(bad))})"


def _within(got, want, bound, must, what):
    """Entries in `must` within `bound` of `want`; every other entry kept the NaN payload."""
    got = np.asarray(got).reshape(want.shape)
    must = np.broadcast_to(must, want.shape)
    keep = got[~must].view(np.int64) == NAN_BITS
    assert keep.all(), f"{what}: {int((~keep).sum())} stray stores"
    g, w, b = got[must], want[must], np.broadcast_to(bound, want.shape)[must]
    assert np.isfinite(g).all(), f"{what}: {int((~np.isfinite(g)).sum())} entries not written or not finite"
    bad = np.abs(g - w) > b
    assert not bad.any(), f"{what}: {int(bad.sum())} of {g.size} entries outside the bound " \
                          f"(worst excess ratio {float(np.max(np.abs(g - w) / np.maximum(b, 1e-300))):.3g})"


def _augmented(X, y, sw=None, pad_fill=None, rng=None):
    """Gram of the augmented design [sqrt(sw) X | sqrt(sw) y | sqrt(sw) | 0] (pa x pa), padding rows and columns
    replaced by pad_fill ("nan", "random" or None = the zeros of a real Gram)."""
    n, p = X.shape
    pa = _round_up(p + 2, 8)
    s = np.ones(n) if sw is None else np.sqrt(sw)
    Xa = np.zeros((n, pa))
    Xa[:, :p], Xa[:, p], Xa[:, p + 1] = s[:, None] * X, s * y, s
    G = Xa.T @ Xa
    if pad_fill == "nan":
        G[p + 2:, :] = G[:, p + 2:] = np.nan
    elif pad_fill == "random":
        G[p + 2:, :] = rng.standard_normal((pa - p - 2, pa))
        G[:, p + 2:] = rng.standard_normal((pa, pa - p - 2))
    return G


# ---- K1: design packing across the 65 535-row grid chunks ----------------------------------------------------------
N_PACK = 2 * 65535 + 3
PACK_EDGE_ROWS = [65534, 65535, 65536, 131069, 131070, 131071, 131072]


@pytest.mark.parametrize("wide", [False, True], ids=["lda_padded", "lda_wide_col_perm"])
@pytest.mark.parametrize("weighted", [False, True], ids=["unweighted", "sw"])
@pytest.mark.parametrize("permuted", [False, True], ids=["rows", "row_perm"])
def test_pack_design_across_row_chunks(engine, permuted, weighted, wide):
    """Three grid chunks of rows (65 535, 65 535, 3): with row_perm the chunk offset goes into the permutation,
    without it into X, y and sw.  Bitwise: one square root and one product per entry."""
    rng = np.random.default_rng(100 + 4 * permuted + 2 * weighted + wide)
    n, p, ldx = N_PACK, 5, 7
    Xfull = rng.standard_normal((n, ldx))
    y = rng.standard_normal(n)
    sw = 0.1 + 3.0 * rng.random(n) if weighted else None
    cp = rng.permutation(p).astype(np.int32) if wide else None
    rp = rng.permutation(n).astype(np.int64) if permuted else None
    lda = int(engine.lib.slm_padded_cols(p)) + (6 if wide else 0)
    Xd, yd = _dev(engine, Xfull), _dev(engine, y)
    swd = None if sw is None else _dev(engine, sw)
    cpd = None if cp is None else _dev(engine, cp)
    rpd = None if rp is None else _dev(engine, rp)
    out = Buf(engine, n * lda)
    _ok(engine, engine.lib.slm_pack_design(engine.h, engine._ptr(Xd), ldx, engine._ptr(yd), engine._ptr(swd),
                                           engine._ptr(cpd), engine._ptr(rpd), n, p, out.ptr, lda, engine.stream),
        "slm_pack_design")
    ri = rp if permuted else np.arange(n)
    ci = cp if wide else np.arange(p)
    s = np.sqrt(sw[ri]) if weighted else np.ones(n)
    want = np.zeros((n, lda))
    want[:, :p] = s[:, None] * Xfull[ri][:, ci]
    want[:, p] = s * y[ri]
    want[:, p + 1] = s
    got = out.fetch().reshape(n, lda)
    for r in PACK_EDGE_ROWS:
        _bits_equal(got[r], want[r], f"row {r}")
    _bits_equal(got, want, "packed design")


# ---- complements of the fold blocks ---------------------------------------------------------------------------------
@pytest.mark.parametrize("F", [1, 2, 15, 16])
def test_gram_complement_ordered_sums(engine, F):
    """Total = 0.0 + G_0 + G_1 + ..., complement f = ascending sum over g != f (0 for F = 1), bit for bit on blocks
    where any other order changes bits."""
    rng = np.random.default_rng(200 + F)
    pa = 40  # 1600 entries: a partial last block of 256 threads
    blocks = A.mixed_magnitudes(rng, (F, pa, pa))
    gb = Buf(engine, F * pa * pa, init=blocks)
    gt = Buf(engine, pa * pa)
    _ok(engine, engine.lib.slm_gram_complement(engine.h, gb.ptr, F, pa, gt.ptr, engine.stream), "slm_gram_complement")
    _bits_equal(gt.fetch(), A.ordered_total(blocks), "total")
    _bits_equal(gb.fetch(), np.stack(A.ordered_complements(list(blocks))), "complements")


def test_gram_complement_rejects_17_blocks(engine):
    rng = np.random.default_rng(217)
    pa, F = 8, 17
    blocks = rng.standard_normal((F, pa, pa))
    gb = Buf(engine, F * pa * pa, init=blocks)
    gt = Buf(engine, pa * pa)
    assert engine.lib.slm_gram_complement(engine.h, gb.ptr, F, pa, gt.ptr, engine.stream) != 0
    _bits_equal(gb.fetch(), blocks, "blocks of a rejected call")
    _bits_equal(gt.fetch(), _nan(pa * pa), "total of a rejected call")


# ---- row-sharded form: packed upper triangles -----------------------------------------------------------------------
@pytest.mark.parametrize("nb", [1, 2, 5, 15, 16])
@pytest.mark.parametrize("pa", [8, 40, 256, 264, 1032])
def test_triangle_path_matches_single_gpu_complement(engine, pa, nb):
    """slm_tri_pack = G[triu], slm_tri_unpack restores G, slm_tri_complement writes the nb complements and the total
    as full, exactly symmetric matrices with the ordered sums of the single-GPU kernel, and slm_gram_allreduce on one
    rank (NULL communicator) equals slm_gram_complement bit for bit.  Outputs with a gap between the matrices
    (g_stride > pa * pa) check that nothing lands between them."""
    rng = np.random.default_rng(300 + pa + nb)
    half = A.mixed_magnitudes(rng, (nb, pa, pa))
    blocks = half + half.transpose(0, 2, 1)
    tri = int(engine.lib.slm_tri_size(pa))
    assert tri == pa * (pa + 1) // 2
    iu = np.triu_indices(pa)
    Gd = _dev(engine, blocks)
    buf = Buf(engine, nb * tri)
    _ok(engine, engine.lib.slm_tri_pack(engine.h, engine._ptr(Gd), pa * pa, pa, nb, buf.ptr, engine.stream),
        "slm_tri_pack")
    packed = buf.fetch()
    _bits_equal(packed, blocks[:, iu[0], iu[1]], "packed triangles")

    gs = pa * pa + 8
    un = Buf(engine, nb * gs)
    _ok(engine, engine.lib.slm_tri_unpack(engine.h, buf.ptr, pa, nb, un.ptr, gs, engine.stream), "slm_tri_unpack")
    want = _nan((nb, gs))
    want[:, :pa * pa] = blocks.reshape(nb, -1)
    _bits_equal(un.fetch(), want, "unpacked Grams")

    ref = np.stack(A.ordered_complements(list(blocks)) + [A.ordered_total(blocks)])
    tc = Buf(engine, (nb + 1) * gs)
    _ok(engine, engine.lib.slm_tri_complement(engine.h, buf.ptr, pa, nb, tc.ptr, gs, engine.stream),
        "slm_tri_complement")
    got = tc.fetch().reshape(nb + 1, gs)
    want = _nan((nb + 1, gs))
    want[:, :pa * pa] = ref.reshape(nb + 1, -1)
    _bits_equal(got, want, "training Grams and total from the packed triangles")
    mats = got[:, :pa * pa].reshape(nb + 1, pa, pa)
    assert np.array_equal(mats.view(np.int64), mats.transpose(0, 2, 1).view(np.int64)), "not exactly symmetric"

    ar = Buf(engine, (nb + 1) * pa * pa, init=np.concatenate([blocks.reshape(-1), np.zeros(pa * pa)]))
    abuf = Buf(engine, nb * tri)
    _ok(engine, engine.lib.slm_gram_allreduce(engine.h, None, ar.ptr, pa * pa, pa, nb, abuf.ptr, engine.stream),
        "slm_gram_allreduce")
    gc = Buf(engine, nb * pa * pa, init=blocks)
    gt = Buf(engine, pa * pa)
    _ok(engine, engine.lib.slm_gram_complement(engine.h, gc.ptr, nb, pa, gt.ptr, engine.stream), "slm_gram_complement")
    sharded = ar.fetch()
    _bits_equal(sharded, np.concatenate([gc.fetch(), gt.fetch()]), "sharded vs single-GPU training Grams")
    _bits_equal(sharded, ref, "sharded training Grams vs the ordered sums")


@pytest.mark.parametrize("nb", [0, 17])
def test_triangle_path_rejects_block_counts(engine, nb):
    pa = 8
    tri = int(engine.lib.slm_tri_size(pa))
    slots = max(nb, 1) + 1
    G = Buf(engine, slots * pa * pa, init=np.arange(slots * pa * pa, dtype=np.float64))
    buf = Buf(engine, slots * tri, init=np.ones(slots * tri))
    assert engine.lib.slm_tri_complement(engine.h, buf.ptr, pa, nb, G.ptr, pa * pa, engine.stream) != 0
    assert engine.lib.slm_gram_allreduce(engine.h, None, G.ptr, pa * pa, pa, nb, buf.ptr, engine.stream) != 0
    _bits_equal(G.fetch(), np.arange(slots * pa * pa, dtype=np.float64), "Grams of a rejected call")
    _bits_equal(buf.fetch(), np.ones(slots * tri), "buffer of a rejected call")


# ---- centring --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("weighted", [False, True], ids=["integer_n", "weighted_n"])
@pytest.mark.parametrize("p", [254, 255, 256])
def test_gram_center_is_one_rank_one_update(engine, p, weighted):
    """G[:p+1, :p+1] - outer(s, s) / n with s the ones row, n = its last entry (sum of the weights): one product,
    one division and one subtraction per entry, bit for bit.  p + 1 = 255, 256, 257 rows and columns around a
    256-wide block; the ones row and column and the padding keep their bits."""
    rng = np.random.default_rng(400 + p + weighted)
    n = 300
    X = rng.standard_normal((n, p)) + 2.0
    y = rng.standard_normal(n) + 5.0
    sw = 0.2 + rng.random(n) if weighted else None
    G = _augmented(X, y, sw, pad_fill="random", rng=rng)
    pa = G.shape[0]
    nn = G[p + 1, p + 1]
    assert (nn == n) != weighted
    gb = Buf(engine, pa * pa, init=G)
    _ok(engine, engine.lib.slm_gram_center(engine.h, gb.ptr, pa, p, engine.stream), "slm_gram_center")
    s = G[p + 1, :p + 1]
    want = G.copy()
    want[:p + 1, :p + 1] = G[:p + 1, :p + 1] - np.outer(s, s) / nn
    _bits_equal(gb.fetch(), want, "centred Gram")


# ---- overlap gather and fold-back ------------------------------------------------------------------------------------
@pytest.mark.parametrize("padded", [False, True], ids=["pae_pe_plus_2", "pae_padded"])
def test_gram_gather_unsorted_repeats(engine, padded):
    """Ge[a][b] = G[idx[a]][idx[b]], then the y and ones rows and columns, zeros beyond pe + 2: pe = 601 spans three
    256-wide column blocks.  G's padding is NaN, so a read outside the gathered rows shows."""
    rng = np.random.default_rng(500 + padded)
    p, pe = 250, 601
    X = rng.standard_normal((400, p))
    G = _augmented(X, rng.standard_normal(400), pad_fill="nan")
    pa = G.shape[0]
    idx = rng.integers(0, p, size=pe).astype(np.int32)
    pae = int(engine.lib.slm_padded_cols(pe)) if padded else pe + 2
    Gd, idd = _dev(engine, G), _dev(engine, idx)
    out = Buf(engine, pae * pae)
    _ok(engine, engine.lib.slm_gram_gather(engine.h, engine._ptr(Gd), pa, p, engine._ptr(idd), pe, out.ptr, pae,
                                           engine.stream), "slm_gram_gather")
    full = np.concatenate([idx, [p, p + 1]])
    want = np.zeros((pae, pae))
    want[:pe + 2, :pe + 2] = G[np.ix_(full, full)]
    _bits_equal(out.fetch(), want, "gathered Gram")


@pytest.mark.parametrize("K", [1, 128, 129, 300])
def test_fold_back_ordered_sums(engine, K):
    """coef[j] = ascending sum over the copies of feature j (0, 1, 2 or 7 of them, scattered through an unsorted
    extended order), bit for bit; K = 128 / 129 / 300 around the 128-column blocks, columns >= K keep their NaN."""
    rng = np.random.default_rng(600 + K)
    p = 40
    copies = rng.permutation(np.resize([0, 1, 2, 7], p))
    idx = np.repeat(np.arange(p), copies)
    rng.shuffle(idx)
    pe = len(idx)
    inv_ptr = np.concatenate([[0], np.cumsum(np.bincount(idx, minlength=p))]).astype(np.int32)
    inv_idx = np.argsort(idx, kind="stable").astype(np.int32)
    ldz = _round_up(K, 8) + 8
    Be = _nan((pe, ldz))
    Be[:, :K] = A.mixed_magnitudes(rng, (pe, K))
    Bd, ipd, iid = _dev(engine, Be), _dev(engine, inv_ptr), _dev(engine, inv_idx)
    out = Buf(engine, p * ldz)
    _ok(engine, engine.lib.slm_fold_back(engine.h, engine._ptr(Bd), engine._ptr(ipd), engine._ptr(iid), p, ldz, K,
                                         out.ptr, engine.stream), "slm_fold_back")
    want = _nan((p, ldz))
    want[:, :K] = A.fold_back(Be, inv_ptr, inv_idx, p, K)
    _bits_equal(out.fetch(), want, "folded-back coefficients")


# ---- intercepts ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("weighted", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("K", [1, 8, 9, 130])
@pytest.mark.parametrize("p", [1, 31, 32, 33, 1000])
def test_intercepts_within_dot_bound(engine, p, K, weighted):
    """intercept[k] = (ones[p] - ones[:p] . B[:, k]) / n from the ones row of the Gram, within
    gamma_{p+2} (|ones[p]| + sum |ones_j B_jk|) / n of the exact value.  Only the ones row may be read (every other
    Gram row is NaN); entries >= K keep their NaN."""
    rng = np.random.default_rng(700 + p + 7 * K + weighted)
    n = p + 50
    X = rng.standard_normal((n, p)) + 1.5
    y = rng.standard_normal(n) + 3.0
    sw = 0.3 + rng.random(n) if weighted else None
    G = _augmented(X, y, sw)
    pa = G.shape[0]
    G[:p + 1, :] = np.nan
    G[p + 2:, :] = np.nan
    G[p + 1, p + 2:] = np.nan
    ldz = _round_up(K, 8) + 8
    B = _nan((p, ldz))
    B[:, :K] = rng.standard_normal((p, K))
    Gd, Bd = _dev(engine, G), _dev(engine, B)
    out = Buf(engine, ldz)
    _ok(engine, engine.lib.slm_intercepts(engine.h, engine._ptr(Gd), pa, p, engine._ptr(Bd), ldz, K, out.ptr,
                                          engine.stream), "slm_intercepts")
    ones = G[p + 1]
    nn = ones[p + 1]
    want, bound = np.zeros(ldz), np.zeros(ldz)
    for k in range(K):
        terms = ones[:p] * B[:, k]
        d = math.fsum(terms)
        want[k] = (ones[p] - d) / nn
        bound[k] = A.gamma(p + 2) * (abs(ones[p]) + np.abs(terms).sum()) / abs(nn) + 2 * U * abs(want[k])
    _within(out.fetch(), want, bound, np.arange(ldz) < K, "intercepts")


# ---- adaptive reweighting --------------------------------------------------------------------------------------------
ADAPTIVE_NULLS = ["none", "a1", "a2", "gw", "all"]


@pytest.mark.parametrize("nulls", ADAPTIVE_NULLS)
@pytest.mark.parametrize("K", [1, 3, 4, 5])
@pytest.mark.parametrize("form", ["lasso", "group", "sparse_group"])
def test_adaptive_update(engine, form, K, nulls):
    """W1[j][k] = a1[k] (alpha[k] / (|B[j][k]| + eps)) bit for bit; W2[g][k] = (a2[k] gw[g]) (alpha[k] /
    (||B_g[:, k]|| + eps)) and dnorm[k] = ||new - old|| within their bounds.  Lasso form: no group pointer,
    Gn = p = 300 rows over 64 group lanes; group forms: 150 groups of 1 to 40 rows.  K = 1, 3, 4, 5 around the
    4-column blocks; zero coefficients and an all-zero group; a1 / a2 / gw NULL (= 0, 0, 1) in turn."""
    rng = np.random.default_rng(800 + 10 * K + ADAPTIVE_NULLS.index(nulls) + 100 * len(form))
    if form == "lasso":
        p = Gn = 300
        gptr = None
        sizes = np.ones(p, dtype=np.int64)
    else:
        Gn = 150
        sizes = rng.integers(1, 41, size=Gn)
        sizes[:2] = [1, 40]
        gptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
        p = int(gptr[-1])
    has_w1, has_w2 = form != "group", form != "lasso"
    ldz = 16
    B = _nan((p, ldz))
    B[:, :K] = rng.standard_normal((p, K)) * np.where(rng.random((p, K)) < 0.2, 0.0, 1.0)
    starts = np.concatenate([[0], np.cumsum(sizes)])
    g0 = Gn // 2
    B[starts[g0]:starts[g0 + 1], :K] = 0.0  # an all-zero group (a zero coefficient in the lasso form)
    alpha = 0.1 + rng.random(K)
    a1 = None if nulls in ("a1", "all") else 0.5 + rng.random(K)
    a2 = None if nulls in ("a2", "all") else 0.5 + rng.random(K)
    gw = None if nulls in ("gw", "all") else 0.5 + rng.random(Gn)
    eps = 1e-6
    W1_old = _nan((p, ldz))
    W1_old[:, :K] = rng.random((p, K))
    W2_old = _nan((Gn, ldz))
    W2_old[:, :K] = 10.0 * rng.random((Gn, K))

    Bd = _dev(engine, B)
    dv = {nm: (None if v is None else _dev(engine, v)) for nm, v in
          (("gptr", gptr), ("gw", gw), ("a1", a1), ("a2", a2), ("alpha", alpha))}
    W1 = Buf(engine, p * ldz, init=W1_old) if has_w1 else None
    W2 = Buf(engine, Gn * ldz, init=W2_old) if has_w2 else None
    dn = Buf(engine, ldz)
    P = engine._ptr
    _ok(engine, engine.lib.slm_adaptive_update(engine.h, P(Bd), p, ldz, K, Gn, P(dv["gptr"]), P(dv["gw"]), P(dv["a1"]),
                                               P(dv["a2"]), P(dv["alpha"]), eps, W1.ptr if W1 else None,
                                               W2.ptr if W2 else None, dn.ptr, engine.stream), "slm_adaptive_update")

    s1 = np.zeros(K) if a1 is None else a1
    s2 = np.zeros(K) if a2 is None else a2
    gwv = np.ones(Gn) if gw is None else gw
    d_sq = [[] for _ in range(K)]  # squared differences and their error bounds, per column
    d_err = [[] for _ in range(K)]
    if has_w1:
        want1 = W1_old.copy()
        want1[:, :K] = s1[None, :] * (alpha[None, :] / (np.abs(B[:, :K]) + eps))
        _bits_equal(W1.fetch(), want1, "W1")
        d1 = want1[:, :K] - W1_old[:, :K]
        for k in range(K):
            d_sq[k].append(d1[:, k] ** 2)
            d_err[k].append(np.zeros(p))
    if has_w2:
        want2 = W2_old.copy()
        bound2 = np.zeros((Gn, ldz))
        for g in range(Gn):
            a, b = starts[g], starts[g + 1]
            for k in range(K):
                nrm = math.sqrt(math.fsum(B[a:b, k] ** 2))
                want2[g, k] = (s2[k] * gwv[g]) * (alpha[k] / (nrm + eps))
                bound2[g, k] = A.gamma(b - a + 10) * abs(want2[g, k])
        _within(W2.fetch(), want2, bound2, np.arange(ldz)[None, :] < K, "W2")
        d2 = want2[:, :K] - W2_old[:, :K]
        for k in range(K):
            d_sq[k].append(d2[:, k] ** 2)
            d_err[k].append(bound2[:, k] + 2 * U * np.abs(d2[:, k]))
    want_dn, bound_dn = np.zeros(ldz), np.zeros(ldz)
    for k in range(K):
        sq = np.concatenate(d_sq[k])
        want_dn[k] = math.sqrt(math.fsum(sq))
        bound_dn[k] = np.sqrt(np.sum(np.concatenate(d_err[k]) ** 2)) + A.gamma(sq.size + 4) * want_dn[k]
    _within(dn.fetch(), want_dn, bound_dn, np.arange(ldz) < K, "dnorm")


# ---- Lipschitz constants: block power iteration ----------------------------------------------------------------------
LIPS_P = [1, 7, 8, 127, 128, 129, 1000]


def _spectra(rng, p, count=16):
    """`count` Grams p x p with different spectra: all-zero, rank one, spike over a flat bulk, Gaussian Grams of
    n < p and n > p rows over 16 orders of magnitude, a graded diagonal."""
    out = [np.zeros((p, p))]
    v = rng.standard_normal(p)
    out.append(np.outer(v, v))
    Xs = A.spike_over_bulk(int(rng.integers(1 << 30)), p + 10, p, 0.8)
    out.append(Xs.T @ Xs)
    out.append(np.diag(np.geomspace(1.0, 1e-6, p)[rng.permutation(p)]))
    f = len(out)
    while len(out) < count:
        n = max(1, p // 2 + 7 * f) if f % 2 else p + 3 * f
        X = rng.standard_normal((n, p)) * 10.0 ** (f - 9)
        out.append(X.T @ X)
        f += 1
    return out


@pytest.mark.parametrize("p", LIPS_P)
def test_lipschitz_matches_power_iteration_emulation(engine, p):
    """16 Grams in one call: every lambda equals the CPU emulation of the block power iteration (start vectors of
    Gram f of the call, largest Rayleigh quotient over columns and iterations) to 1e-12 and is a lower bound of
    lambda_max; slm_lipschitz_dev returns the same bits on the device.  The Grams' unused rows and columns are NaN."""
    rng = np.random.default_rng(900 + p)
    grams = _spectra(rng, p)
    nf = len(grams)
    pa = int(engine.lib.slm_padded_cols(p))
    G = np.full((nf, pa, pa), np.nan)
    for f, g in enumerate(grams):
        G[f, :p, :p] = g
    Gd = _dev(engine, G)
    iters = engine.LIPSCHITZ_ITERS
    nbytes = engine.lib.slm_lipschitz_workspace(p, nf)
    import torch

    work = torch.empty(nbytes, dtype=torch.uint8, device=engine.device)
    lam = (ctypes.c_double * nf)()
    _ok(engine, engine.lib.slm_lipschitz(engine.h, engine._ptr(Gd), pa * pa, pa, p, nf, iters, engine._ptr(work), lam,
                                         engine.stream), "slm_lipschitz")
    lam = np.frombuffer(lam, dtype=np.float64, count=nf).copy()
    for f, g in enumerate(grams):
        emu = A.power_lambda(g, iters, f)
        top = np.linalg.eigvalsh(g)[-1] if f else 0.0
        assert abs(lam[f] - emu) <= 1e-12 * emu, (f, lam[f], emu)
        assert lam[f] <= max(top, 0.0) * (1 + 1e-12), (f, lam[f], top)
    assert lam[0] == 0.0
    out = Buf(engine, nf)
    _ok(engine, engine.lib.slm_lipschitz_dev(engine.h, engine._ptr(Gd), pa * pa, pa, p, nf, iters, engine._ptr(work),
                                             out.ptr, engine.stream), "slm_lipschitz_dev")
    _bits_equal(out.fetch(), lam, "slm_lipschitz_dev vs slm_lipschitz")


def test_lasso_converges_with_underestimated_lipschitz(engine):
    """On a spike over a flat bulk (Gram eigenvalues n and 0.8 n) the power iteration's estimate times the 1.10
    margin stays below lambda_max; the Lasso grid still converges to the oracle's solutions."""
    import oracle.reference as R
    from sparselm_b200.engine import PenaltyGrid

    rng = np.random.default_rng(1000)
    n, p = 1200, 1000
    X = A.spike_over_bulk(1000, n, p, 0.8)
    w = np.zeros(p)
    w[rng.choice(p, 30, replace=False)] = 2.0 * rng.standard_normal(30)
    y = X @ w + 0.5 * rng.standard_normal(n)
    lam_max = np.linalg.eigvalsh(X.T @ X)[-1]
    fd = engine.prepare(X, y)
    L = fd.lipschitz(engine, "full")
    assert L * n < lam_max, (L * n, lam_max)  # the step size 1/L is longer than 1/lambda_max
    amax = np.abs(X.T @ y).max() / n
    alphas = amax * np.geomspace(0.5, 0.005, 6)
    grid = PenaltyGrid(p=p, lam1=alphas)
    res = engine.solve(fd.G_full[None], p, [n], [L], [grid], tol=1e-12)
    assert (res["status"][0, :grid.K] == 0).all(), res["status"]
    B = res["B"][0].cpu().numpy()
    labels = np.arange(p)
    for k, a in enumerate(alphas):
        pen = R.Penalty(labels, np.full(p, a), np.zeros(p), np.zeros(p))
        b_ref, _ = R.solve(X, y, pen, tol=1e-14)
        assert np.abs(B[:, k] - b_ref).max() <= 1e-6 * np.abs(b_ref).max(), (k, np.abs(B[:, k] - b_ref).max())
        obj, obj_ref = R.objective(X, y, B[:, k], pen), R.objective(X, y, b_ref, pen)
        assert abs(obj - obj_ref) <= 1e-8 * abs(obj_ref), (k, obj, obj_ref)


# ---- standardize=True: group whitening -------------------------------------------------------------------------------
def _whiten(engine, G, p, gptr, shift=None, ridge=None, ridge_scale=0.0):
    """slm_group_whiten_factors + slm_gram_whiten on one Gram: (W blocks, R blocks, info, Gout, wptr)."""
    import torch

    pa = G.shape[0]
    sizes = np.diff(gptr)
    wptr = np.concatenate([[0], np.cumsum(sizes * sizes)]).astype(np.int64)
    Gd, gpd, wpd = _dev(engine, G), _dev(engine, gptr, np.int32), _dev(engine, wptr)
    shd = None if shift is None else _dev(engine, shift, np.float64)
    rdd = None if ridge is None else _dev(engine, ridge, np.float64)
    W, Rs = Buf(engine, wptr[-1]), Buf(engine, wptr[-1])
    info = torch.zeros(1, dtype=torch.int32, device=engine.device)
    Gn = len(gptr) - 1
    P = engine._ptr
    _ok(engine, engine.lib.slm_group_whiten_factors(engine.h, P(Gd), pa, p, P(gpd), P(wpd), Gn, P(shd), W.ptr, Rs.ptr,
                                                    P(info), engine.stream), "slm_group_whiten_factors")
    tmp = torch.empty((pa, pa), dtype=torch.float64, device=engine.device)
    out = Buf(engine, pa * pa)
    _ok(engine, engine.lib.slm_gram_whiten(engine.h, P(Gd), pa, p, P(gpd), P(wpd), Gn, W.ptr, P(rdd),
                                           float(ridge_scale), P(tmp), out.ptr, engine.stream), "slm_gram_whiten")
    w, r = W.fetch(), Rs.fetch()
    Wb = [w[wptr[g]:wptr[g + 1]].reshape(sizes[g], sizes[g]) for g in range(Gn)]
    Rb = [np.triu(r[wptr[g]:wptr[g + 1]].reshape(sizes[g], sizes[g])) for g in range(Gn)]
    return Wb, Rb, int(info.item()), out.fetch().reshape(pa, pa), (gpd, wpd, W)


def _check_factors(Wb, Rb, blocks, what):
    """R^T R = A within the Cholesky backward-error bound gamma_{m+1} |R|^T |R| (doubled for the rounding of the
    check's own product); W = R^{-1} upper triangular with W^T A W = I within 4 (m + 2) u kappa(A)."""
    for g, (Wg, Rg, Ag) in enumerate(zip(Wb, Rb, blocks)):
        m = Ag.shape[0]
        assert np.isfinite(Wg).all(), f"{what}: group {g}: W not written"
        assert (np.tril(Wg, -1) == 0).all(), f"{what}: group {g}: W not upper triangular"
        bwd = np.abs(Rg.T @ Rg - Ag)
        assert (bwd <= 2 * A.gamma(m + 2) * (np.abs(Rg).T @ np.abs(Rg))).all(), f"{what}: group {g}: R^T R != A"
        kappa = np.linalg.cond(Ag)
        err = np.abs(Wg.T @ Ag @ Wg - np.eye(m)).max()
        assert err <= 4 * (m + 2) * U * kappa, f"{what}: group {g}: |W^T A W - I| = {err:.3g}, kappa {kappa:.3g}"


def _check_whitened(Gout, G, Wb, gptr, p, ridge, ridge_scale, what):
    """Gout = Wf^T G Wf (Wf = blockdiag(W_g) with the identity on rows >= p: the c row is whitened, the y, ones and
    padding rows copied) + ridge_scale ridge_g W_g^T W_g on the diagonal blocks, within 2 gamma_{2m+8} of the absolute
    products; the copied block [p:, p:] is bitwise G's."""
    pa = G.shape[0]
    Wf = np.eye(pa)
    Rf = np.zeros((pa, pa))  # the folded ridge
    Rs = np.zeros((pa, pa))  # its absolute products
    for g, Wg in enumerate(Wb):
        a, b = gptr[g], gptr[g + 1]
        Wf[a:b, a:b] = Wg
        if ridge is not None:
            Rf[a:b, a:b] = ridge_scale * ridge[g] * (Wg.T @ Wg)
            Rs[a:b, a:b] = ridge_scale * ridge[g] * (np.abs(Wg).T @ np.abs(Wg))
    want = Wf.T @ G @ Wf + Rf
    absw = np.abs(Wf)
    mmax = int(np.diff(gptr).max())
    scale = absw.T @ np.abs(G) @ absw + Rs
    _within(Gout, want, 2 * A.gamma(2 * mmax + 8) * scale, np.ones((pa, pa), dtype=bool), what)
    _bits_equal(Gout[p:, p:], G[p:, p:], f"{what}: copied y / ones / padding block")


def _check_unwhiten(engine, handles, Wb, gptr, p, what):
    """slm_coef_unwhiten with K = 130 columns of ldz = 136: B = blockdiag(W) Bg within gamma_{m+1} |W| |Bg|;
    columns >= K keep their NaN."""
    gpd, wpd, W = handles
    K, ldz = 130, 136
    rng = np.random.default_rng(p)
    Bg = _nan((p, ldz))
    Bg[:, :K] = rng.standard_normal((p, K))
    Bgd = _dev(engine, Bg)
    out = Buf(engine, p * ldz)
    _ok(engine, engine.lib.slm_coef_unwhiten(engine.h, engine._ptr(Bgd), p, ldz, K, engine._ptr(gpd), engine._ptr(wpd),
                                             len(gptr) - 1, W.ptr, out.ptr, engine.stream), "slm_coef_unwhiten")
    want, bound = np.zeros((p, ldz)), np.zeros((p, ldz))
    for g, Wg in enumerate(Wb):
        a, b = gptr[g], gptr[g + 1]
        want[a:b, :K] = Wg @ Bg[a:b, :K]
        bound[a:b, :K] = A.gamma(b - a + 2) * (np.abs(Wg) @ np.abs(Bg[a:b, :K]))
    _within(out.fetch(), want, bound, np.arange(ldz)[None, :] < K, f"{what}: unwhitened coefficients")


@pytest.mark.parametrize("case", ["one_group_300", "singletons_1500", "ridged"])
def test_group_whitening(engine, case):
    """Factors of a 300-row group (more rows than the 256 threads of the factorisation), of 1500 singleton groups
    (the group search over many groups) and of a ridged structure with shifted blocks and the ridge folded into the
    Gram at the scale n; the full pa x pa whitened Gram; coefficients back for 130 columns."""
    rng = np.random.default_rng(1100 + len(case))
    shift = ridge = None
    ridge_scale = 0.0
    if case == "one_group_300":
        p, n = 300, 700
        X = rng.standard_normal((n, p)) @ (np.eye(p) + 0.3 * rng.standard_normal((p, p)) / np.sqrt(p))
        gptr = np.array([0, p])
    elif case == "singletons_1500":
        p, n = 1500, 200
        X = rng.standard_normal((n, p)) * np.geomspace(0.1, 10.0, p)
        gptr = np.arange(p + 1)
    else:
        sizes = [3, 7, 1, 20, 5, 64]
        p = sum(sizes)
        n = 3 * p
        X = rng.standard_normal((n, p)) @ (np.eye(p) + 0.2 * rng.standard_normal((p, p)))
        gptr = np.concatenate([[0], np.cumsum(sizes)])
        dl = 0.1 + rng.random(len(sizes))
        shift, ridge, ridge_scale = np.sqrt(dl), dl, float(n)
    G = _augmented(X, rng.standard_normal(n) + 1.0, pad_fill="random", rng=rng)
    Wb, Rb, info, Gout, handles = _whiten(engine, G, p, gptr, shift, ridge, ridge_scale)
    assert info == 0
    blocks = [G[a:b, a:b] + (0.0 if shift is None else shift[g] * np.eye(b - a))
              for g, (a, b) in enumerate(zip(gptr[:-1], gptr[1:]))]
    _check_factors(Wb, Rb, blocks, case)
    _check_whitened(Gout, G, Wb, gptr, p, ridge, ridge_scale, case)
    _check_unwhiten(engine, handles, Wb, gptr, p, case)


@pytest.mark.parametrize("factor", [1.01, 0.99], ids=["pivot_above", "pivot_below"])
def test_group_whitening_pivot_threshold(engine, factor):
    """A block whose last pivot is 1.01 x or 0.99 x the threshold 1e-13 m max(diag): above it factors accurately
    and info stays 0; below it info counts the group (once, the other group is fine) and Engine.whiten raises
    ValueError.  The block is R0^T R0 with R0 = I plus 0.25 in row 0 and a small last diagonal entry, so every step of
    the factorisation but the last pivot's rounding is exact."""
    import torch

    m, m2 = 8, 5
    p = m + m2
    dmax = 1.0625
    tol = dmax * 1e-13 * m  # the kernel's threshold, evaluated in its order
    Ab = np.full((m, m), 0.0625)
    Ab[0, :] = Ab[:, 0] = 0.25
    Ab[0, 0] = 1.0
    np.fill_diagonal(Ab[1:, 1:], dmax)
    Ab[m - 1, m - 1] = 0.0625 + factor * tol
    assert ((Ab[m - 1, m - 1] - 0.0625) > tol) == (factor > 1)  # the pivot the kernel meets at the last step
    rng = np.random.default_rng(1200)
    Y = rng.standard_normal((20, m2))
    G = np.zeros((_round_up(p + 2, 8),) * 2)
    G[:m, :m] = Ab
    G[m:p, m:p] = Y.T @ Y
    G[p, :p] = G[:p, p] = rng.standard_normal(p)
    G[p, p] = 50.0
    G[p + 1, p + 1] = 20.0
    gptr = np.array([0, m, p])
    Wb, Rb, info, Gout, _ = _whiten(engine, G, p, gptr)
    assert info == (0 if factor > 1 else 1)
    if factor > 1:
        _check_factors(Wb, Rb, [Ab, G[m:p, m:p]], "pivot above the threshold")
        assert abs(Rb[0][m - 1, m - 1] - math.sqrt(factor * tol)) <= 1e-5 * math.sqrt(factor * tol)
        engine.whiten(torch.from_numpy(G[None]).to(engine.device), p, gptr, np.array([20.0]))
    else:
        _check_factors(Wb[1:], Rb[1:], [G[m:p, m:p]], "the well-conditioned group")
        with pytest.raises(ValueError, match="positive definite"):
            engine.whiten(torch.from_numpy(G[None]).to(engine.device), p, gptr, np.array([20.0]))


# ---- conjugate gradients ---------------------------------------------------------------------------------------------
def _cg(engine, G, p, shift=None, tol=1e-13, max_iter=None):
    """slm_gram_cg on one Gram: (rc, solution, the [p][8] output, iterations, relres)."""
    import torch

    pa = G.shape[0]
    max_iter = 10 * p + 100 if max_iter is None else max_iter
    Gd = _dev(engine, G)
    shd = None if shift is None else _dev(engine, shift, np.float64)
    nbytes = engine.lib.slm_gram_cg_workspace(p)
    work = torch.empty(nbytes, dtype=torch.uint8, device=engine.device)
    X8 = Buf(engine, 8 * p)
    iters, rel = ctypes.c_int32(-1), ctypes.c_double(-1.0)
    rc = engine.lib.slm_gram_cg(engine.h, engine._ptr(Gd), pa, p, engine._ptr(shd), float(tol), int(max_iter),
                                engine._ptr(work), nbytes, X8.ptr, ctypes.byref(iters), ctypes.byref(rel),
                                engine.stream)
    x8 = X8.fetch().reshape(p, 8)
    return rc, x8[:, 0].copy(), x8, int(iters.value), float(rel.value)


def _cg_gram(rng, n, p, shifted):
    """Gram of [X | y | 1 | 0] with rows and columns past the c row NaN (not read by the solve), and a shift."""
    X = rng.standard_normal((n, p))
    G = _augmented(X, rng.standard_normal(n))
    G[p + 1:, :] = G[:, p + 1:] = np.nan
    shift = 0.5 + n * 0.05 * rng.random(p) if shifted else None
    return G, shift


def _true_relres(G, p, shift, x):
    """||c - (G + S) x|| / ||c|| in float64 and the rounding allowance of the kernel's recomputation."""
    A_ = G[:p, :p] + (0.0 if shift is None else np.diag(shift))
    c = G[p, :p]
    r = c - A_ @ x
    nc = np.linalg.norm(c)
    allow = 2 * A.gamma(p + 4) * np.linalg.norm(np.abs(A_) @ np.abs(x) + np.abs(c)) / nc
    return np.linalg.norm(r) / nc, allow


@pytest.mark.parametrize("shifted", [False, True], ids=["plain", "shift"])
@pytest.mark.parametrize("p", [1, 31, 1023, 1024, 1025, 2100])
def test_gram_cg_matches_solve(engine, p, shifted):
    """(G + diag(shift)) x = c against numpy.linalg.solve, p across the 1024-thread stride of the vector kernels:
    forward error within kappa times the attained residual, reported relres equal to the recomputed one."""
    rng = np.random.default_rng(1300 + p + shifted)
    n = p + p // 2 + 20
    G, shift = _cg_gram(rng, n, p, shifted)
    rc, x, x8, iters, rel = _cg(engine, G, p, shift)
    _ok(engine, rc, "slm_gram_cg")
    assert (x8[:, 1:] == 0.0).all()
    A_ = G[:p, :p] + (0.0 if shift is None else np.diag(shift))
    ref = np.linalg.solve(A_, G[p, :p])
    ev = np.linalg.eigvalsh(A_)
    kappa = ev[-1] / ev[0]
    true_rel, allow = _true_relres(G, p, shift, x)
    assert abs(rel - true_rel) <= allow, (rel, true_rel, allow)
    assert rel <= 4e-13 + allow, (rel, iters)
    err = np.linalg.norm(x - ref) / np.linalg.norm(ref)
    assert err <= 2 * kappa * (rel + allow + p * U), (err, kappa, rel)


def test_gram_cg_minimum_norm_when_p_exceeds_n(engine):
    """p > n: G is singular and consistent; from x = 0 the iterates stay in range(G), so the solution is the
    minimum-norm one, with no component in the null space of X."""
    rng = np.random.default_rng(1400)
    n, p = 60, 150
    X = rng.standard_normal((n, p))
    y = rng.standard_normal(n)
    G = _augmented(X, y)
    rc, x, _, iters, rel = _cg(engine, G, p)
    _ok(engine, rc, "slm_gram_cg")
    _, _, Vt = np.linalg.svd(X)
    null = Vt[n:]
    assert np.linalg.norm(null @ x) <= 1e-10 * np.linalg.norm(x)
    ref = np.linalg.pinv(X) @ y
    assert np.linalg.norm(x - ref) <= 1e-9 * np.linalg.norm(ref)
    assert rel <= 4e-13


def test_gram_cg_zero_right_hand_side(engine):
    """c = 0: x = 0 after 0 iterations, relres 0."""
    rng = np.random.default_rng(1500)
    n, p = 80, 40
    G = _augmented(rng.standard_normal((n, p)), np.zeros(n))
    rc, x, x8, iters, rel = _cg(engine, G, p)
    _ok(engine, rc, "slm_gram_cg")
    assert iters == 0 and rel == 0.0
    assert (x8 == 0.0).all()


@pytest.mark.parametrize("shifted", [False, True], ids=["plain", "shift"])
def test_gram_cg_reports_true_residual_when_not_converged(engine, shifted):
    """kappa ~ 1e10 and max_iter = 15: all iterations run, the reported relres is the recomputed
    ||c - (G + S) x|| / ||c|| to rounding, and it is above the tolerance (the call does not claim convergence)."""
    rng = np.random.default_rng(1600 + shifted)
    p = 300
    Q, _ = np.linalg.qr(rng.standard_normal((p, p)))
    A_ = (Q * np.geomspace(1.0, 1e-10, p)) @ Q.T
    A_ = 0.5 * (A_ + A_.T)
    pa = _round_up(p + 2, 8)
    G = np.full((pa, pa), np.nan)
    G[:p, :p] = A_
    G[p, :p] = G[:p, p] = rng.standard_normal(p)
    shift = 1e-9 * rng.random(p) if shifted else None
    tol, max_iter = 1e-13, 15
    rc, x, _, iters, rel = _cg(engine, G, p, shift, tol=tol, max_iter=max_iter)
    _ok(engine, rc, "slm_gram_cg")
    assert iters == max_iter
    true_rel, allow = _true_relres(G, p, shift, x)
    assert abs(rel - true_rel) <= allow, (rel, true_rel, allow)
    assert rel > 4 * tol


def test_gram_cg_nan_in_c_row_is_an_error(engine):
    """A NaN in c = X^T y makes the residual non-finite: the call returns the library's error code 7."""
    rng = np.random.default_rng(1700)
    n, p = 50, 20
    G = _augmented(rng.standard_normal((n, p)), rng.standard_normal(n))
    G[p, 3] = np.nan
    rc, *_ = _cg(engine, G, p)
    assert rc == 7
    assert b"non-finite residual" in engine.lib.slm_last_error(engine.h)

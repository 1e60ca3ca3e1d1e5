"""slm_newton_step (csrc/newton_kernels.cuh) column by column against the float64 reference of one Newton step
(tests/newton_reference.py), at the sizes where the blocked factorisation changes shape: active-set sizes
around every multiple of the 16-wide sub-blocks and the 64-wide panels up to ~2000 coordinates, mixed in one
call so that columns sit out at different panels; more than 32 trailing-update problems per panel (one GEMM
flush); up to SLM_MAX_FOLDS Grams with unsorted, repeated fold indices; a group longer than a panel; both
feeds of the trailing-update GEMM; well-conditioned and overlap-expanded (kappa(H) ~ 1e4 - 1e6) Hessians.

The factor and the inverses of its diagonal blocks are read from the caller-owned workspace (white box), so
that a wrong factorisation shows even where the line search would hide it behind a shorter step."""

import ctypes
import os

import numpy as np
import pytest

import newton_reference as NR
import oracle.reference as R

pytestmark = pytest.mark.gpu

EPS = np.finfo(np.float64).eps
NB = 64           # panel width of the blocked Cholesky (NW_NB)
MAX_FOLDS = 16    # SLM_MAX_FOLDS
DEFAULT_TMA = 15  # the engine's default "tma" mask (slm_ctx::tma_mask): bit 0 feeds the trailing update by TMA
ENGINE_TMA = int(os.environ.get("SLM_TMA", DEFAULT_TMA))  # the mask the engine was created with
# bound constants: backward error of the factor / the inverses / the solve, in units of m * eps
C_FACTOR, C_INV, C_SOLVE = 4.0, 4.0, 4.0

SIZES = [0, 1, 2, 15, 16, 17, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 257, 500]
MULTI = [3, 150, 5, 70, 2, 40, 9, 20]  # multi-feature groups ahead of a run of singleton groups


def _round_up(v, m):
    return (v + m - 1) // m * m


def workspace_views(work, p, k, m_max):
    """The step's intermediates in the caller-owned workspace, as laid out by slm_newton_step
    (sparselm_b200/csrc/engine.cu; a layout change there has to be made here too):
      H    [k][ldh][ldh] at 0, ldh = max(8, round_up(m_max, 8)), over the compacted active coordinates; after the
           step its upper triangle is the factor U (H = U'U)
      INV  [k][npan][64][64] at k * ldv^2 (ldv = round_up(p, 8)), npan = max(1, ceil(m_max / 64)): the upper
           triangular inverse of every diagonal 64 x 64 block of U
      U, KK, DP, GS, GRAD, DIR  [k][ldv] each, after k * ceil(p / 64) * 64^2 doubles reserved for INV."""
    wd = work.view(-1)
    ldv = _round_up(p, 8)
    ldh = max(8, _round_up(m_max, 8))
    npan = max(1, -(-m_max // NB))
    H = wd[: k * ldh * ldh].view(k, ldh, ldh)
    o = k * ldv * ldv
    INV = wd[o:o + k * npan * NB * NB].view(k, npan, NB, NB)
    o += k * (-(-p // NB)) * NB * NB
    vec = {}
    for name in ("U", "KK", "DP", "GS", "GRAD", "DIR"):
        vec[name] = wd[o:o + k * ldv].view(k, ldv)
        o += k * ldv
    return dict(H=H, INV=INV, **vec)


def run_step(engine, case, X0w, work=None, fill=0.0):
    """One slm_newton_step on a copy of X0w [k][ldv] (device); returns (X after the step, out [k][4], workspace)."""
    import torch

    p, F, k = case["p"], case["F"], X0w.shape[0]
    Gn = len(case["gptr"]) - 1
    nbytes = engine.lib.slm_newton_workspace(p, Gn, k, F)
    if work is None:
        work = torch.full(((nbytes + 7) // 8,), fill, dtype=torch.float64, device=engine.device)
    X = X0w.clone()
    out = torch.full((k, 4), fill, dtype=torch.float64, device=engine.device)
    fh = np.ascontiguousarray(case["fold"], dtype=np.int32)
    Gs, pa = case["Gs_dev"], case["Gs_dev"].shape[-1]
    engine._ck(engine.lib.slm_newton_step(
        engine.h, engine._ptr(Gs), pa * pa, pa, p, F, k, fh.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
        engine._ptr(case["nobs_dev"]), engine._ptr(X), engine._ptr(case["w2_dev"]), engine._ptr(case["d2_dev"]),
        engine._ptr(case["gptr_dev"]), engine._ptr(case["gid_dev"]), Gn, engine._ptr(work), nbytes, engine._ptr(out),
        engine.stream), "slm_newton_step")
    torch.cuda.synchronize(engine.device)
    return X, out, work


# ---- problems -------------------------------------------------------------------------------------------------
def _grams(engine, rng, p, F, n):
    """F Grams [F][pa][pa] of random designs with n rows (rows/cols < p: X'X, row / col p: X'y), built on the device."""
    import torch

    pa = engine.padded_cols(p)
    Gs = torch.zeros((F, pa, pa), dtype=torch.float64, device=engine.device)
    gen = torch.Generator(device=engine.device).manual_seed(int(rng.integers(1 << 30)))
    for f in range(F):
        X = torch.randn((n, p), generator=gen, dtype=torch.float64, device=engine.device)
        w = torch.randn(p, generator=gen, dtype=torch.float64, device=engine.device) * (torch.rand(
            p, generator=gen, dtype=torch.float64, device=engine.device) < 0.2)
        y = X @ w + 0.3 * torch.randn(n, generator=gen, dtype=torch.float64, device=engine.device)
        Xa = torch.cat([X, y[:, None]], 1)
        Gs[f, :p + 1, :p + 1] = Xa.T @ Xa
    return Gs


def _support(rng, gptr, m, big_first):
    """Groups whose sizes add up to exactly m: some multi-feature groups, the rest singletons."""
    sizes = np.diff(gptr)
    multi = [g for g in range(len(sizes)) if sizes[g] > 1]
    single = [g for g in range(len(sizes)) if sizes[g] == 1]
    chosen, left = [], m
    order = list(rng.permutation(multi))
    if big_first:
        order.sort(key=lambda g: -sizes[g])
    for g in order:
        if sizes[g] <= left and (big_first or rng.random() < 0.6):
            chosen.append(g)
            left -= sizes[g]
    assert left <= len(single), (m, left, len(single))  # the layout needs enough singleton groups
    chosen += list(rng.choice(single, left, replace=False))
    return chosen


def _finish(engine, case):
    import torch

    dev = engine.device
    p, k = case["p"], len(case["fold"])
    gptr = case["gptr"]
    case["gid"] = NR.group_ids(gptr)
    case["Gs"] = case["Gs_dev"].cpu().numpy()
    case["gptr_dev"] = torch.from_numpy(gptr.astype(np.int32)).to(dev)
    case["gid_dev"] = torch.from_numpy(case["gid"].astype(np.int32)).to(dev)
    case["nobs_dev"] = torch.from_numpy(case["nobs"]).to(dev)
    case["w2_dev"] = torch.from_numpy(np.ascontiguousarray(case["w2"])).to(dev)
    case["d2_dev"] = None if case["d2"] is None else torch.from_numpy(np.ascontiguousarray(case["d2"])).to(dev)
    ldv = _round_up(p, 8)
    X0w = np.zeros((k, ldv))
    X0w[:, :p] = case["X0"]
    case["X0w"] = torch.from_numpy(X0w).to(dev)
    case["ref"] = [NR.newton_step(case["Gs"][case["fold"][c]], p, case["nobs"][c], case["X0"][c], case["w2"][c],
                                  None if case["d2"] is None else case["d2"][c], gptr) for c in range(k)]
    return case


def _sized_case(engine, seed, p, F, ms, ridge, backtrack):
    """Columns with exactly ms[c] active coordinates (in shuffled order), random folds, per-column n."""
    rng = np.random.default_rng(seed)
    sizes = MULTI + [1] * (p - sum(MULTI))
    gptr = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    Gn = len(sizes)
    n = 3 * p
    ms = list(rng.permutation(ms))
    k = len(ms)
    X0 = np.zeros((k, p))
    for c, m in enumerate(ms):
        for g in _support(rng, gptr, m, big_first=m >= 257):
            X0[c, gptr[g]:gptr[g + 1]] = rng.standard_normal(gptr[g + 1] - gptr[g])
    w2 = 0.05 * (0.5 + rng.random((k, Gn)))
    for c in np.flatnonzero(np.array(ms) > 0)[:backtrack]:  # far start, strong penalty: the step has to backtrack
        X0[c] *= 1e-3
        w2[c] *= 40.0
    if F == MAX_FOLDS:  # every fold used, unsorted, repeated
        fold = rng.permutation(np.concatenate([np.arange(F), rng.integers(0, F, k - F)]))
    else:
        fold = rng.integers(0, F, k)
    case = dict(p=p, F=F, gptr=gptr, fold=fold, nobs=n * (0.5 + rng.random(k)), X0=X0, w2=w2,
                d2=((rng.random((k, Gn)) < 0.3) * 0.2) if ridge else None, Gs_dev=_grams(engine, rng, p, F, n))
    return _finish(engine, case)


def _overlap_case(engine, seed):
    """C4's structure: an overlap-expanded Gram (duplicated columns) with weak group weights."""
    import torch

    rng = np.random.default_rng(seed)
    n, p, G = 900, 500, 50
    X = rng.standard_normal((n, p))
    base = rng.permutation(np.repeat(np.arange(G), p // G))
    extra = rng.random(p) < 0.3
    gl = [[int(base[j])] + ([int((base[j] + 1 + rng.integers(G - 1)) % G)] if extra[j] else []) for j in range(p)]
    idx, lab, Gn = R.expand_overlap(gl, p)
    pe = len(idx)
    gptr = np.concatenate([[0], np.cumsum(np.bincount(lab, minlength=Gn))]).astype(np.int64)
    y = X @ (rng.standard_normal(p) * (rng.random(p) < 0.2)) + rng.standard_normal(n)
    pa = engine.padded_cols(p)
    Gf = np.zeros((pa, pa))
    Xa = np.hstack([X, y[:, None], np.ones((n, 1))])
    Gf[:p + 2, :p + 2] = Xa.T @ Xa
    ext = torch.from_numpy(idx.astype(np.int32)).to(engine.device)
    Gs = engine.gram_gather(torch.from_numpy(Gf).to(engine.device)[None], p, ext, pe)  # y's row / column follow
    k = 36
    X0 = np.zeros((k, pe))
    for c in range(k):
        for g in rng.choice(Gn, int(Gn * (0.2 + 0.8 * rng.random())), replace=False):
            X0[c, gptr[g]:gptr[g + 1]] = rng.standard_normal(gptr[g + 1] - gptr[g])
    w2 = 10.0 ** rng.uniform(-4, -3, (k, 1)) * (0.5 + rng.random((k, Gn)))
    case = dict(p=pe, F=1, gptr=gptr, fold=np.zeros(k, dtype=np.int64), nobs=np.full(k, float(n)), X0=X0, w2=w2,
                d2=None, Gs_dev=Gs.contiguous())
    return _finish(engine, case)


_CASES = {}


def _case(engine, name):
    if name not in _CASES:
        if name == "sizes":  # every size of SIZES, one column of C4's size, 28 more with rows at the first panel
            rng = np.random.default_rng(1)
            ms = SIZES + [1959] + list(rng.integers(65, 400, 28))
            _CASES[name] = _sized_case(engine, 2, 2100, 3, ms, ridge=True, backtrack=2)
        elif name == "folds":  # m_max = 577 (odd, = 1 mod 8), SLM_MAX_FOLDS Grams, no ridge (D2 = NULL)
            rng = np.random.default_rng(3)
            ms = SIZES + [577] + list(rng.integers(65, 300, 24))
            _CASES[name] = _sized_case(engine, 4, 640, MAX_FOLDS, ms, ridge=False, backtrack=1)
        elif name == "overlap":
            _CASES[name] = _overlap_case(engine, 5)
    return _CASES[name]


@pytest.fixture()
def tma_mask(engine, request):
    engine.set_option("tma", request.param)
    yield request.param
    engine.set_option("tma", ENGINE_TMA)


# ---- checks ---------------------------------------------------------------------------------------------------
def _bits(a):
    return np.ascontiguousarray(a).view(np.int64)


def check_column(case, c, Xk, outk, views, well_conditioned):
    """Everything one column of one step must satisfy; returns whether its line-search decision was compared."""
    ref = case["ref"][c]
    p = case["p"]
    G, n = case["Gs"][case["fold"][c]], case["nobs"][c]
    x0 = case["X0"][c]
    act, m = ref["act"], len(ref["act"])
    Href = ref["H"]
    on = ref["on"]
    acc, t, dec, flag = outk
    assert np.isfinite(Xk).all() and np.isfinite(outk).all(), c
    assert acc in (0.0, 1.0) and flag in (0.0, 1.0)
    if m:
        # factor: backward error, independent of kappa (|U|'|U| <= max diag H); plus the assembly's rounding
        U = np.triu(views["H"][c, :m, :m])
        asm = 4 * EPS * (np.abs(np.diag(G)[act]) / n + ref["kk"][act]).max()
        err = np.abs(U.T @ U - Href).max()
        assert err <= C_FACTOR * m * EPS * np.abs(Href).max() + asm, (c, m, err, np.abs(Href).max())
        # inverses of the diagonal blocks: U_pp INV_pp = I on the leading nb x nb block of every panel
        for pn in range(-(-m // NB)):
            j0 = pn * NB
            nb = min(NB, m - j0)
            Upp, Vpp = U[j0:j0 + nb, j0:j0 + nb], views["INV"][c, pn, :nb, :nb]
            assert np.all(np.tril(Vpp, -1) == 0.0), (c, pn)
            res = np.abs(Upp @ Vpp - np.eye(nb))
            assert np.all(res <= C_INV * nb * EPS * (np.abs(Upp) @ np.abs(Vpp)) + 1e-300), (c, pn, res.max())
    # direction (read back from the workspace): zero off the support, small backward residual on it
    d = views["DIR"][c, :p]
    assert np.all(d[~on] == 0.0), c
    gref = ref["grad_a"]
    # the gradient comes through the Gram apply (another summation order than the reference's)
    geps = p * EPS * (np.abs(G[:p, :p][act]) @ np.abs(x0) + np.abs(G[p, :p][act])) / n
    if m:
        da = d[act]
        r = np.abs(Href @ da + gref).max()
        hn = np.abs(Href).sum(1).max()
        bound = C_SOLVE * m * EPS * (hn * np.abs(da).max() + np.abs(gref).max()) + geps.max()
        assert r <= bound, (c, m, r, bound)
        # decrement: -g'd; a backward error dH of the solve moves it by d'dH d, a gradient error by 2 geps'|d|
        dr = ref["d"][act]
        dbound = C_SOLVE * m * EPS * (np.linalg.norm(Href) * (dr @ dr) + np.abs(gref) @ np.abs(dr)) \
            + 2 * geps @ np.abs(dr) + 1e-300
        assert abs(dec - ref["dec"]) <= dbound, (c, m, dec, ref["dec"], dbound)
    else:
        assert dec == 0.0
    # line search: the reference's decision, unless one of its tests was within rounding of the threshold
    rel_d = np.abs(d - ref["d"]).max() / max(np.abs(ref["d"]).max(), 1e-300) + C_SOLVE * max(m, 1) * EPS
    close = any(abs(dphi - thr) <= 8 * rel_d * size for (_, dphi, thr, size) in ref["trials"])
    if not close:
        assert bool(acc) == ref["accepted"] and t == ref["t"], (c, m, acc, t, ref["accepted"], ref["t"])
    x0w = case["X0w_host"][c]
    if acc:
        assert t > 0 and t <= 1 and np.log2(t) == np.round(np.log2(t))
        np.testing.assert_array_equal(Xk[:p], x0 + t * d)  # the update itself: t is a power of two
        # every accepted step lowers phi (float64, from the Gram), by the Armijo fraction of the kernel's decrement
        dphi = NR.objective_change(G, p, n, x0, Xk[:p], case["w2"][c], None if case["d2"] is None else case["d2"][c],
                                   case["gptr"])
        assert dphi <= 0.5 * NR.ARMIJO * t * -dec, (c, dphi, t, dec)
        if well_conditioned and not close:
            assert np.abs(Xk[:p] - ref["x_new"]).max() <= 1e-10 * np.abs(x0).max(), c
    else:  # a column that is not accepted is left alone
        assert t == 0.0
        assert np.array_equal(_bits(Xk), _bits(x0w)), c
    # inactive coordinates and the padding columns [p, ldv) of X: bitwise unchanged
    assert np.array_equal(_bits(Xk[:p][~on]), _bits(x0w[:p][~on])), c
    assert np.array_equal(_bits(Xk[p:]), _bits(x0w[p:])), c
    if well_conditioned:
        assert ref["ok"] and flag == 0.0, c
    return not close


def _check_call(engine, case, well_conditioned):
    """Reference checks on a zero-filled workspace, then bitwise equality with a repeated call and with a call on a
    NaN-poisoned workspace and NaN padding columns of X."""
    p, k = case["p"], len(case["fold"])
    case["X0w_host"] = case["X0w"].cpu().numpy()
    X, out, work = run_step(engine, case, case["X0w"])
    Xh, outh = X.cpu().numpy(), out.cpu().numpy()
    m_max = max(len(r["act"]) for r in case["ref"])
    views = {kk: v.cpu().numpy() for kk, v in workspace_views(work, p, k, m_max).items()}
    compared = sum(check_column(case, c, Xh[c], outh[c], views, well_conditioned) for c in range(k))
    assert compared >= k - 2, (compared, k)
    # same call again: bitwise the same
    X2, out2, _ = run_step(engine, case, case["X0w"])
    assert np.array_equal(_bits(X2.cpu().numpy()), _bits(Xh)) and np.array_equal(_bits(out2.cpu().numpy()), _bits(outh))
    # poisoned workspace and padding (production hands torch.empty memory in)
    ldv = case["X0w"].shape[1]
    X0n = case["X0w"].clone()
    if ldv > p:
        X0n[:, p:] = float("nan")
    X3, out3, _ = run_step(engine, case, X0n, fill=float("nan"))
    X3h = X3.cpu().numpy()
    assert np.isfinite(X3h[:, :p]).all() and np.isfinite(out3.cpu().numpy()).all()
    assert np.array_equal(_bits(X3h[:, :p]), _bits(Xh[:, :p])) and np.array_equal(_bits(out3.cpu().numpy()), _bits(outh))
    assert np.isnan(X3h[:, p:]).all()
    return Xh, outh


# ---- tests ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tma_mask", [DEFAULT_TMA, 0], indirect=True, ids=["tma", "cpasync"])
@pytest.mark.parametrize("name", ["sizes", "folds"])
def test_newton_step_matches_reference_across_panels(engine, tma_mask, name):
    case = _case(engine, name)
    ms = [len(r["act"]) for r in case["ref"]]
    assert set(SIZES) <= set(ms) and sum(m > NB for m in ms) >= 33        # > 32 GEMM problems at the first panel
    assert max(ms) % 8 in (1, 7)                                          # odd m_max: the round_up(rows, 2) tail
    Xh, outh = _check_call(engine, case, well_conditioned=True)
    ts = outh[:, 1][outh[:, 0] == 1]
    assert ts.min() < 1.0 and ts.max() == 1.0                             # backtracked and full steps


@pytest.mark.parametrize("tma_mask", [DEFAULT_TMA, 0], indirect=True, ids=["tma", "cpasync"])
def test_newton_step_matches_reference_on_an_overlap_expanded_gram(engine, tma_mask):
    case = _case(engine, "overlap")
    kappa = [np.linalg.cond(r["H"]) for r in case["ref"]]
    assert 1e4 <= max(kappa) <= 1e6 and max(len(r["act"]) for r in case["ref"]) > 4 * NB
    _check_call(engine, case, well_conditioned=False)


def test_newton_step_with_no_active_coordinate_leaves_everything_alone(engine):
    """The all-empty call (m_max = 0): nothing factored, every column unchanged, out = {0, 0, 0, 0}."""
    rng = np.random.default_rng(6)
    p, k = 70, 5
    gptr = np.concatenate([[0], np.cumsum([7] * 10)]).astype(np.int64)
    case = dict(p=p, F=2, gptr=gptr, fold=np.array([1, 0, 1, 1, 0]), nobs=np.full(k, 200.0), X0=np.zeros((k, p)),
                w2=0.1 * np.ones((k, 10)), d2=None, Gs_dev=_grams(engine, rng, p, 2, 200))
    _finish(engine, case)
    X, out, _ = run_step(engine, case, case["X0w"], fill=float("nan"))
    assert np.array_equal(_bits(X.cpu().numpy()), _bits(case["X0w"].cpu().numpy()))
    assert np.array_equal(out.cpu().numpy(), np.zeros((k, 4)))


def test_newton_step_on_a_singular_hessian_keeps_its_contract(engine):
    """Duplicated features as singleton groups, no ridge: H = G_AA/n is singular wherever both copies are active.
    Whether the factorisation flags it is up to rounding; either way no NaN reaches X, a column that is not
    accepted is unchanged and an accepted one lowers phi."""
    import torch

    rng = np.random.default_rng(7)
    n, q, dup = 600, 220, 80
    X = rng.standard_normal((n, q))
    X = np.hstack([X, X[:, :dup]])                       # features q.. q+dup-1 repeat the first dup
    p = X.shape[1]
    y = X @ (rng.standard_normal(p) * (rng.random(p) < 0.3)) + rng.standard_normal(n)
    pa = engine.padded_cols(p)
    Gf = np.zeros((1, pa, pa))
    Xa = np.hstack([X, y[:, None]])
    Gf[0, :p + 1, :p + 1] = Xa.T @ Xa
    gptr = np.arange(p + 1, dtype=np.int64)
    k = 6
    X0 = np.zeros((k, p))
    for c in range(k):
        on = rng.choice(p, 150 + 30 * c, replace=False)
        on = np.union1d(on, [0, q])                       # both copies of feature 0 in every column
        X0[c, on] = rng.standard_normal(len(on))
    case = dict(p=p, F=1, gptr=gptr, fold=np.zeros(k, dtype=np.int64), nobs=np.full(k, float(n)), X0=X0,
                w2=0.01 * np.ones((k, p)), d2=None, Gs_dev=torch.from_numpy(Gf).to(engine.device))
    _finish(engine, case)
    x0w = case["X0w"].cpu().numpy()
    Xk, out, _ = run_step(engine, case, case["X0w"], fill=float("nan"))
    Xk, out = Xk.cpu().numpy(), out.cpu().numpy()
    assert np.isfinite(Xk[:, :p]).all()
    for c in range(k):
        acc, t, dec, flag = out[c]
        assert acc in (0.0, 1.0) and flag in (0.0, 1.0) and (flag == 1.0 or np.isfinite(dec)), (c, out[c])
        if acc:
            assert flag == 0.0 and dec > 0, (c, out[c])
            dphi = NR.objective_change(case["Gs"][0], p, n, X0[c], Xk[c, :p], case["w2"][c], None, gptr)
            assert dphi <= 0.5 * NR.ARMIJO * t * -dec, (c, dphi, t, dec, flag)
            assert np.all(Xk[c, :p][X0[c] == 0] == 0.0)
        else:
            assert t == 0.0 and np.array_equal(_bits(Xk[c]), _bits(x0w[c])), c


def test_newton_step_on_every_visible_device():
    """The kernels' shared-memory limits are raised per device: a Newton step runs on every visible device of
    one process, matches the reference there and gives the same result on each (one device: the reference only)."""
    import torch

    from sparselm_b200.engine import get_engine

    results = []
    for dev in range(torch.cuda.device_count()):
        eng = get_engine(dev)
        with torch.cuda.device(dev):
            case = _sized_case(eng, 8, 600, 2, [0, 17, 65, 130, 200, 257], ridge=True, backtrack=0)
            case["X0w_host"] = case["X0w"].cpu().numpy()
            X, out, work = run_step(eng, case, case["X0w"])
            results.append((X.cpu().numpy(), out.cpu().numpy()))
            k, m_max = len(case["fold"]), max(len(r["act"]) for r in case["ref"])
            views = {kk: v.cpu().numpy() for kk, v in workspace_views(work, case["p"], k, m_max).items()}
            for c in range(k):
                check_column(case, c, results[-1][0][c], results[-1][1][c], views, True)
    for X, out in results[1:]:
        assert np.array_equal(_bits(X), _bits(results[0][0])) and np.array_equal(_bits(out), _bits(results[0][1]))

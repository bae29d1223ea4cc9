"""``invpref_fold_in_users`` / ``invpref_fold_in_items`` (csrc/foldin.cu) against the fp64 references of
tests/_foldin_ref.py, and ``invpref_recommend_rows`` / ``invpref_top_users_rows`` against ``recommend`` / ``top_users``.

Accuracy bounds (per row, elementwise, n = history length, kappa = 2-norm condition number of the system matrix at
the solution, computed per case):
  explicit: |ours - ref| <= 1/2 ulp32 + C * (D + n) * kappa * 2^-53 * max|ref|
  implicit: |ours - ref| <= 2 ulp32   + C * (D + n) * kappa * 2^-53 * max|ref|,   C = 16.
The rounding term grows with D + n, not with D alone: every Gram entry is a sum of n products in CSR order (the
reference sums in numpy's order), so its rounding error grows with the history length as well as with the
factorisation's D.  For long histories (n = 100 000 in test_explicit_long_history) this is looser than a D-only
bound.  The ulp term is taken of max(|ref|, |ours|), because the two may straddle a power of two.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import _foldin_ref as ref
from test_gpu_eval_topk import csr_of, dense_lists, one_hot, random_lists
from test_gpu_recommend import EXCL_CASES, ref_recommend, _hot

gpu = pytest.mark.gpu
CONST = 16
LAMS = [1e-3, 1.0, 1e3]


def _dev():
    return torch.device("cuda:0")


def _tables(n_users, n_items, D, seed, scale=0.3):
    rng = np.random.default_rng(seed)
    U = rng.normal(0, scale, (n_users, D)).astype(np.float32)
    I = rng.normal(0, scale, (n_items, D)).astype(np.float32)
    return U, I


def _hp(U, I, implicit):
    d = _dev()
    return _hot(torch.from_numpy(U).to(d), torch.from_numpy(I).to(d), implicit)


def _fold(hp, side, off, ids, y, lam, max_iter=25):
    d = _dev()
    fn = hp.fold_in_users if side == "users" else hp.fold_in_items
    rows, it = fn(torch.from_numpy(off).to(d), torch.from_numpy(ids).to(d), torch.from_numpy(y).to(d), lam,
                  max_iter, return_iters=True)
    return rows.cpu().numpy(), it.cpu().numpy()


def _ulp32(x):
    return np.spacing(np.abs(x).astype(np.float32)).astype(np.float64)


def _check_rows(ours, want, V, hists, lam, implicit, ulps):
    for r, (ids, y) in enumerate(hists):
        w = want[r]
        if not len(ids):
            assert not ours[r].any() and not np.signbit(ours[r]).any(), r
            continue
        Vh = V[ids].astype(np.float64)
        kappa = ref.condition(Vh, y, lam, w, implicit)
        big = np.maximum(np.abs(w), np.abs(ours[r]))
        bound = ulps * _ulp32(big) + CONST * (V.shape[1] + len(ids)) * kappa * 2.0 ** -53 * np.abs(w).max()
        err = np.abs(ours[r] - w)
        assert (err <= bound).all(), (r, len(ids), float(err.max()), float(bound[np.argmax(err - bound)]), kappa)


def _lengths(D):
    return sorted({0, 1, max(D - 1, 0), D, D + 1, 15, 16, 17, 31, 32, 33, 1000})


def _histories(rng, n_cat, lengths, implicit):
    hists = []
    for L in lengths:
        ids = rng.integers(0, min(n_cat, max(L // 2, 1) + 3), L)      # duplicates in every long history
        y = (rng.random(L) < 0.5).astype(np.float32) if implicit else rng.integers(1, 6, L).astype(np.float32)
        hists.append((ids.astype(np.int64), y))
    return hists


def _csr(hists):
    off = np.zeros(len(hists) + 1, np.int64)
    off[1:] = np.cumsum([len(h[0]) for h in hists])
    ids = np.concatenate([h[0] for h in hists]) if hists else np.zeros(0, np.int64)
    y = np.concatenate([h[1] for h in hists]) if hists else np.zeros(0, np.float32)
    return off, ids.astype(np.int64), y.astype(np.float32)


# ==== 1. explicit fold-in against the fp64 solve ====================================================================
@gpu
@pytest.mark.parametrize("D", [1, 3, 17, 40, 64, 65, 127, 128])
@pytest.mark.parametrize("side", ["users", "items"])
def test_explicit_against_fp64_solve(D, side):
    U, I = _tables(700, 600, D, D)
    hp = _hp(U, I, False)
    V = I if side == "users" else U
    rng = np.random.default_rng(D + 7)
    hists = _histories(rng, V.shape[0], _lengths(D), False)
    off, ids, y = _csr(hists)
    for lam in LAMS:
        rows, it = _fold(hp, side, off, ids, y, lam)
        want = np.stack([ref.explicit(V[h[0]], h[1], lam) for h in hists])
        _check_rows(rows, want, V, hists, lam, False, 0.5)
        assert (it == np.array([1 if len(h[0]) else 0 for h in hists])).all()


@gpu
def test_explicit_long_history():
    D = 40
    U, I = _tables(100, 5000, D, 1)
    hp = _hp(U, I, False)
    rng = np.random.default_rng(2)
    hists = [(rng.integers(0, 5000, 100_000).astype(np.int64), rng.integers(1, 6, 100_000).astype(np.float32)),
             (np.arange(3, dtype=np.int64), np.ones(3, np.float32))]
    off, ids, y = _csr(hists)
    rows, _ = _fold(hp, "users", off, ids, y, 1.0)
    want = np.stack([ref.explicit(I[h[0]], h[1], 1.0) for h in hists])
    _check_rows(rows, want, I, hists, 1.0, False, 0.5)


# ==== 2. implicit fold-in against the Newton reference ==============================================================
def _implicit_hists(rng, V, kind, lengths):
    hists = []
    for L in lengths:
        ids = rng.integers(0, V.shape[0], L).astype(np.int64)
        if kind == "separable":
            w = rng.normal(size=V.shape[1])
            y = (V[ids].astype(np.float64) @ w > 0).astype(np.float32)
        elif kind == "positive":
            y = np.ones(L, np.float32)
        elif kind == "fractional":
            y = rng.random(L).astype(np.float32)
        else:
            y = (rng.random(L) < 0.5).astype(np.float32)
        hists.append((ids, y))
    return hists


@gpu
@pytest.mark.parametrize("D", [1, 3, 17, 40, 64, 128])
@pytest.mark.parametrize("kind", ["random", "separable", "positive", "fractional", "norm30"])
def test_implicit_against_newton_reference(D, kind):
    U, I = _tables(300, 400, D, D + 100)
    if kind == "norm30":
        I = (I * (30.0 / np.linalg.norm(I, axis=1, keepdims=True))).astype(np.float32)
    hp = _hp(U, I, True)
    rng = np.random.default_rng(D * 10 + len(kind))
    hists = _implicit_hists(rng, I, kind, [0, 1, D, D + 1, 33, 300])
    off, ids, y = _csr(hists)
    for lam in ([1e-2, 1.0, 1e2] if D <= 64 else [1.0]):
        rows, it = _fold(hp, "users", off, ids, y, lam, max_iter=100)
        for r, h in enumerate(hists):
            w, wit = ref.newton(I[h[0]], h[1], lam, max_iter=100)
            assert (it[r] == 0) == (wit == 0) and (wit == 0 or 1 <= it[r] <= 100), (r, it[r], wit)
            if wit == 0:
                assert not rows[r].any()
                continue
            Vh = I[h[0]].astype(np.float64)
            kappa = ref.condition(Vh, h[1], lam, w, True)
            big = np.maximum(np.abs(w), np.abs(rows[r]))
            bound = 2 * _ulp32(big) + CONST * (D + len(h[0])) * kappa * 2.0 ** -53 * np.abs(w).max()
            assert (np.abs(rows[r] - w) <= bound).all(), (r, lam, float(np.abs(rows[r] - w).max()))
            # stationarity of the fp32 result: |g(u32)| <= |H| |u32 - u*|
            H = ref.hessian(w, Vh, h[1], lam)
            g = ref.gradient(rows[r].astype(np.float64), Vh, h[1].astype(np.float64), lam)
            assert np.abs(g).max() <= np.linalg.norm(H, 2) * np.sqrt(D) * (2 * _ulp32(big).max() + bound.max())


@gpu
@pytest.mark.parametrize("seed", [1134, 2570])
def test_implicit_backtracking_and_first_step(seed):
    V, y, lam = ref.damped_problem(seed)
    steps = []
    want, wit = ref.newton(V, y, lam, max_iter=100, steps=steps)
    assert min(steps) < 1.0
    U = np.zeros((3, V.shape[1]), np.float32)
    hp = _hp(U, V, True)
    hist = [(np.arange(len(y), dtype=np.int64), y)]
    off, ids, yy = _csr(hist)
    rows, it = _fold(hp, "users", off, ids, yy, lam, max_iter=100)
    assert it[0] == wit
    assert np.abs(rows[0] - want).max() <= 2 * _ulp32(np.abs(want).max()) + 1e-12 * np.abs(want).max()
    # max_iter = 1: the first damped step; not converged -> -1
    rows1, it1 = _fold(hp, "users", off, ids, yy, lam, max_iter=1)
    w1, wit1 = ref.newton(V, y, lam, max_iter=1)
    assert it1[0] == wit1 == -1
    assert np.abs(rows1[0] - w1).max() <= 2 * _ulp32(np.abs(w1).max())
    # a row that cannot converge in max_iter reports -max_iter
    k = max(2, abs(wit) - 1)
    _, itk = _fold(hp, "users", off, ids, yy, lam, max_iter=k)
    assert itk[0] == (-k if k < wit else wit)


# ==== 3. invariance =================================================================================================
@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
def test_results_do_not_depend_on_the_batch(implicit):
    D = 40
    U, I = _tables(200, 3000, D, 11)
    hp = _hp(U, I, implicit)
    rng = np.random.default_rng(12)
    hists = _histories(rng, 3000, list(rng.integers(0, 120, 1000)) + [0, 5000], implicit)
    off, ids, y = _csr(hists)
    rows, it = _fold(hp, "users", off, ids, y, 0.5)
    again, it2 = _fold(hp, "users", off, ids, y, 0.5)
    assert np.array_equal(rows.view(np.uint32), again.view(np.uint32)) and np.array_equal(it, it2)
    perm = rng.permutation(len(hists))
    p_rows, p_it = _fold(hp, "users", *_csr([hists[i] for i in perm]), 0.5)
    assert np.array_equal(p_rows.view(np.uint32), rows[perm].view(np.uint32)) and np.array_equal(p_it, it[perm])
    for sel in ([0], [len(hists) - 1], list(range(0, len(hists), 3))):
        s_rows, s_it = _fold(hp, "users", *_csr([hists[i] for i in sel]), 0.5)
        assert np.array_equal(s_rows.view(np.uint32), rows[sel].view(np.uint32)) and np.array_equal(s_it, it[sel])


# ==== 4. edge cases =================================================================================================
@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
def test_empty_nan_inf_rows(implicit):
    D = 16
    U, I = _tables(50, 80, D, 3)
    I[7, 3] = np.nan
    I[9, 0] = np.inf
    hp = _hp(U, I, implicit)
    y = lambda n: np.ones(n, np.float32) if implicit else np.full(n, 3.0, np.float32)
    ok = (np.array([1, 2, 3, 4, 5], np.int64), y(5))
    nan_score = (np.array([1, 2, 3], np.int64), np.array([1, np.nan, 0], np.float32))
    hists = [ok, (np.zeros(0, np.int64), y(0)), nan_score, (np.array([1, 7, 2], np.int64), y(3)), ok,
             (np.array([9, 1], np.int64), y(2)), ok]
    rows, it = _fold(hp, "users", *_csr(hists), 1.0)
    for r in (2, 3, 5):
        assert np.isnan(rows[r]).all(), r
    for r in (0, 4, 6):
        assert np.isfinite(rows[r]).all() and np.array_equal(rows[r], rows[0])
    assert not rows[1].any() and it[1] == 0
    alone, _ = _fold(hp, "users", *_csr([ok]), 1.0)
    assert np.array_equal(alone[0].view(np.uint32), rows[0].view(np.uint32))


@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
def test_out_of_range_ids(implicit):
    from invpref_kdd_2022_b200 import _lib
    D = 24
    U, I = _tables(50, 80, D, 4)
    hp = _hp(U, I, implicit)
    d = _dev()
    ids = np.array([3, -1, 5, 80, 5, 2 ** 40, 79], np.int64)
    y = np.array([1, 0, 1, 1, 0, 1, 1], np.float32)
    keep = np.array([0, 2, 4, 6])
    with pytest.raises(IndexError):
        _fold(hp, "users", np.array([0, 7], np.int64), ids, y, 1.0)
    out = torch.empty((1, D), dtype=torch.float32, device=d)
    t = lambda a: torch.from_numpy(a).to(d)
    off_t, ids_t, y_t = t(np.array([0, 7], np.int64)), t(ids), t(y)
    p = _lib.make_params(hp.params)
    _lib.check(hp.lib.invpref_fold_in_users(C.byref(hp.desc), C.byref(p), _lib.ptr(off_t), _lib.ptr(ids_t),
                                            _lib.ptr(y_t), 1, 1.0, 25, _lib.ptr(out), None, _lib.stream_ptr()))
    want, _ = _fold(hp, "users", np.array([0, 4], np.int64), ids[keep], y[keep], 1.0)
    assert np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32))


# ==== 5. top-k on external rows =====================================================================================
@gpu
@pytest.mark.parametrize("case", EXCL_CASES)
def test_recommend_rows_equals_recommend(case):
    rng = np.random.default_rng(EXCL_CASES.index(case) + 50)
    n_users, n, k = 5, 20011, 64
    tab = one_hot(rng, n_users, n, 8, False, a_range=30)
    excl = random_lists(rng, n_users, n, 40, out_of_range=False)
    if case == "empty_lists":
        excl = csr_of([np.zeros(0, np.int64)] * n_users)
    elif case == "every_item":
        excl = csr_of([np.arange(n)] * n_users)
    elif case == "fewer_than_k":
        excl = csr_of([np.setdiff1d(np.arange(n), rng.choice(n, j, replace=False)) for j in (0, 1, 3, 63, 10)])
    elif case == "out_of_range":
        excl = csr_of([np.concatenate([[-(2 ** 40), -5, -1], excl[1][excl[0][u]:excl[0][u + 1]], [n, n + 1]])
                       for u in range(n_users)])
    elif case == "long_lists_across_edges":
        excl = csr_of([np.unique(np.concatenate([np.arange(e - 300, e + 300) for e in (1152, 5000, 15000)[u % 3:]]))
                       for u in range(n_users)])
    elif case == "no_lists":
        excl = None
    d = _dev()
    Ut, It = tab.device(d)
    for implicit in (False, True):
        hp = _hot(Ut, It, implicit)
        users = np.arange(n_users)
        ex = None if excl is None else tuple(torch.from_numpy(np.ascontiguousarray(x)).to(d) for x in excl)
        for kk in (1, k, 256):
            top, sc = hp.recommend(torch.from_numpy(users).to(d), kk, ex)
            top2, sc2 = hp.recommend_rows(Ut[torch.from_numpy(users).to(d)].contiguous(), kk, ex)
            assert torch.equal(top, top2) and torch.equal(sc.view(torch.int32), sc2.view(torch.int32))
            if not implicit:
                want, ws = ref_recommend(tab.z(users).astype(np.float32), dense_lists(excl, users, n), kk)
                assert np.array_equal(top2.cpu().numpy(), want)
        # top_users_rows on item rows (exclusion lists over the b rows) against top_users on their item ids
        items = rng.choice(n, 7, replace=False)
        ex_u = random_lists(rng, 7, n_users, 2, out_of_range=False)
        per = {int(items[r]): ex_u[1][ex_u[0][r]:ex_u[0][r + 1]] for r in range(7)}
        ex_full = csr_of([per.get(i, np.zeros(0, np.int64)) for i in range(n)])
        to_dev = lambda c: tuple(torch.from_numpy(np.ascontiguousarray(x)).to(d) for x in c)
        it_t = torch.from_numpy(items).to(d)
        for kk in (1, 3, n_users):
            top, sc = hp.top_users_rows(It[it_t].contiguous(), kk, to_dev(ex_u))
            top2, sc2 = hp.top_users(it_t, kk, to_dev(ex_full))
            assert torch.equal(top, top2) and torch.equal(sc.view(torch.int32), sc2.view(torch.int32))


@gpu
def test_round_trip_recovers_the_user_rows():
    D, n_items = 32, 20000
    U, I = _tables(64, n_items, D, 21, scale=0.5)
    hp = _hp(U, I, False)
    rng = np.random.default_rng(22)
    users = np.arange(64)
    hists = []
    for u in users:
        ids = rng.choice(n_items, 4 * D, replace=False).astype(np.int64)
        hists.append((ids, (I[ids].astype(np.float64) @ U[u].astype(np.float64)).astype(np.float32)))
    lam = 1e-6
    rows, _ = _fold(hp, "users", *_csr(hists), lam)
    err = np.abs(rows - U).max(axis=1)
    for r, h in enumerate(hists):
        Vh = I[h[0]].astype(np.float64)
        kappa = ref.condition(Vh, h[1], lam)
        # the planted scores are rounded to fp32: the recovered row moves by up to kappa * that rounding
        tol = 2 * _ulp32(np.abs(U[r]).max()) + kappa * (2.0 ** -24 * np.abs(h[1]).max() * np.sqrt(len(h[1]))
                                                         / np.linalg.norm(Vh, 2) + lam * np.abs(U[r]).max())
        assert err[r] <= tol, (r, err[r], tol)
    d = _dev()
    top, _ = hp.recommend(torch.from_numpy(users).to(d), 50)
    top_f, _ = hp.recommend_rows(torch.from_numpy(rows).to(d), 50)
    top, top_f = top.cpu().numpy(), top_f.cpu().numpy()
    z = U.astype(np.float64) @ I.T.astype(np.float64)
    for r in users:
        s = np.sort(z[r])[::-1][:51]
        margin = err[r] * np.abs(I).sum(axis=1).max() * 2 + 1e-5
        cut = int(np.argmax(np.diff(-s) <= margin)) if (np.diff(-s) <= margin).any() else 50
        assert set(top[r, :cut].tolist()) == set(top_f[r, :cut].tolist()), r


# ==== 6. model API ==================================================================================================
def _model(cls, D=16, n_users=60, n_items=90):
    torch.manual_seed(0)
    return cls(n_users, n_items, 2, D).to(_dev())


@gpu
@pytest.mark.parametrize("which", ["explicit", "implicit"])
def test_model_api(which):
    from invpref_kdd_2022_b200 import _lib
    from invpref_kdd_2022_b200.dataloader import interaction_csr
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    cls = InvPrefImplicit if which == "implicit" else InvPrefExplicit
    m = _model(cls)
    rng = np.random.default_rng(5)
    new_users = rng.integers(0, 4, 40)
    items = rng.integers(0, 90, 40)
    y = (rng.random(40) < 0.5).astype(np.float32) if m.implicit else rng.integers(1, 6, 40).astype(np.float32)
    off, its, ys = interaction_csr(new_users, items, y, 4)
    rows = m.fold_in_users(off, its, ys, 0.5)                                          # numpy input
    d = _dev()
    rows_t, it = m.fold_in_users(torch.from_numpy(off).to(d), torch.from_numpy(its).to(d),
                                 torch.from_numpy(ys).to(d), 0.5, return_iters=True)
    assert rows.shape == (4, 16) and rows.dtype == torch.float32 and torch.equal(rows, rows_t)
    assert it.dtype == torch.int32
    I = m.embed_item_invariant.weight.detach().cpu().numpy()
    for r in range(4):
        sel = slice(off[r], off[r + 1])
        want = ref.newton(I[its[sel]], ys[sel], 0.5, 25)[0] if m.implicit else ref.explicit(I[its[sel]], ys[sel], 0.5)
        assert np.abs(rows[r].cpu().numpy() - want).max() <= 1e-5 * max(1.0, np.abs(want).max())
    top, sc = m.recommend_rows(rows, 5, exclude=(off, its))
    assert top.shape == (4, 5)
    for r in range(4):
        assert not set(top[r].cpu().tolist()) & set(its[off[r]:off[r + 1]].tolist())
    off_i, us, ys_i = interaction_csr(rng.integers(0, 3, 30), rng.integers(0, 60, 30), ys[:30], 3)
    irows = m.fold_in_items(off_i, us, ys_i, 2.0)
    users, _ = m.top_users_rows(irows, 4)
    assert users.shape == (3, 4)
    # errors before any launch
    n0 = _lib.launch_count()
    bad = [((np.array([1, 40]), its, ys), 0.5, 25, ValueError),            # offsets do not start at 0
           ((np.array([0, 30, 20, 40]), its, ys), 0.5, 25, ValueError),     # decreasing
           ((np.array([0, 39]), its, ys), 0.5, 25, ValueError),             # does not end at len(ids)
           ((off, its, ys[:-1]), 0.5, 25, ValueError),
           ((off, its, ys), 0.0, 25, ValueError), ((off, its, ys), -1.0, 25, ValueError),
           ((off, its, ys), float("nan"), 25, ValueError), ((off, its, ys), float("inf"), 25, ValueError),
           ((off, its, ys), 0.5, 0, ValueError),
           ((off, np.where(its == its[0], 90, its), ys), 0.5, 25, IndexError),
           ((off, np.where(its == its[0], -1, its), ys), 0.5, 25, IndexError)]
    for (o, i_, s_), lam, mi, exc in bad:
        with pytest.raises(exc):
            m.fold_in_users(o, i_, s_, lam, max_iter=mi)
    with pytest.raises(IndexError):
        m.fold_in_items(off_i, np.where(us == us[0], 60, us), ys_i, 1.0)
    big = _model(cls, D=129)
    with pytest.raises(RuntimeError, match="D <= 128"):
        big.fold_in_users(off, its, ys, 1.0)
    assert _lib.launch_count() == n0
    with pytest.raises(RuntimeError):
        cls(10, 20, 2, 8).fold_in_users(off, its % 20, ys, 1.0)                      # a CPU model


@gpu
def test_lazy_flush_behaviour():
    from invpref_kdd_2022_b200.models import InvPrefExplicit
    d = _dev()
    m = InvPrefExplicit(300, 2000, 2, 64).to(d)
    hp = m.hot_path(lr=1e-2, lazy=True)
    assert hp.lazy
    rng = np.random.default_rng(4)
    t = lambda x: torch.from_numpy(x).to(d)
    for _ in range(3):
        B = 512
        hp.train_step(t(rng.integers(0, 30, B)), t(rng.integers(0, 2000, B)), t(rng.random(B).astype(np.float32)),
                      t(rng.integers(0, 2, B)), t(np.ones(B, np.float32)), c_inv=1.0, c_ea=1.0, c_env=1.0, c_L2=0.0,
                      c_L1=0.0, alpha=1.0, use_class_rw=False, use_rec_rw=False)
    assert hp._dirty
    off = np.array([0, 3, 5], np.int64)
    m.fold_in_users(off, np.array([1, 2, 3, 4, 5]), np.ones(5, np.float32), 1.0)
    assert hp._dirty                                         # reads only the item table
    users = np.array([40, 41, 299, 100, 200, 41])
    rows = m.fold_in_items(off[:2], users[:3], np.ones(3, np.float32), 1.0)
    assert not hp._dirty
    flushed = _hot(hp.params["Uinv"].clone(), hp.params["Iinv"].clone(), False)
    want = flushed.fold_in_items(t(off[:2]), t(users[:3]), t(np.ones(3, np.float32)), 1.0)
    assert torch.equal(rows.view(torch.int32), want.view(torch.int32))
    for _ in range(2):
        B = 512
        hp.train_step(t(rng.integers(0, 30, B)), t(rng.integers(0, 2000, B)), t(rng.random(B).astype(np.float32)),
                      t(rng.integers(0, 2, B)), t(np.ones(B, np.float32)), c_inv=1.0, c_ea=1.0, c_env=1.0, c_L2=0.0,
                      c_L1=0.0, alpha=1.0, use_class_rw=False, use_rec_rw=False)
    assert hp._dirty
    top, sc = m.top_users_rows(rows, 10)
    assert not hp._dirty
    flushed = _hot(hp.params["Uinv"].clone(), hp.params["Iinv"].clone(), False)
    top2, sc2 = flushed.top_users_rows(rows, 10)
    assert torch.equal(top, top2) and torch.equal(sc.view(torch.int32), sc2.view(torch.int32))


@gpu
def test_profiler_sees_both_kernels():
    from torch.profiler import ProfilerActivity, profile
    names = set()
    for implicit in (False, True):
        U, I = _tables(20, 30, 8, 9)
        hp = _hp(U, I, implicit)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _fold(hp, "users", np.array([0, 3], np.int64), np.array([1, 2, 3], np.int64), np.ones(3, np.float32), 1.0)
            torch.cuda.synchronize()
        names |= {e.name for e in prof.events() if "fold_in_kernel" in e.name}
    assert any("fold_in_kernel<false>" in n or "ILb0E" in n for n in names), names
    assert any("fold_in_kernel<true>" in n or "ILb1E" in n for n in names), names

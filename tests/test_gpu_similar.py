"""``invpref_similar_items`` / ``model.similar_items`` (cosine item-to-item top-k) and ``invpref_top_users`` /
``model.top_users`` (item-to-user top-k): the streaming top-k kernel of eval.cu with other query and catalogue tables,
against the exact references of test_gpu_eval_topk.py and test_gpu_recommend.py.

Cosine is checked bit for bit on an exact family: rows with entries in {-1, 0, 1} and exactly 4^m non-zeros, so that
|row| = 2^m and every cosine is an integer over 2^(m_q + m_i), exact in fp32 whatever the summation order, with large
tie groups.  Zero rows, non-finite rows and rows whose squared norm overflows fp32 join that family with the scores
the header defines for them.  Dense random rows are checked against the fp64 cosine through intervals whose width
follows from the documented operation order.  top_users is recommend with the tables swapped: integer and
exact-sigmoid tables give every key exactly.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from test_gpu_eval_topk import Tables, check_interval_topk, csr_of, dense_lists, exact_sigmoid, one_hot, random_lists
from test_gpu_recommend import EXCL_CASES, SLICES, TI, TU, _hot, _model, ref_recommend, slice_edges

gpu = pytest.mark.gpu
U32 = 2.0 ** -24            # unit roundoff of fp32


# ---- the exact cosine family --------------------------------------------------------------------------------------
def exact_rows(rng, n, D):
    """fp32 [n, D]: entries in {-1, 0, 1}, row i with exactly 4^m[i] non-zeros at random places (4^m <= D), so its
    norm is 2^m[i]."""
    mmax = 0
    while 4 ** (mmax + 1) <= D:
        mmax += 1
    m = rng.integers(0, mmax + 1, n)
    rank = np.argsort(np.argsort(rng.random((n, D)), axis=1), axis=1)      # a random permutation of 0..D-1 per row
    signs = rng.choice(np.array([-1.0, 1.0], np.float32), (n, D))
    return np.where(rank < (4 ** m)[:, None], signs, np.float32(0)).astype(np.float32)


def add_special_rows(rng, X, n_zero=0, n_nan=0, n_inf=0, n_huge=0):
    """Rows set to zero, rows with one NaN or one +-inf entry, and rows (1e20 on dims 0..3) whose squared norm
    overflows fp32; returns the ids of each kind."""
    n, D = X.shape
    ids = rng.choice(n, n_zero + n_nan + n_inf + n_huge, replace=False)
    z, nn, nf, hg = np.split(ids, np.cumsum([n_zero, n_nan, n_inf]))
    X[z] = 0.0
    X[nn, rng.integers(0, D, nn.size)] = np.nan
    X[nf, rng.integers(0, D, nf.size)] = rng.choice([np.inf, -np.inf], nf.size)
    if hg.size:
        assert D >= 4
        X[hg] = 0.0
        X[hg, :4] = np.float32(1e20)
    return z, nn, nf, hg


def ref_cos_keys(X, q):
    """fp32 [b, n]: the scores invpref_similar_items defines -- (z * inv_norm[q]) * inv_norm[i] + 0 with
    inv_norm = 1 / sqrt(fp32 sum of squares), 0 for a zero sum -- for rows of the exact family (where every step is
    exact) and the special rows of add_special_rows: NaN wherever a row holds NaN or inf, +0 for a zero row against a
    finite row, and for an overflowing row (inverse norm 1 / inf = 0) +0 against finite rows and NaN against another
    overflowing row (their dot product is +inf in fp32)."""
    X = np.asarray(X, dtype=np.float32)
    q = np.asarray(q, dtype=np.int64)
    fin = np.isfinite(X).all(1)
    Xf = np.where(fin[:, None], X, np.float32(0)).astype(np.float64)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        n2 = (Xf * Xf).sum(1).astype(np.float32).astype(np.float64)
        inv = np.where(n2 == 0, 0.0, 1.0 / np.sqrt(n2))
        z = (Xf[q] @ Xf.T).astype(np.float32).astype(np.float64)
        s = (z * inv[q][:, None]) * inv[None, :] + 0.0
    s = np.where(fin[q][:, None] & fin[None, :], s, np.nan)
    return s.astype(np.float32)


def kernel_order_fp32(X, q):
    """The documented operation order in plain fp32 (a multiply and an add where the kernel has one fmaf; on the exact
    family no step rounds, so both agree)."""
    X = np.asarray(X, dtype=np.float32)
    n, D = X.shape
    n2 = np.zeros(n, np.float32)
    z = np.zeros((len(q), n), np.float32)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        for d in range(D):
            n2 = n2 + X[:, d] * X[:, d]
            z = z + X[q, d][:, None] * X[None, :, d]
        inv = np.where(n2 == 0, np.float32(0), np.float32(1) / np.sqrt(n2)).astype(np.float32)
        return (z * inv[q][:, None]) * inv[None, :] + np.float32(0)


def self_excluded(q, n):
    ex = np.zeros((len(q), n), dtype=bool)
    ex[np.arange(len(q)), q] = True
    return ex


def assert_same(top, sc, want, ws, what):
    bad = np.argwhere(top != want)
    assert bad.size == 0, (what, bad[:5].tolist(), top[tuple(bad[0])], want[tuple(bad[0])])
    assert np.array_equal(np.isnan(sc), np.isnan(ws)), what
    fin = ~np.isnan(ws)
    assert np.array_equal(sc[fin].view(np.uint32), ws[fin].view(np.uint32)), what          # bit for bit


# ---- calling the library ------------------------------------------------------------------------------------------
def _items_hot(It, implicit=False):
    """A HotPath whose item table is It (the user table is a small stand-in: similar_items reads only items)."""
    Ut = torch.zeros((3, It.shape[1]), dtype=torch.float32, device=It.device)
    return _hot(Ut, It, implicit)


def run_similar(X, q, ks, implicit=False):
    dev = torch.device("cuda:0")
    q = np.asarray(q, dtype=np.int64)
    hp = _items_hot(torch.from_numpy(np.ascontiguousarray(X)).to(dev), implicit)
    keys = ref_cos_keys(X, q)
    excluded = self_excluded(q, X.shape[0])
    qt = torch.from_numpy(q).to(dev)
    for k in ks:
        top, sc = hp.similar_items(qt, k)
        want, ws = ref_recommend(keys, excluded, k)
        assert_same(top.cpu().numpy(), sc.cpu().numpy(), want, ws, k)


def run_top_users(tab, implicit, items, ks, excl=None):
    """top_users on tables where `tab` is seen from the items: tab.U = the item table (queries), tab's catalogue = the
    user table; keys[r, u] = score(u, items[r]) exactly (explicit, or implicit with z in the exact set)."""
    dev = torch.device("cuda:0")
    items = np.asarray(items, dtype=np.int64)
    It, Ut = tab.device(dev)
    hp = _hot(Ut, It, implicit)
    z = tab.z(items)
    keys = exact_sigmoid(z) if implicit else z.astype(np.float32)
    excluded = dense_lists(excl, items, tab.n_items)
    ex = None if excl is None else tuple(torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in excl)
    it = torch.from_numpy(items).to(dev)
    for k in ks:
        top, sc = hp.top_users(it, k, ex)
        want, ws = ref_recommend(keys, excluded, k)
        assert_same(top.cpu().numpy(), sc.cpu().numpy(), want, ws, k)


def exact_implicit_tables(rng, n_items, n_users, D):
    """Item rows in {0, 1, 2}^D, one-hot user rows a(u) e_c(u) with a in {0, 17, 30, -89, -200}: every z is in the set
    where the fp32 sigmoid is exact (0, >= 17, <= -89)."""
    return Tables(rng.integers(0, 3, (n_items, D)), a=rng.choice([0.0, 17.0, 30.0, -89.0, -200.0], n_users),
                  c=rng.integers(0, D, n_users))


# ==== CPU: the references ===========================================================================================
@pytest.mark.parametrize("D", [1, 3, 17, 40, 64, 256])
def test_exact_family_norms_and_cosines_are_exact(D):
    """Norms are powers of two, and the documented operation order in fp32 reproduces the fp64 reference bit for bit:
    no step rounds, so the kernel's order of summation cannot matter."""
    rng = np.random.default_rng(D)
    X = exact_rows(rng, 300, D)
    assert set(np.unique(X).tolist()) <= {-1.0, 0.0, 1.0}
    nnz = (X != 0).sum(1)
    assert np.isin(nnz, [4 ** m for m in range(5)]).all() and (nnz <= D).all()
    assert len(np.unique(nnz)) == len([m for m in range(5) if 4 ** m <= D])
    q = np.concatenate([np.arange(10), rng.integers(0, 300, 20)])
    want = ref_cos_keys(X, q)
    got = kernel_order_fp32(X, q)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert not np.signbit(want[want == 0]).any()                        # a zero cosine is +0
    assert len(np.unique(want)) < want.size // 4                          # large tie groups


def test_special_rows_reference():
    rng = np.random.default_rng(7)
    X = exact_rows(rng, 200, 17)
    z, nn, nf, hg = add_special_rows(rng, X, 10, 5, 5, 6)
    q = np.concatenate([z[:2], nn[:2], nf[:2], hg[:2], [i for i in range(200) if i not in set(np.r_[z, nn, nf, hg])][:4]])
    s = ref_cos_keys(X, q)
    got = kernel_order_fp32(X, q)
    assert np.array_equal(np.isnan(s), np.isnan(got))
    assert np.array_equal(s[~np.isnan(s)].view(np.uint32), got[~np.isnan(got)].view(np.uint32))
    bad = np.r_[nn, nf]
    assert np.isnan(s[:, bad]).all() and np.isnan(s[2:6]).all()
    ok = np.setdiff1d(np.arange(200), bad)
    assert (s[:2][:, ok].view(np.uint32) == 0).all()                         # zero rows: +0 against finite rows
    finite_ok = np.setdiff1d(ok, hg)
    assert (s[6:8][:, finite_ok].view(np.uint32) == 0).all()                 # overflowing rows: +0 ...
    assert np.isnan(s[6:8][:, hg]).all()                                     # ... NaN against each other


def test_dense_cosine_bound_holds_for_the_documented_order():
    """The interval half-width of the dense test, (2D + 8) * 2^-24, bounds the fp32 evaluation of the documented order
    (here with separate roundings of every multiply and add, a looser evaluation than the kernel's fmaf)."""
    rng = np.random.default_rng(3)
    for D in (3, 17, 64, 256):
        X = (rng.standard_normal((400, D)) * np.exp2(rng.integers(-20, 21, (400, 1)))).astype(np.float32)
        q = np.arange(40)
        got = kernel_order_fp32(X, q).astype(np.float64)
        Xd = X.astype(np.float64)
        nrm = np.linalg.norm(Xd, axis=1)
        cos = (Xd[q] @ Xd.T) / nrm[q][:, None] / nrm[None, :]
        assert np.abs(got - cos).max() <= (2 * D + 8) * U32, D


def test_transposed_csr_lists_the_users_of_each_item():
    from invpref_kdd_2022_b200.dataloader import user_item_csr
    rng = np.random.default_rng(5)
    u, i = rng.integers(0, 30, 700), rng.integers(0, 50, 700)
    off, users = user_item_csr(i, u, 50)
    assert off.size == 51 and off.dtype == np.int64 and users.dtype == np.int64
    for item in range(50):
        assert users[off[item]:off[item + 1]].tolist() == sorted(set(u[i == item].tolist()))


def test_argument_checks_come_before_any_launch():
    """Bad sizes are INVPREF_ERR_BAD_ARG and b == 0 is a no-op, with no device memory touched (null pointers)."""
    from invpref_kdd_2022_b200 import _lib
    lib = _lib.load()
    d = _lib.make_desc(50, 100, 2, 16, 0, 0, 0)
    p = _lib.Params(*([C.c_void_p(256)] * 7))          # never dereferenced on these paths
    one = C.c_void_p(512)
    sim = lambda b, k, items=one, inv=one: lib.invpref_similar_items(C.byref(d), C.byref(p), items, b, k, inv, one,
                                                                      one, None)
    top = lambda b, k, off=None, ex=None: lib.invpref_top_users(C.byref(d), C.byref(p), one, b, off, ex, k, one, one,
                                                                None)
    for k in (0, -1, 257, 101):
        assert sim(1, k) == -3
    for k in (0, 257, 51):
        assert top(1, k) == -3
    assert sim(-1, 5) == -3 and top(-1, 5) == -3
    assert sim(1, 5, items=None) == -3 and sim(1, 5, inv=None) == -3
    assert top(1, 5, off=one, ex=None) == -3
    assert sim(0, 5, items=None, inv=None) == 0 and top(0, 50) == 0
    assert lib.invpref_similar_items(C.byref(d), None, one, 1, 5, one, one, one, None) == -3


# ==== GPU: similar_items, exact ======================================================================================
def _size_cases():
    return [1, 2, TI - 1, TI, TI + 1, SLICES * TI - 1, SLICES * TI, SLICES * TI + 1, 4099, (1 << 20) + 3]


@gpu
@pytest.mark.parametrize("n_items", _size_cases())
def test_similar_items_item_counts(n_items):
    """Partial, full and one-past item tiles, the smallest catalogue split over 8 cluster slices and one item either
    side of it, 2^20 + 3 items; queries on item 0, the last item and the slice edges, a repeated query."""
    rng = np.random.default_rng(n_items)
    X = exact_rows(rng, n_items, 17)
    q = [0, n_items - 1, 0] + (slice_edges(n_items) if n_items >= SLICES * TI else [n_items // 2])
    ks = sorted({1, min(n_items, 37), min(n_items, 256)})
    run_similar(X, q, ks)


@gpu
@pytest.mark.parametrize("D", [1, 3, 17, 40, 64, 128, 256])
def test_similar_items_dims(D):
    """Scalar and float4 dims, one and several staged chunks of the item tile."""
    rng = np.random.default_rng(100 + D)
    X = exact_rows(rng, 3001, D)
    run_similar(X, rng.integers(0, 3001, 6), [1, 33, 256])


@gpu
@pytest.mark.parametrize("k", [1, 2, 31, 32, 33, 255, 256])
def test_similar_items_k(k):
    rng = np.random.default_rng(200 + k)
    X = exact_rows(rng, 20000, 17)
    run_similar(X, rng.integers(0, 20000, 7), [k])


@gpu
@pytest.mark.parametrize("n_items", [1, 2, 200, 256])
def test_similar_items_k_equals_n_items(n_items):
    """Every other item, ranked; the last slot is item -1 / score -inf because the query itself is left out."""
    rng = np.random.default_rng(300 + n_items)
    X = exact_rows(rng, n_items, 17)
    q = np.arange(n_items) if n_items <= 2 else rng.integers(0, n_items, 9)
    run_similar(X, q, [n_items])


@gpu
@pytest.mark.parametrize("b", [1, TU - 1, TU, TU + 1, 65537])
def test_similar_items_batch_sizes(b):
    """Partial, full and one-past query tiles and 65 537 queries, repeated query ids in the batch."""
    rng = np.random.default_rng(400 + b)
    n = 300 if b > 1000 else 5000
    X = exact_rows(rng, n, 17)
    q = rng.integers(0, n, b)
    if b > 1:
        q[-1] = q[0]
    run_similar(X, q, [40])


@gpu
@pytest.mark.parametrize("D", [17, 64])
def test_similar_items_zero_nan_inf_and_overflowing_rows(D):
    """Zero rows (+0 against everything finite: ties by id), rows with a NaN or an inf entry (NaN against every row:
    on top), rows whose squared norm overflows fp32 (+0 against finite rows, NaN against each other); queries of
    each kind, k up to 256 so that the NaN group, the +0 group and the self-exclusion all fall inside the top k."""
    rng = np.random.default_rng(500 + D)
    n = 4099
    X = exact_rows(rng, n, D)
    z, nn, nf, hg = add_special_rows(rng, X, 400, 30, 30, 20)
    q = np.concatenate([z[:3], nn[:2], nf[:2], hg[:3], rng.integers(0, n, 6)])
    run_similar(X, q, [1, 25, 70, 256])


@gpu
def test_similar_items_all_zero_rows():
    """Every score +0: the k lowest ids other than the query, in order."""
    X = np.zeros((3000, 8), np.float32)
    q = np.array([0, 5, 2999, 5])
    run_similar(X, q, [1, 10, 256])
    hp = _items_hot(torch.from_numpy(X).cuda())
    top, sc = hp.similar_items(torch.tensor([5], device="cuda:0"), 8)
    assert top.cpu().tolist() == [[0, 1, 2, 3, 4, 6, 7, 8]]
    assert (sc.cpu().numpy().view(np.uint32) == 0).all()


@gpu
def test_similar_items_ignores_the_sigmoid_of_the_implicit_model():
    rng = np.random.default_rng(8)
    X = exact_rows(rng, 2100, 40)
    run_similar(X, rng.integers(0, 2100, 5), [1, 50], implicit=True)


# ==== GPU: similar_items, dense rows ================================================================================
@gpu
@pytest.mark.parametrize("D", [3, 40, 64, 256])
def test_similar_items_dense_rows_against_fp64(D):
    """Random normal rows with norms spread over 2^-20 .. 2^20 against the fp64 cosine.  Bound per score:
    (2D + 8) * 2^-24 -- the fmaf chain of z contributes D u |q| |x|, the two inverse norms (D / 2 + 2) u each relative,
    the two products u each -- so a returned score lies in [cos - bound, cos + bound] rounded outwards to fp32.
    Ranks the intervals cannot order must stay few: at most twice the number of neighbouring fp64 cosines in the top
    k + 1 that lie within twice the bound of each other (which no evaluation within the bound could order), plus 5."""
    rng = np.random.default_rng(600 + D)
    n, b, k = 20011, 24, 50
    X = (rng.standard_normal((n, D)) * np.exp2(rng.integers(-20, 21, (n, 1)))).astype(np.float32)
    q = rng.integers(0, n, b)
    dev = torch.device("cuda:0")
    hp = _items_hot(torch.from_numpy(X).to(dev))
    top, sc = hp.similar_items(torch.from_numpy(q).to(dev), k)
    top, sc = top.cpu().numpy(), sc.cpu().numpy()
    Xd = X.astype(np.float64)
    nrm = np.linalg.norm(Xd, axis=1)
    cos = (Xd[q] @ Xd.T) / nrm[q][:, None] / nrm[None, :]
    bound = (2 * D + 8) * U32
    lo = np.nextafter((cos - bound).astype(np.float32), np.float32(-np.inf))
    hi = np.nextafter((cos + bound).astype(np.float32), np.float32(np.inf))
    lo[np.arange(b), q] = hi[np.arange(b), q] = -np.inf                       # the query itself: never a candidate
    cls = np.broadcast_to(np.arange(n, dtype=np.float64), (b, n))             # no two rows alike
    assert not (top == q[:, None]).any()
    undecided = check_interval_topk(top, sc, lo, hi, cls, k)
    c = cos.copy()
    c[np.arange(b), q] = -np.inf
    best = -np.sort(-c, axis=1)[:, :k + 1]
    inseparable = int((best[:, :-1] - best[:, 1:] <= 2 * bound).sum())
    assert undecided <= 2 * inseparable + 5, (undecided, inseparable)


# ==== GPU: top_users ================================================================================================
@gpu
@pytest.mark.parametrize("n_users", [1, TI - 1, TI, TI + 1, SLICES * TI - 1, SLICES * TI, SLICES * TI + 1, 4099,
                                     (1 << 20) + 3])
def test_top_users_user_counts(n_users):
    """User tiles at and around their edges, 8 cluster slices, 2^20 + 3 users; one-hot user rows (many equal
    scores), transposed exclusion lists with entries outside [0, n_users), a repeated item."""
    rng = np.random.default_rng(700 + n_users)
    n_items = 6
    tab = one_hot(rng, n_items, n_users, 40, False)
    excl = random_lists(rng, n_items, n_users, min(300, max(1, n_users // 4)))
    ks = sorted({1, min(n_users, 37), min(n_users, 256)})
    run_top_users(tab, False, [0, 1, 4, 1, 5], ks, excl)


@gpu
@pytest.mark.parametrize("n_users", [TI + 1, SLICES * TI + 1, (1 << 20) + 3])
def test_top_users_implicit_exact_sigmoid(n_users):
    rng = np.random.default_rng(800 + n_users)
    tab = exact_implicit_tables(rng, 5, n_users, 16)
    excl = random_lists(rng, 5, n_users, 40)
    run_top_users(tab, True, [0, 3, 4, 3], sorted({1, min(n_users, 60), min(n_users, 256)}), excl)


def _excl_case(case, rng, n_q, n):
    """The exclusion lists of test_gpu_recommend.test_recommend_exclusion, over n_q query rows and n catalogue rows."""
    excl = random_lists(rng, n_q, n, 40, out_of_range=False)
    if case == "empty_lists":
        return csr_of([np.zeros(0, np.int64)] * n_q)
    if case == "every_item":                         # all -1 and -inf
        return csr_of([np.arange(n)] * n_q)
    if case == "fewer_than_k":
        keep = [rng.choice(n, j, replace=False) for j in (0, 1, 3, 63, 10)]
        return csr_of([np.setdiff1d(np.arange(n), kp) for kp in keep])
    if case == "out_of_range":
        return csr_of([np.concatenate([[-(2 ** 40), -5, -1], excl[1][excl[0][u]:excl[0][u + 1]], [n, n + 1, 2 ** 40]])
                       for u in range(n_q)])
    if case == "long_lists_across_edges":
        edges = [TI * 9] + slice_edges(n)
        return csr_of([np.unique(np.concatenate([np.arange(e - 300, e + 300) for e in edges[u % 3::2]]))
                       for u in range(n_q)])
    assert case == "no_lists"
    return None


@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
@pytest.mark.parametrize("case", EXCL_CASES)
def test_top_users_exclusion(case, implicit):
    rng = np.random.default_rng(900 + EXCL_CASES.index(case) + 10 * implicit)
    n_items, n = 5, 20011
    tab = exact_implicit_tables(rng, n_items, n, 8) if implicit else one_hot(rng, n_items, n, 8, False, a_range=30)
    run_top_users(tab, implicit, np.arange(n_items), [1, 64, 256], _excl_case(case, rng, n_items, n))


@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
def test_top_users_and_recommend_give_the_same_score_bits(implicit):
    """Dense random tables: every (user, item) score of top_users(all items, k = n_users) equals the one of
    recommend(all users, k = n_items) bit for bit (the fmaf operands are swapped, the products are the same)."""
    rng = np.random.default_rng(10 + implicit)
    n_users, n_items, D = 200, 256, 40
    dev = torch.device("cuda:0")
    Ut = torch.from_numpy(rng.standard_normal((n_users, D)).astype(np.float32)).to(dev)
    It = torch.from_numpy(rng.standard_normal((n_items, D)).astype(np.float32)).to(dev)
    hp = _hot(Ut, It, implicit)
    tr, sr = hp.recommend(torch.arange(n_users, device=dev), n_items)
    tu, su = hp.top_users(torch.arange(n_items, device=dev), n_users)
    tr, sr, tu, su = (x.cpu().numpy() for x in (tr, sr, tu, su))
    by_rec = np.full((n_users, n_items), np.nan, np.float32)
    by_rec[np.arange(n_users)[:, None], tr] = sr
    by_top = np.full((n_users, n_items), np.nan, np.float32)
    by_top[tu, np.arange(n_items)[:, None]] = su
    assert not np.isnan(by_rec).any() and not np.isnan(by_top).any()      # every pair once
    assert np.array_equal(by_rec.view(np.uint32), by_top.view(np.uint32))


# ==== GPU: model API ================================================================================================
def _set_items(m, X):
    with torch.no_grad():
        m.embed_item_invariant.weight.copy_(torch.from_numpy(X))


@gpu
@pytest.mark.parametrize("which", ["explicit", "implicit"])
def test_model_similar_items_and_top_users_match_the_reference(which):
    from invpref_kdd_2022_b200.dataloader import user_item_csr
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    dev = torch.device("cuda:0")
    cls = InvPrefImplicit if which == "implicit" else InvPrefExplicit
    m = _model(cls, dev)                        # 50 users, 3000 items, D 16, integer rows
    rng = np.random.default_rng(12)
    # top_users: the transposed keys of recommend's integer tables (see test_gpu_recommend._model)
    pairs = np.stack([rng.integers(0, 50, 4000), rng.integers(0, 3000, 4000)], 1)
    off, users = user_item_csr(pairs[:, 1], pairs[:, 0], 3000)
    items = np.array([7, 0, 2999, 7, 1234])
    U = m.embed_user_invariant.weight.detach().cpu().numpy().astype(np.float64)
    I = m.embed_item_invariant.weight.detach().cpu().numpy().astype(np.float64)
    z = I[items] @ U.T + 0.0
    for excl in (None, (off, users), (torch.from_numpy(off).to(dev), torch.from_numpy(users).to(dev))):
        top, sc = m.top_users(items, 20, exclude=excl)
        assert top.dtype == torch.int64 and sc.dtype == torch.float32 and top.shape == (5, 20)
        ex = dense_lists(None if excl is None else (off, users), items, 50)
        want, _ = ref_recommend(z, ex, 20)
        assert np.array_equal(top.cpu().numpy(), want)
        if which == "explicit":                                      # integer scores: exact
            assert np.array_equal(sc.cpu().numpy(), np.take_along_axis(z, want, 1).astype(np.float32))
    # similar_items: exact-family item rows, numpy and tensor ids
    X = exact_rows(rng, 3000, 16)
    add_special_rows(rng, X, n_zero=40)
    _set_items(m, X)
    q = np.array([3, 0, 2999, 3])
    want, ws = ref_recommend(ref_cos_keys(X, q), self_excluded(q, 3000), 30)
    for ids in (q, torch.from_numpy(q).to(dev)):
        top, sc = m.similar_items(ids, 30)
        assert_same(top.cpu().numpy(), sc.cpu().numpy(), want, ws, which)


def _lazy_model(dev):
    from invpref_kdd_2022_b200.models import InvPrefExplicit
    m = InvPrefExplicit(300, 2000, 2, 64).to(dev)
    hp = m.hot_path(lr=1e-2, lazy=True)
    assert hp.lazy
    rng = np.random.default_rng(4)
    t = lambda x: torch.from_numpy(x).to(dev)
    for _ in range(4):
        B = 512
        hp.train_step(t(rng.integers(0, 30, B)), t(rng.integers(0, 2000, B)), t(rng.random(B).astype(np.float32)),
                      t(rng.integers(0, 2, B)), t(np.ones(B, np.float32)), c_inv=1.0, c_ea=1.0, c_env=1.0, c_L2=0.0,
                      c_L1=0.0, alpha=1.0, use_class_rw=False, use_rec_rw=False)
    assert hp._dirty
    return m, hp


@gpu
def test_model_top_users_after_lazy_steps_equals_flushed_tables():
    """After lazy-Adam train steps without a flush, top_users sees the caught-up user rows: it equals top_users on a
    copy of the flushed tables."""
    dev = torch.device("cuda:0")
    m, hp = _lazy_model(dev)
    items = torch.arange(3, 2000, 97, device=dev)
    top, sc = m.top_users(items, 30)
    assert not hp._dirty
    ref = _hot(hp.params["Uinv"].clone(), hp.params["Iinv"].clone(), False)
    top2, sc2 = ref.top_users(items, 30)
    assert torch.equal(top, top2) and torch.equal(sc.view(torch.int32), sc2.view(torch.int32))


@gpu
def test_model_similar_items_needs_no_flush():
    """similar_items reads only the item table, which lazy Adam never defers: the user rows stay behind."""
    dev = torch.device("cuda:0")
    m, hp = _lazy_model(dev)
    items = torch.arange(0, 2000, 111, device=dev)
    top, sc = m.similar_items(items, 40)
    assert hp._dirty
    ref = _items_hot(hp.params["Iinv"].clone())
    top2, sc2 = ref.similar_items(items, 40)
    assert torch.equal(top, top2) and torch.equal(sc.view(torch.int32), sc2.view(torch.int32))


@gpu
def test_model_similar_items_and_top_users_reject_bad_input():
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    dev = torch.device("cuda:0")
    m = _model(InvPrefImplicit, dev, n_items=100)       # 50 users, 100 items
    for call in (lambda ids: m.similar_items(ids, 5), lambda ids: m.top_users(ids, 5)):
        with pytest.raises(IndexError):
            call(torch.tensor([0, 100], device=dev))
        with pytest.raises(IndexError):
            call(torch.tensor([-1], device=dev))
    for k in (0, 257, 101):                              # 101 > n_items
        with pytest.raises(RuntimeError, match="bad argument"):
            m.similar_items(torch.tensor([0], device=dev), k)
    for k in (0, 257, 51):                               # 51 > n_users
        with pytest.raises(RuntimeError, match="bad argument"):
            m.top_users(torch.tensor([0], device=dev), k)
    top, sc = m.similar_items(torch.tensor([4], device=dev), 100)
    assert sorted(top[0, :99].cpu().tolist()) == [i for i in range(100) if i != 4]
    assert top[0, 99].item() == -1 and sc[0, 99].item() == float("-inf")
    top, sc = m.top_users(torch.tensor([4], device=dev), 50)
    assert sorted(top[0].cpu().tolist()) == list(range(50))
    for call in (lambda: m.similar_items(torch.zeros(0, dtype=torch.int64, device=dev), 5),
                 lambda: m.top_users(np.zeros(0, np.int64), 5)):
        top, sc = call()
        assert top.shape == (0, 5) and sc.shape == (0, 5)
    with pytest.raises(RuntimeError, match="exclude"):          # offsets shorter than n_items + 1
        m.top_users(torch.tensor([0], device=dev), 5, exclude=(np.zeros(51, np.int64), np.zeros(1, np.int64)))
    with pytest.raises(RuntimeError, match="exclude"):
        m.top_users(torch.tensor([0], device=dev), 5, exclude=(np.zeros(101, np.int32), np.zeros(1, np.int64)))
    with pytest.raises(RuntimeError, match="exclude"):
        m.top_users(torch.tensor([0], device=dev), 5, exclude=(np.zeros(101, np.int64), np.zeros(1, np.float32)))
    cpu = InvPrefExplicit(10, 20, 2, 8)
    with pytest.raises(RuntimeError):
        cpu.similar_items(torch.tensor([0]), 3)
    with pytest.raises(RuntimeError):
        cpu.top_users(torch.tensor([0]), 3)

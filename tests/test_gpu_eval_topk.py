"""The fused implicit evaluator ``invpref_eval_topk`` (eval.cu) and its two helpers ``invpref_mask_scores`` /
``invpref_hits_from_csr`` against exact host references.

The evaluator scores every item of a user, masks the train positives (-1024), lifts the item pool (+1024), finds the
k-th largest key by a 3-pass radix select (11 + 11 + 10 bits) and collects the survivors, ties going to the lowest
item id.  Its tables are built here so that the reference knows every key exactly:

* explicit scoring: integer-valued tables with |z| < 2^24, so every dot product is exact in fp32 in any summation
  order; ``top_items``, ``top_scores``, ``hits`` and ``n_gt`` must then match the reference bit for bit;
* one-hot item tables (row i = a(i) * e_c(i), so z_ui = a(i) * Uinv[u, c(i)]) place scores and tie groups on chosen
  item ids at any ``n_items``, in particular on each of the three shared-memory paths of ``launch_eval_topk``;
* implicit scoring: z exact on a 1/8 grid with |z| <= 8, where neighbouring sigmoid values lie hundreds of fp32 ulps
  apart; the reference gives each item an fp32 interval around the fp64 sigmoid, and z in {0, >= 17, <= -89}
  gives exactly 0.5, 1 and 0.

The reference ranking is ``np.lexsort`` per user: key descending, NaN above everything (as ``torch.topk``), ties to
the lower item id.  The tests without the ``gpu`` mark check the reference helpers themselves.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

gpu = pytest.mark.gpu

# ---- restatement of launch_eval_topk's shared-memory plan (eval.cu) ----------------------------------------------
EV_THREADS, EV_MAXK, SMEM_CAP = 256, 256, 200 * 1024
PATHS = ("cache", "bitmap", "search")      # score cache + bitmaps / bitmaps, recomputed scores / binary search


def eval_path(n_items, D):
    """Which memory path launch_eval_topk takes: 'cache' (every adjusted score kept in shared memory), 'bitmap'
    (mask / pool bitmaps, scores recomputed in each of the 3 histogram sweeps and the collect sweep) or 'search'
    (recomputed scores and a binary search in the CSR lists per item and sweep)."""
    words = (n_items + 31) // 32
    base = ((D + 3) & ~3) * 4 + 2048 * 4 + EV_THREADS * 4 + EV_MAXK * 8
    if base + 2 * words * 4 > SMEM_CAP:
        return "search"
    base += 2 * words * 4
    return "cache" if base + n_items * 4 <= SMEM_CAP else "bitmap"


def path_bounds(D):
    """(largest n_items on the cache path, largest n_items on the bitmap path) at dimension D."""
    def last(path):
        lo, hi = 1, 1 << 22                     # the path index never decreases with n_items
        while lo < hi:
            mid = (lo + hi + 1) // 2
            if PATHS.index(eval_path(mid, D)) <= PATHS.index(path):
                lo = mid
            else:
                hi = mid - 1
        return lo
    return last("cache"), last("bitmap")


# ---- reference ranking -----------------------------------------------------------------------------------------
def ref_order(keys):
    """Items of every row of fp32 `keys` [b, n] in the order the evaluator promises: key descending, NaN above
    everything (torch.topk's order), equal keys by ascending item id.  -0.0 and +0.0 are equal keys."""
    keys = np.asarray(keys, dtype=np.float64)
    b, n = keys.shape
    nan = np.isnan(keys)
    neg = np.where(nan, 0.0, -keys)
    rows = np.repeat(np.arange(b), n)
    items = np.tile(np.arange(n), b)
    order = np.lexsort((items, neg.ravel(), (~nan).ravel(), rows))
    return items[order].reshape(b, n)


def brute_order(row):
    """The same ranking of one row by pairwise comparison (checks ref_order)."""
    def above(x, y):                            # item x ranks above item y
        kx, ky = row[x], row[y]
        if np.isnan(kx) or np.isnan(ky):
            return np.isnan(kx) and (not np.isnan(ky) or x < y)
        return kx > ky or (kx == ky and x < y)
    n = len(row)
    return np.array(sorted(range(n), key=functools.cmp_to_key(lambda x, y: -1 if above(x, y) else 1)))


def dense_lists(csr, users, n_items):
    """bool [b, n_items]: item i is in the list of users[r] (entries outside [0, n_items) are ignored)."""
    m = np.zeros((len(users), n_items), dtype=bool)
    if csr is None:
        return m
    off, items = csr
    for r, u in enumerate(users):
        it = items[off[u]:off[u + 1]]
        m[r, it[(it >= 0) & (it < n_items)]] = True
    return m


def adjust(s, masked, pooled):
    """evaluate.py:98 and :110 on fp32 scores: masked := -1024, then pooled += 1024 (masked and pooled -> 0)."""
    s = np.where(masked, np.float32(-1024.0), np.asarray(s, dtype=np.float32))
    with np.errstate(invalid="ignore"):
        return np.where(pooled, s + np.float32(1024.0), s).astype(np.float32)


def exact_sigmoid(z):
    """sigmoidf_ (common.cuh: 1 / (1 + expf(-z))) where it is exact in fp32: 0.5 at 0, 1 from 17 up, 0 from -89
    down, NaN at NaN."""
    z = np.asarray(z, dtype=np.float64)
    ok = np.isnan(z) | (z == 0) | (z >= 17) | (z <= -89)
    assert ok.all(), "z outside the exact set {0, >= 17, <= -89, NaN}"
    return np.where(np.isnan(z), np.nan, np.where(z == 0, 0.5, np.where(z > 0, 1.0, 0.0))).astype(np.float32)


SIGMOID_ULPS = 8   # expf is within 2 ulp; 1 + e and the division round once each: at most 6 ulp of the sigmoid


def sigmoid_interval(z, masked, pooled):
    """fp32 bounds (lo, hi) [b, n] of the evaluator's adjusted implicit key: the fp64 sigmoid rounded to fp32,
    widened by SIGMOID_ULPS, exact where exact_sigmoid is; masked / pooled applied to both ends (fp32 rounding of
    s + 1024 is monotone, so the bounds stay bounds)."""
    z = np.asarray(z, dtype=np.float64)
    with np.errstate(over="ignore"):
        s = (1.0 / (1.0 + np.exp(-z))).astype(np.float32)
    lo, hi = s.copy(), s.copy()
    for _ in range(SIGMOID_ULPS):
        lo = np.nextafter(lo, np.float32(-np.inf))
        hi = np.nextafter(hi, np.float32(np.inf))
    lo, hi = np.maximum(lo, np.float32(0)), np.minimum(hi, np.float32(1))
    ex = np.isnan(z) | (z == 0) | (z >= 17) | (z <= -89)
    e = exact_sigmoid(np.where(ex, z, 0.0))
    lo, hi = np.where(ex, e, lo), np.where(ex, e, hi)
    return adjust(lo, masked, pooled), adjust(hi, masked, pooled)


def check_interval_topk(top, sc, lo, hi, cls, k):
    """The evaluator's (top, scores) [b, k] against per-item key intervals [lo, hi] [b, n].  Items of one class
    `cls` [b, n] (same z, same mask / pool state) have the same key in any deterministic kernel.  Returns the number
    of ranks the intervals could not decide (items straddling the k-th score, overlapping neighbours)."""
    b, n = lo.shape
    rk = lambda x: np.where(np.isnan(x), np.inf, np.asarray(x, dtype=np.float64))   # implicit keys are finite
    lo, hi, s = rk(lo), rk(hi), rk(sc)
    assert top.shape == (b, k) and ((top >= 0) & (top < n)).all()
    assert (np.diff(np.sort(top, 1), axis=1) > 0).all(), "an item returned twice"
    L, H, K = (np.take_along_axis(x, top, 1) for x in (lo, hi, cls))
    assert ((s >= L) & (s <= H)).all(), "a returned score outside its item's interval"
    assert (s[:, :-1] >= s[:, 1:]).all(), "scores not descending"
    eq = s[:, :-1] == s[:, 1:]
    assert (top[:, :-1][eq] < top[:, 1:][eq]).all(), "equal scores not in ascending item order"
    by_cls = np.lexsort((s, K))
    Ks, ss = np.take_along_axis(K, by_cls, 1), np.take_along_axis(s, by_cls, 1)
    assert not ((Ks[:, 1:] == Ks[:, :-1]) & (ss[:, 1:] != ss[:, :-1])).any(), "one class, two scores"
    last, last_item, last_cls = s[:, -1:], top[:, -1:], K[:, -1:]
    out = np.ones((b, n), dtype=bool)
    out[np.arange(b)[:, None], top] = False
    assert not (out & (lo > last)).any(), "an item surely above the k-th score was left out"
    known_eq = ((lo == hi) & (lo == last)) | (cls == last_cls)
    ids = np.arange(n)[None, :]
    assert not (out & known_eq & (ids < last_item)).any(), "a tie at the k-th score did not go to the lowest id"
    # undecided: classes left out although their interval reaches the k-th score, and neighbouring ranks of
    # different classes whose intervals overlap without being the same single value
    r, i = np.nonzero(out & (hi >= last) & ~known_eq)
    undecided = len(np.unique(np.stack([r.astype(np.float64), cls[r, i]]), axis=1).T) if r.size else 0
    overl = (H[:, 1:] >= L[:, :-1]) & ~((L[:, 1:] == H[:, 1:]) & (L[:, :-1] == H[:, :-1]) & (L[:, 1:] == L[:, :-1]))
    overl &= K[:, 1:] != K[:, :-1]
    return undecided + int(overl.sum())


# ---- tables -------------------------------------------------------------------------------------------------------
class Tables:
    """Uinv [n_users, D] and an item table, with the exact fp64 z = Uinv[u] . Iinv[i] of any user batch.  Either
    dense (`I` given) or one-hot (row i = a[i] * e_{c[i]})."""

    def __init__(self, U, I=None, a=None, c=None):
        self.U = np.asarray(U, dtype=np.float32)
        self.D = self.U.shape[1]
        if I is not None:
            self.I = np.asarray(I, dtype=np.float32)
            self.n_items = self.I.shape[0]
            self.a = self.c = None
        else:
            self.I = None
            self.a, self.c = np.asarray(a, dtype=np.float32), np.asarray(c, dtype=np.int64)
            self.n_items = self.a.size

    def z(self, users):
        """fp64 [b, n]; `+ 0.0` because the kernel's sum starts from +0, so an all-zero product sum is +0."""
        Ub = self.U[np.asarray(users)].astype(np.float64)
        with np.errstate(invalid="ignore", over="ignore"):
            if self.I is not None:
                z = Ub @ self.I.astype(np.float64).T
            else:
                z = self.a.astype(np.float64)[None, :] * Ub[:, self.c]
        return z + 0.0

    def device(self, dev):
        Ut = torch.from_numpy(self.U).to(dev)
        if self.I is not None:
            It = torch.from_numpy(self.I).to(dev)
        else:
            It = torch.zeros((self.n_items, self.D), dtype=torch.float32, device=dev)
            It[torch.arange(self.n_items, device=dev), torch.from_numpy(self.c).to(dev)] = torch.from_numpy(self.a).to(dev)
        return Ut, It


def one_hot(rng, n_users, n_items, D, implicit, a_range=64):
    """Random one-hot tables: explicit a, U integers in [-a_range, a_range]; implicit a in [-8, 8] integers and U on
    the 1/8 grid of [-1, 1], so z is on the 1/8 grid with |z| <= 8 (many equal z: large tie classes)."""
    c = rng.integers(0, D, n_items)
    if implicit:
        a = rng.integers(-8, 9, n_items)
        U = rng.integers(-8, 9, (n_users, D)) / 8.0
    else:
        a = rng.integers(-a_range, a_range + 1, n_items)
        U = rng.integers(-a_range, a_range + 1, (n_users, D))
    return Tables(U, a=a, c=c)


def random_lists(rng, n_users, n_items, mean_len, out_of_range=True):
    """CSR over users of ascending unique item lists; with `out_of_range` some lists also hold ids < 0 and >= n_items
    (at both ends, so the lists stay sorted), which every consumer ignores."""
    lists = []
    for u in range(n_users):
        m = int(rng.integers(0, 2 * mean_len + 1))
        it = np.unique(rng.integers(0, n_items, m))
        if out_of_range and u % 3 == 1:
            it = np.concatenate([[-7, -1], it, [n_items, n_items + 5]])
        lists.append(it)
    return csr_of(lists)


def csr_of(lists):
    off = np.zeros(len(lists) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(x) for x in lists])
    items = np.concatenate([np.asarray(x, dtype=np.int64) for x in lists]) if lists else np.zeros(0, np.int64)
    return off, items.astype(np.int64)


# ---- calling the library ------------------------------------------------------------------------------------------
def _dev():
    return torch.device("cuda:0")


def call_eval_topk(Ut, It, implicit, users, k, mask=None, pool=None, gt=None, scores=True, hits=True, b=None):
    """invpref_eval_topk as ImplicitTestManager._hits_fused calls it (a HotPath on the given tables, the params
    struct of its tensors); returns (status, top, top_scores, hits, n_gt) as CUDA tensors (None where not asked)."""
    from invpref_kdd_2022_b200 import _lib
    from invpref_kdd_2022_b200.engine import HotPath
    dev = Ut.device
    E = torch.zeros((1, Ut.shape[1]), dtype=torch.float32, device=dev)
    hp = HotPath({"Uinv": Ut, "Iinv": It, "Uenv": Ut, "Ienv": It, "E": E, "W": E,
                  "b": torch.zeros(1, dtype=torch.float32, device=dev)}, implicit, False, False)
    users_t = torch.as_tensor(np.asarray(users, dtype=np.int64)).to(dev)
    nb = len(users) if b is None else b
    kk = max(int(k), 1)

    def up(lst):
        if lst is None:
            return None, None
        off, items = lst
        items = items if len(items) else np.zeros(1, np.int64)            # empty lists: a valid pointer
        return torch.from_numpy(np.ascontiguousarray(off)).to(dev), torch.from_numpy(np.ascontiguousarray(items)).to(dev)

    (m_off, m_it), (p_off, p_it), (g_off, g_it) = up(mask), up(pool), up(gt)
    top = torch.full((max(nb, 1), kk), -1, dtype=torch.int64, device=dev)
    sc = torch.full((max(nb, 1), kk), -7.0, dtype=torch.float32, device=dev) if scores else None
    ht = torch.full((max(nb, 1), kk), 7, dtype=torch.uint8, device=dev) if hits else None
    ng = torch.full((max(nb, 1),), -1, dtype=torch.int64, device=dev) if hits else None
    p = _lib.make_params(hp.params)
    rc = hp.lib.invpref_eval_topk(C.byref(hp.desc), C.byref(p), _lib.ptr(users_t), int(nb), _lib.ptr(m_off),
                                  _lib.ptr(m_it), _lib.ptr(p_off), _lib.ptr(p_it), _lib.ptr(g_off), _lib.ptr(g_it),
                                  int(k), _lib.ptr(top), _lib.ptr(sc), _lib.ptr(ht), _lib.ptr(ng), _lib.stream_ptr())
    torch.cuda.synchronize()
    return rc, top, sc, ht, ng


def run_eval_topk(tab, implicit, users, ks, mask=None, pool=None, gt=None, hits=True):
    """Runs the evaluator for every k of `ks` on the same inputs and checks each result against the reference:
    bit for bit (explicit scoring, or implicit with every z in the exact set), else by intervals.  Returns the
    number of undecided ranks (0 on the exact checks)."""
    n = tab.n_items
    users = np.asarray(users, dtype=np.int64)
    Ut, It = tab.device(_dev())
    z = tab.z(users)
    masked, pooled = dense_lists(mask, users, n), dense_lists(pool, users, n)
    exact = not implicit or bool((np.isnan(z) | (z == 0) | (z >= 17) | (z <= -89)).all())
    if exact:
        keys = adjust(exact_sigmoid(z) if implicit else z.astype(np.float32), masked, pooled)
        order = ref_order(keys)
    else:
        lo, hi = sigmoid_interval(z, masked, pooled)
        cls = np.where(masked, np.where(pooled, 3e9, 2e9), np.where(np.isnan(z), 4e9, z + 1e6 * pooled))
    in_gt = dense_lists(gt, users, n)
    undecided = 0
    for k in ks:
        rc, top, sc, ht, ng = call_eval_topk(Ut, It, implicit, users, k, mask, pool, gt, hits=hits and gt is not None)
        assert rc == 0, rc
        top, sc = top.cpu().numpy(), sc.cpu().numpy()
        if exact:
            want = order[:, :k]
            bad = np.argwhere(top != want)
            assert bad.size == 0, (k, bad[:5].tolist(), top[tuple(bad[0])], want[tuple(bad[0])])
            ws = np.take_along_axis(keys, want, 1)
            assert np.array_equal(np.isnan(sc), np.isnan(ws)), k
            fin = ~np.isnan(ws)
            assert np.array_equal(sc[fin].view(np.uint32), ws[fin].view(np.uint32)), k       # bit for bit
        else:
            undecided += check_interval_topk(top, sc, lo, hi, cls, k)
        if hits and gt is not None:
            off, _ = gt
            assert np.array_equal(ht.cpu().numpy(), np.take_along_axis(in_gt, top, 1).astype(np.uint8)), k
            assert np.array_equal(ng.cpu().numpy(), off[users + 1] - off[users]), k
    return undecided


# ==== CPU: the reference helpers ====================================================================================
def test_ref_order_matches_pairwise_ranking_on_small_random_rows():
    rng = np.random.default_rng(0)
    for trial in range(300):
        n = int(rng.integers(1, 40))
        row = rng.integers(-3, 4, n).astype(np.float32)            # few distinct values: many ties
        if trial % 3 == 0:
            sp = rng.random(n)
            row[sp < 0.1] = np.nan
            row[(sp >= 0.1) & (sp < 0.2)] = np.inf
            row[(sp >= 0.2) & (sp < 0.3)] = -np.inf
        if trial % 5 == 0:
            row[rng.random(n) < 0.3] = -0.0
        assert np.array_equal(ref_order(row[None, :])[0], brute_order(row)), row


def test_ref_order_puts_nan_above_inf_and_ties_to_the_lower_id():
    neg_nan = np.array([0xffc00000], dtype=np.uint32).view(np.float32)[0]
    row = np.array([1.0, np.nan, -np.inf, np.inf, neg_nan, -1024.0, -2000.0, 1.0, 0.0, -0.0], dtype=np.float32)
    assert ref_order(row[None, :])[0].tolist() == [1, 4, 3, 0, 7, 8, 9, 5, 6, 2]
    two = np.stack([row, row[::-1].copy()])              # rows are ranked independently
    assert ref_order(two)[1].tolist() == [5, 8, 6, 2, 9, 0, 1, 4, 3, 7]


def test_adjust_and_exact_sigmoid():
    s = np.array([3.0, -5000.0, np.nan, 0.5, 7.0], dtype=np.float32)
    m = np.array([True, False, False, True, False])
    p = np.array([True, True, True, False, False])
    assert adjust(s, m, p).tolist()[:2] == [0.0, -3976.0]
    assert np.isnan(adjust(s, m, p)[2]) and adjust(s, m, p).tolist()[3:] == [-1024.0, 7.0]
    assert exact_sigmoid([0.0, 17.0, 1e9, np.inf, -89.0, -np.inf]).tolist() == [0.5, 1.0, 1.0, 1.0, 0.0, 0.0]
    with pytest.raises(AssertionError):
        exact_sigmoid([1.0])
    lo, hi = sigmoid_interval(np.array([[1.0, 0.0, -3.5]]), np.zeros((1, 3), bool), np.array([[True, False, False]]))
    want = 1.0 / (1.0 + np.exp(-np.array([1.0, 0.0, -3.5])))
    assert lo[0, 1] == hi[0, 1] == 0.5
    assert lo[0, 2] < want[2] < hi[0, 2]
    assert lo[0, 0] == hi[0, 0] == np.float32(1024) + np.float32(want[0])      # 8 ulp of 0.73 vanish in 1024.73


def test_path_helper_matches_the_documented_thresholds():
    assert path_bounds(40) == (45500, 773504)
    assert [eval_path(n, 40) for n in (1, 45500, 45501, 773504, 773505)] == \
        ["cache", "cache", "bitmap", "bitmap", "search"]
    for D in (1, 3, 17, 40, 64, 128, 256):
        c, b = path_bounds(D)
        assert 44000 < c < 47000 and 770000 < b < 776000, D
        assert (eval_path(c, D), eval_path(c + 1, D), eval_path(b, D), eval_path(b + 1, D)) == \
            ("cache", "bitmap", "bitmap", "search")


def test_interval_check_rejects_a_wrong_order():
    z = np.array([[0.125 * j for j in range(-8, 8)]])
    lo, hi = sigmoid_interval(z, np.zeros_like(z, bool), np.zeros_like(z, bool))
    cls = z.copy()
    good = np.argsort(-z[0])[None, :4]
    sc = ((lo + hi) / 2).astype(np.float32)
    assert check_interval_topk(good, np.take_along_axis(sc, good, 1), lo, hi, cls, 4) == 0
    bad = good[:, [1, 0, 2, 3]]
    with pytest.raises(AssertionError):
        check_interval_topk(bad, np.take_along_axis(sc, bad, 1), lo, hi, cls, 4)
    skip = good.copy()
    skip[0, 3] = np.argsort(-z[0])[4]
    with pytest.raises(AssertionError):
        check_interval_topk(skip, np.take_along_axis(sc, skip, 1), lo, hi, cls, 4)


# ==== GPU: invpref_eval_topk ========================================================================================
def _path_cases():
    out = []
    for D in (40, 3):                                    # float4 and scalar dot product
        c, b = path_bounds(D)
        out += [(c, D, "cache"), (c + 1, D, "bitmap"), (b, D, "bitmap"), (b + 1, D, "search")]
    return out + [(n, 40, "cache") for n in (1, 7, 255, 256, 257, 4099)]


@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
@pytest.mark.parametrize("n_items,D,path", _path_cases(), ids=lambda v: str(v))
def test_eval_topk_on_each_memory_path(n_items, D, path, implicit):
    """Every shared-memory path at its bounds and one past them, and small item counts (one item, partial stripes
    of 256): one-hot tables with many equal scores, mask / pool / gt lists with entries outside [0, n_items),
    a duplicate user, k = 1, 37 and 256 (capped at n_items)."""
    assert eval_path(n_items, D) == path
    rng = np.random.default_rng(n_items * 7 + D + implicit)
    n_users = 6
    tab = one_hot(rng, n_users, n_items, D, implicit)
    mean = min(300, max(1, n_items // 4))
    mask, pool, gt = (random_lists(rng, n_users, n_items, mean) for _ in range(3))
    users = [0, 1, 4, 1, 5]
    ks = sorted({1, min(n_items, 37), min(n_items, 256)})
    undecided = run_eval_topk(tab, implicit, users, ks, mask, pool, gt)
    assert undecided <= 0.01 * len(users) * sum(ks), undecided


@gpu
@pytest.mark.parametrize("D", [1, 3, 17, 40, 64, 128, 256])
def test_eval_topk_dot_product_widths(D):
    """Dense integer tables (|z| <= 64 * 64 * 256 < 2^24): the scalar loop (D % 4 != 0) and the float4 loop."""
    rng = np.random.default_rng(D)
    n_users, n = 5, 997
    tab = Tables(rng.integers(-64, 65, (n_users, D)), I=rng.integers(-64, 65, (n, D)))
    mask, pool, gt = (random_lists(rng, n_users, n, 40) for _ in range(3))
    run_eval_topk(tab, False, np.arange(n_users), [1, 33, 256], mask, pool, gt)


@gpu
@pytest.mark.parametrize("k", [1, 2, 31, 32, 33, 255, 256])
def test_eval_topk_k(k):
    rng = np.random.default_rng(100 + k)
    n_users, n = 7, 4099
    tab = one_hot(rng, n_users, n, 8, False, a_range=20)
    mask, pool, gt = (random_lists(rng, n_users, n, 50) for _ in range(3))
    run_eval_topk(tab, False, np.arange(n_users), [k], mask, pool, gt)


@gpu
@pytest.mark.parametrize("n", [1, 7, 33, 200, 256])
def test_eval_topk_k_equals_n_items_on_an_arbitrary_score_matrix(n):
    """Identity item table (D = n_items): z = Uinv[u, i], any score matrix; here small integers with ties."""
    rng = np.random.default_rng(200 + n)
    n_users = 6
    tab = Tables(rng.integers(-3, 4, (n_users, n)), I=np.eye(n))
    mask, pool, gt = (random_lists(rng, n_users, n, max(1, n // 4)) for _ in range(3))
    run_eval_topk(tab, False, np.arange(n_users), [n], mask, pool, gt)


def order_key(x):
    """eval.cu's order-preserving integer image of an fp32 score (used here only to state what a case covers)."""
    b = np.asarray(x, dtype=np.float32).view(np.uint32).astype(np.uint64)
    return np.where(b & 0x80000000, ~b & 0xffffffff, b | 0x80000000)


def need_eq(keys, k):
    """How many items equal to the k-th largest key belong to the top k (the radix select's need_eq)."""
    kth = np.sort(keys)[::-1][k - 1]
    return k - int((keys > kth).sum())


def _tie_layout(name, rng):
    """(item scores a [n], k, need_eq of the row a, tie group ids) of one tie-group layout.  `negative_<layout>`:
    the same threshold structure with every key negative."""
    if name.startswith("negative_"):
        a, k, eq, grp = _tie_layout(name[len("negative_"):], rng)
        if name.startswith("negative_top_"):   # group values negated (same bits below the sign), all else below
            a[grp] = -a[grp]
            rest = np.setdiff1d(np.arange(a.size), grp)
            a[rest] = a[grp].min() - 1 - rng.integers(0, 1000, rest.size)
        else:                                  # shifted below zero, order unchanged
            a -= a.max() + 1
        return a, k, eq, grp
    n = 60000 if name == "all_equal_n60000" else 4099
    a = rng.integers(-40, 41, n).astype(np.float64)
    free = lambda m, avoid=(): rng.choice(np.setdiff1d(np.arange(n), np.asarray(avoid, np.int64)), m, replace=False)
    if name == "need_eq_1":                    # k - 1 distinct scores above, group of 50 at the threshold
        k, grp = 40, free(50)
        a[grp] = 50
        a[free(39, grp)] = 100 + np.arange(39)
        return a, k, 1, grp
    if name in ("part_of_group", "whole_group"):
        k, size, above = 100, (300 if name == "part_of_group" else 40), 90 if name == "part_of_group" else 60
        grp = free(size)
        a[grp] = 500
        a[free(above, grp)] = 1000 + np.arange(above)
        return a, k, k - above, grp
    if name == "group_of_1025_over_17_stripes":   # ids 1 mod 4: every stripe of 256, every warp
        grp = np.arange(1, n, 4)
        a[grp] = 500
        a[free(100, grp)] = 1000 + np.arange(100)
        return a, 256, 156, grp
    if name == "group_on_stripe_edges":
        grp = np.array([0, 255, 256, 511, 512, 767, 2047, 2048, 4098])
        a[grp] = 500
        a[free(3, grp)] = 1000 + np.arange(3)
        return a, 8, 5, grp
    if name == "group_at_the_last_items":
        grp = np.array([4095, 4097, 4098])
        a[grp] = 500
        a[free(4, grp)] = 1000 + np.arange(4)
        return a, 6, 2, grp
    if name.startswith("all_equal"):
        a[:] = 7
        return a, 256, 256, np.arange(n)
    if name in ("top_11_bits_shared", "top_22_bits_shared"):     # radix pass 2 / pass 3 decides
        vals = (1025 + np.arange(6)) if name == "top_11_bits_shared" else (2 ** 23 + 1 + np.arange(6))
        grp = free(300)
        a[grp] = vals[np.arange(300) % 6]
        return a, 170, 20, grp                 # three values of 50 items above, 20 of the fourth's 50
    raise KeyError(name)


TIE_LAYOUTS = ["need_eq_1", "part_of_group", "whole_group", "group_of_1025_over_17_stripes", "group_on_stripe_edges",
               "group_at_the_last_items", "all_equal", "all_equal_n60000", "top_11_bits_shared", "top_22_bits_shared",
               "negative_part_of_group", "negative_group_of_1025_over_17_stripes", "negative_top_11_bits_shared",
               "negative_top_22_bits_shared"]


@gpu
@pytest.mark.parametrize("name", TIE_LAYOUTS)
def test_eval_topk_tie_groups_at_the_threshold(name):
    """Tie groups placed on chosen item ids (D = 1: z = a(i) * Uinv[u]).  User 0 sees the layout as built and user 1
    scaled by 2, both with the group at the k-th score; user 2 sees it negated, which moves the group to the bottom
    of the row.  The negative_ layouts put a group of negative keys at the threshold, also where radix pass 2 or 3
    has to split it.  The group at the k-th score must go to its lowest ids, in ascending order."""
    rng = np.random.default_rng(TIE_LAYOUTS.index(name))
    a, k, want_eq, grp = _tie_layout(name, rng)
    n = a.size
    if want_eq is not None:
        assert need_eq(a, k) == want_eq
    if name.startswith("negative_"):
        assert (a < 0).all()
    if "top_" in name:
        bits = 11 if "top_11" in name else 22
        for scale in (1, 2, -1):
            ks = order_key(np.unique(a[grp]) * scale)
            assert len(np.unique(ks >> (32 - bits))) == 1 and len(np.unique(ks)) == 6
    tab = Tables(np.array([[1.0], [2.0], [-1.0]]), a=a, c=np.zeros(n, np.int64))
    gt = random_lists(rng, 3, n, 60)
    mask = pool = None
    if name == "all_equal_n60000":                                             # bitmap path, recomputed scores
        assert eval_path(n, 1) == "bitmap"
        mask, pool = random_lists(rng, 3, n, 100), random_lists(rng, 3, n, 100)
    run_eval_topk(tab, False, [0, 1, 2], [k, 256], mask, pool, gt)


@gpu
@pytest.mark.parametrize("case", ["all_negative", "mixed_signs"])
def test_eval_topk_signs_and_scores_below_the_mask_value(case):
    """Negative keys (the order key flips every bit of a negative float) and unmasked scores below -1024, which rank
    under the masked items."""
    rng = np.random.default_rng(7 if case == "all_negative" else 8)
    n = 4099
    a = rng.integers(-3000, 0, n) if case == "all_negative" else rng.integers(-3000, 3001, n)
    U = np.array([[1.0], [2.0], [3.0]]) if case == "all_negative" else np.array([[1.0], [-1.0], [2.0]])
    tab = Tables(U, a=a, c=np.zeros(n, np.int64))
    mask = csr_of([np.arange(0, n, 7), np.arange(3, 900, 2), np.zeros(0, np.int64)])
    pool = csr_of([np.arange(5, n, 11), np.zeros(0, np.int64), np.arange(0, n, 3)])
    gt = random_lists(rng, 3, n, 100)
    assert (tab.z([0]) < -1024).any()
    run_eval_topk(tab, False, [0, 1, 2], [1, 100, 256], mask, pool, gt)


@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
def test_eval_topk_inf_and_nan_scores(implicit):
    """+inf, -inf and NaN scores: every NaN ranks above +inf as in torch.topk, and all NaN scores tie (lowest id
    first) whatever their sign bit and payload; a masked NaN is -1024, a pooled NaN stays NaN.  Item table column
    a(i) in {+-inf, NaN, NaN with the sign bit, NaN with a payload, finite}; user rows 1, 0 (inf * 0 and NaN * 0 are
    NaN, made by the FMA or passed through it), NaN (every score NaN) and 2.  Implicit finite z in {0, >= 17,
    <= -89}, where the sigmoid is exact."""
    rng = np.random.default_rng(11)
    n = 700
    neg_nan = np.array([0xffc00000], dtype=np.uint32).view(np.float32)[0]
    a = rng.choice([0.0, 17.0, 30.0, -89.0, -200.0], n) if implicit else rng.integers(-50, 51, n).astype(np.float64)
    special = rng.choice(n, 40, replace=False)
    a[special[:10]], a[special[10:20]], a[special[20:30]] = np.inf, -np.inf, np.nan
    a = a.astype(np.float32)
    a[special[30:35]] = neg_nan
    a[special[35:]] = np.array([0x7fc01234], dtype=np.uint32).view(np.float32)[0]       # a NaN with a payload
    tab = Tables(np.array([[1.0], [0.0], [np.nan], [2.0]]), a=a, c=np.zeros(n, np.int64))
    mask = csr_of([np.sort(special[::3]), np.arange(0, n, 5), [], np.sort(special[1::4])])
    pool = csr_of([np.sort(special[::2]), np.arange(0, n, 9), np.arange(0, n, 2), np.sort(special[2::3])])
    gt = random_lists(rng, 4, n, 30)
    run_eval_topk(tab, implicit, [0, 1, 2, 3], [1, 25, 60, 256], mask, pool, gt)


LIST_CASES = ["empty_lists", "mask_every_item", "fewer_than_k_unmasked", "lists_over_256", "out_of_range_entries",
              "no_lists", "no_gt", "duplicate_users"]


@gpu
@pytest.mark.parametrize("case", LIST_CASES)
def test_eval_topk_lists(case):
    """Empty lists, a mask over every item or over all but fewer than k, lists longer than the 256 threads that
    fill the bitmaps, ids outside [0, n_items) (ignored; n_gt still counts them), NULL lists, no gt (hits and n_gt
    NULL too), a user several times in one batch."""
    rng = np.random.default_rng(LIST_CASES.index(case))
    n_users, n, k = 5, 4099, 64
    tab = one_hot(rng, n_users, n, 8, False, a_range=30)
    users = np.arange(n_users)
    mask, pool, gt = (random_lists(rng, n_users, n, 40, out_of_range=False) for _ in range(3))
    hits = True
    if case == "empty_lists":
        mask = pool = gt = csr_of([np.zeros(0, np.int64)] * n_users)
    elif case == "mask_every_item":                     # every key -1024 (pooled ones 0): ties by id
        mask = csr_of([np.arange(n)] * n_users)
    elif case == "fewer_than_k_unmasked":
        keep = [rng.choice(n, j, replace=False) for j in (0, 1, 3, 63, 10)]
        mask = csr_of([np.setdiff1d(np.arange(n), kp) for kp in keep])
        pool = csr_of([np.zeros(0, np.int64)] * n_users)
    elif case == "lists_over_256":
        mask, pool, gt = (random_lists(rng, n_users, n, 1000) for _ in range(3))
        assert (np.diff(mask[0]) > 256).any()
    elif case == "out_of_range_entries":
        ends = lambda off, items, u: np.concatenate([[-(2 ** 40), -5, -1], items[off[u]:off[u + 1]],
                                                     [n, n + 1, 2 ** 40]])
        mask, pool, gt = (csr_of([ends(*lst, u) for u in range(n_users)]) for lst in (mask, pool, gt))
    elif case == "no_lists":
        mask = pool = gt = None
    elif case == "no_gt":
        gt, hits = None, False
    elif case == "duplicate_users":
        users = np.array([3, 3, 0, 3, 4, 0])
    run_eval_topk(tab, False, users, [1, k, 256], mask, pool, gt, hits=hits)


@gpu
@pytest.mark.parametrize("b", [1, 3, 300, 2000])
def test_eval_topk_batch_sizes(b):
    rng = np.random.default_rng(b)
    n_users, n = 2500, 500
    tab = one_hot(rng, n_users, n, 8, False, a_range=30)
    mask, pool, gt = (random_lists(rng, n_users, n, 20) for _ in range(3))
    users = rng.integers(0, n_users, b)
    run_eval_topk(tab, False, users, [40], mask, pool, gt)


@gpu
def test_eval_topk_exact_implicit_ties():
    """Implicit scoring with every z in {0, >= 17, <= -89}: keys 0.5, 1, 0 exactly (1024.5, 1025, 1024 pooled), so
    huge tie groups that the k-th score splits, compared bit for bit, on the cache and on the bitmap path."""
    for n in (4099, 60000):
        rng = np.random.default_rng(n)
        a = rng.choice([0.0, 20.0, -100.0], n)
        tab = Tables(np.array([[1.0], [1.0], [5.0]]), a=a, c=np.zeros(n, np.int64))
        mask, pool, gt = (random_lists(rng, 3, n, 200) for _ in range(3))
        assert run_eval_topk(tab, True, [0, 1, 2], [1, 100, 256], mask, pool, gt) == 0


@gpu
def test_eval_topk_rejects_bad_arguments_before_any_launch():
    from invpref_kdd_2022_b200 import _lib
    BAD = -3
    assert _lib.load().invpref_strerror(BAD).decode().startswith("bad argument")
    rng = np.random.default_rng(0)
    Ut, It = one_hot(rng, 3, 300, 8, False).device(_dev())
    gt = random_lists(rng, 3, 300, 10)
    users = [0, 1, 2]
    assert call_eval_topk(Ut, It, False, users, 0)[0] == BAD
    assert call_eval_topk(Ut, It, False, users, 257)[0] == BAD
    Ut2, It2 = one_hot(rng, 3, 100, 8, False).device(_dev())
    assert call_eval_topk(Ut2, It2, False, users, 101)[0] == BAD                  # k > n_items
    assert call_eval_topk(Ut2, It2, False, users, 100, hits=False)[0] == 0       # k = n_items
    assert call_eval_topk(Ut, It, False, users, 10, gt=None, hits=True)[0] == BAD  # hits / n_gt without gt_off
    assert call_eval_topk(Ut, It, False, users, 10, gt=gt, hits=True)[0] == 0
    rc, top, *_ = call_eval_topk(Ut, It, False, [], 10, gt=gt, b=0)
    assert rc == 0 and bool((top == -1).all())                                    # b = 0: nothing written


# ==== GPU: invpref_mask_scores / invpref_hits_from_csr (9 472 rows / 303 104 look-ups per grid sweep) =============
LIST_LENS = (0, 1, 31, 32, 33, 1000)


def _len_lists(rng, n_items):
    """One user per list length of LIST_LENS; the 1000-long list also holds ids outside [0, n_items)."""
    lists = [np.sort(rng.choice(n_items, m, replace=False)) for m in LIST_LENS]
    lists[-1] = np.concatenate([[-3, -1], lists[-1][2:-2], [n_items, n_items + 9]])
    return csr_of(lists)


@gpu
@pytest.mark.parametrize("add", [0, 1])
@pytest.mark.parametrize("b", [1, 9472, 9473, 20000])
def test_mask_scores_matches_numpy(b, add):
    from invpref_kdd_2022_b200 import _lib
    rng = np.random.default_rng(b + add)
    n_items = 1100
    off, items = _len_lists(rng, n_items)
    users = rng.integers(0, len(LIST_LENS), b)
    rating = rng.normal(0, 1, (b, n_items)).astype(np.float32)
    value = np.float32(1024.0 if add else -1024.0)
    dev = _dev()
    rt, ut = torch.from_numpy(rating).to(dev), torch.from_numpy(users).to(dev)
    ot, it = torch.from_numpy(off).to(dev), torch.from_numpy(items).to(dev)
    _lib.check(_lib.load().invpref_mask_scores(_lib.ptr(rt), b, n_items, _lib.ptr(ut), _lib.ptr(ot), _lib.ptr(it),
                                               C.c_float(value), add, _lib.stream_ptr()), "mask_scores")
    want = rating.copy()
    hit = dense_lists((off, items), users, n_items)
    want[hit] = want[hit] + value if add else value
    assert np.array_equal(rt.cpu().numpy().view(np.uint32), want.view(np.uint32))


@gpu
@pytest.mark.parametrize("with_n_list", [False, True], ids=["n_list_null", "n_list"])
@pytest.mark.parametrize("b,k", [(1, 1), (9472, 32), (9473, 33), (20000, 16)])
def test_hits_from_csr_matches_numpy(b, k, with_n_list):
    """Look-ups at the first and the last element of each list, just outside its range, in it and between its
    entries; b * k = 303 104 is one full grid sweep, 9473 * 33 and 20000 * 16 need more."""
    from invpref_kdd_2022_b200 import _lib
    rng = np.random.default_rng(b * k)
    n_items = 1100
    off, items = _len_lists(rng, n_items)
    users = rng.integers(0, len(LIST_LENS), b)
    top = np.empty((b, k), dtype=np.int64)
    for r, u in enumerate(users):
        lst = items[off[u]:off[u + 1]]
        cand = [-1, 0, n_items - 1, n_items, 2 ** 40, int(rng.integers(0, n_items))]
        if lst.size:
            cand += [lst[0], lst[-1], lst[0] - 1, lst[-1] + 1, lst[lst.size // 2], lst[lst.size // 2] + 1]
        top[r] = rng.choice(cand, k)
    dev = _dev()
    tt, ut = torch.from_numpy(top).to(dev), torch.from_numpy(users).to(dev)
    ot, it = torch.from_numpy(off).to(dev), torch.from_numpy(items).to(dev)
    ht = torch.full((b, k), 7, dtype=torch.uint8, device=dev)
    nl = torch.full((b,), -1, dtype=torch.int64, device=dev) if with_n_list else None
    _lib.check(_lib.load().invpref_hits_from_csr(_lib.ptr(tt), b, k, _lib.ptr(ut), _lib.ptr(ot), _lib.ptr(it),
                                                 _lib.ptr(ht), _lib.ptr(nl), _lib.stream_ptr()), "hits_from_csr")
    sets = [set(items[off[u]:off[u + 1]].tolist()) for u in range(len(LIST_LENS))]
    want = np.array([[int(t in sets[u]) for t in row] for u, row in zip(users, top)], dtype=np.uint8)
    got = ht.cpu().numpy()
    assert np.array_equal(got, want)
    assert b < 100 or 0.1 < want.mean() < 0.9
    if with_n_list:
        assert np.array_equal(nl.cpu().numpy(), off[users + 1] - off[users])


# ==== GPU: the metrics of ImplicitTestManager.evaluate ==============================================================
def fp64_metrics(z, masked, pooled, gt_sets, ks):
    """evaluate.py:11-56 restated in fp64: sigmoid scores, masked := -1024, pooled += 1024, top-k by a stable sort,
    recall / precision / NDCG per user, averaged over users."""
    s = 1.0 / (1.0 + np.exp(-z))
    s = np.where(masked, -1024.0, s) + 1024.0 * pooled
    top = np.argsort(-s, axis=1, kind="stable")
    out = {"ndcg": {}, "recall": {}, "precision": {}}
    for k in ks:
        pre = rec = nd = 0.0
        for r, gt in enumerate(gt_sets):
            hit = np.array([1.0 if it in gt else 0.0 for it in top[r, :k]])
            pre += hit.sum() / k
            rec += hit.sum() / len(gt)
            idcg = sum(1.0 / np.log2(j + 2) for j in range(min(k, len(gt))))
            nd += float((hit / np.log2(np.arange(2, k + 2))).sum()) / (idcg if idcg > 0 else 1.0)
        n = len(gt_sets)
        out["ndcg"][k], out["recall"][k], out["precision"][k] = nd / n, rec / n, pre / n
    return out


@gpu
@pytest.mark.parametrize("use_pool", [False, True], ids=["all_items", "item_pool"])
@pytest.mark.parametrize("mode", ["fused", "step_by_step", "host"])
def test_implicit_evaluator_metrics_match_fp64(mode, use_pool):
    """Tie-free implicit inputs: identity item table (D = n_items = 200), every user's z a permutation of the 1/32
    grid of [-3.125, 3.09] (neighbouring sigmoids >= 1e-3 apart, also after + 1024), top-k above the masked items.
    ImplicitTestManager.evaluate() must then give the fp64 metrics up to summation order."""
    from invpref_kdd_2022_b200.dataloader import YahooImplicitBCELossDataLoader
    from invpref_kdd_2022_b200.evaluate import ImplicitTestManager
    from invpref_kdd_2022_b200.models import InvPrefImplicit
    dev = _dev()
    rng = np.random.default_rng(5)
    n_users, n = 150, 200
    tr = [(u, i, int(rng.random() < 0.8)) for u in range(n_users) for i in rng.choice(n, 12, replace=False)]
    tr.append((n_users - 1, n - 1, 0))
    te = [(u, i, 1) for u in range(0, n_users, 1) if u % 7 for i in rng.choice(n, int(rng.integers(1, 9)), replace=False)]
    loader = YahooImplicitBCELossDataLoader("", dev, train=np.array(tr, np.int64), test=np.array(te, np.int64))
    assert (loader.user_num, loader.item_num) == (n_users, n)
    if use_pool:
        pool = [(u, i) for u in range(n_users) for i in rng.choice(n, 6, replace=False)]
        loader.set_item_pool(np.array(pool, np.int64))
    model = InvPrefImplicit(n_users, n, 2, n).to(dev)
    Z = np.stack([rng.permutation(n) for _ in range(n_users)]).astype(np.float64) / 32.0 - 3.125
    with torch.no_grad():
        model.embed_user_invariant.weight.copy_(torch.from_numpy(Z).float())
        model.embed_item_invariant.weight.copy_(torch.eye(n))
    ks = [1, 5, 20, 50]
    ev = ImplicitTestManager(model, loader, test_batch_size=64, top_k_list=ks, use_item_pool=use_pool,
                             fused=(mode == "fused"))
    if mode == "host":
        ev.evaluate_batch = functools.partial(ev.evaluate_batch, force_host=True)
    fused_calls = []
    hits_fused = ev._hits_fused
    ev._hits_fused = lambda *args: fused_calls.append(args) or hits_fused(*args)
    got = ev.evaluate()
    assert bool(fused_calls) == (mode == "fused")               # the path under test is the one that ran
    users = np.asarray(loader.all_test_users_by_sorted_list)
    masked = dense_lists((loader.mask_off, loader.mask_items), users, n)
    pooled = dense_lists((loader.pool_off, loader.pool_items) if use_pool else None, users, n)
    assert (n - masked.sum(1)).min() > max(ks)                 # the top k never reaches the tied masked items
    want = fp64_metrics(Z[users], masked, pooled, loader.get_sorted_all_test_users_ground_truth, ks)
    for m in want:
        for k in ks:
            assert abs(got[m][k] - want[m][k]) <= 1e-12, (m, k, got[m][k], want[m][k])

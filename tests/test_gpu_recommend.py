"""``invpref_recommend`` / ``model.recommend`` and the evaluator at large catalogues: the streaming top-k kernel of
eval.cu against the exact references of test_gpu_eval_topk.py.

The kernel works on tiles of 32 users and 128 items; with few users it splits the item range over a cluster of up to
8 CTAs (8 slices whenever one tile of users meets at least 8 * 128 items).  Explicit tables hold integers and
implicit z lies in {0, >= 17, <= -89}, so every key is known exactly and results are compared bit for bit.
"""
import numpy as np
import pytest
import torch

from test_gpu_eval_topk import (Tables, csr_of, dense_lists, exact_sigmoid, fp64_metrics, one_hot,
                                random_lists, ref_order, run_eval_topk)

gpu = pytest.mark.gpu
TU, TI, SLICES = 32, 128, 8


def slice_edges(n_items):
    """Item ids where a cluster slice starts, for a batch of at most TU users and n_items >= SLICES * TI."""
    per = -(-n_items // SLICES)
    return [j * per for j in range(1, SLICES)]


# ---- reference ----------------------------------------------------------------------------------------------------
def ref_recommend(keys, excluded, k):
    """(items int64 [b, k], scores fp32 [b, k]): the evaluator's order over the items that are not excluded, item -1
    and score -inf where fewer than k remain."""
    keys = np.asarray(keys, dtype=np.float32)
    b, n = keys.shape
    order = ref_order(keys)
    items = np.full((b, k), -1, dtype=np.int64)
    scores = np.full((b, k), -np.inf, dtype=np.float32)
    for r in range(b):
        o = order[r][~excluded[r, order[r]]][:k]
        items[r, :o.size] = o
        scores[r, :o.size] = keys[r, o]
    return items, scores


def brute_recommend(row, excluded, k):
    """The same for one row by pairwise comparison (checks ref_recommend)."""
    def above(x, y):
        kx, ky = row[x], row[y]
        if np.isnan(kx) or np.isnan(ky):
            return np.isnan(kx) and (not np.isnan(ky) or x < y)
        return kx > ky or (kx == ky and x < y)
    keep = [i for i in range(len(row)) if not excluded[i]]
    best = []
    for i in keep:
        pos = sum(1 for j in keep if j != i and above(j, i))
        if pos < k:
            best.append((pos, i))
    out = [i for _, i in sorted(best)] + [-1] * (k - len(best))
    return np.array(out[:k], dtype=np.int64)


# ---- calling the library ------------------------------------------------------------------------------------------
def _hot(Ut, It, implicit):
    from invpref_kdd_2022_b200.engine import HotPath
    dev = Ut.device
    E = torch.zeros((1, Ut.shape[1]), dtype=torch.float32, device=dev)
    return HotPath({"Uinv": Ut, "Iinv": It, "Uenv": Ut, "Ienv": It, "E": E, "W": E,
                    "b": torch.zeros(1, dtype=torch.float32, device=dev)}, implicit, False, False)


def run_recommend(tab, implicit, users, ks, excl=None):
    """recommend for every k of `ks` against ref_recommend, bit for bit (explicit, or implicit with exact z)."""
    dev = torch.device("cuda:0")
    users = np.asarray(users, dtype=np.int64)
    Ut, It = tab.device(dev)
    hp = _hot(Ut, It, implicit)
    z = tab.z(users)
    keys = exact_sigmoid(z) if implicit else z.astype(np.float32)
    excluded = dense_lists(excl, users, tab.n_items)
    ex = None if excl is None else tuple(torch.from_numpy(np.ascontiguousarray(x)).to(dev) for x in excl)
    ut = torch.from_numpy(users).to(dev)
    for k in ks:
        top, sc = hp.recommend(ut, k, ex)
        top, sc = top.cpu().numpy(), sc.cpu().numpy()
        want, ws = ref_recommend(keys, excluded, k)
        bad = np.argwhere(top != want)
        assert bad.size == 0, (k, bad[:5].tolist(), top[tuple(bad[0])], want[tuple(bad[0])])
        assert np.array_equal(np.isnan(sc), np.isnan(ws)), k
        fin = ~np.isnan(ws)
        assert np.array_equal(sc[fin].view(np.uint32), ws[fin].view(np.uint32)), k


# ==== CPU ===========================================================================================================
def test_recommend_reference_matches_pairwise_ranking():
    rng = np.random.default_rng(0)
    for trial in range(200):
        n = int(rng.integers(1, 30))
        row = rng.integers(-3, 4, n).astype(np.float32)
        if trial % 3 == 0:
            row[rng.random(n) < 0.15] = np.nan
            row[rng.random(n) < 0.1] = -np.inf
        excluded = rng.random(n) < (0.9 if trial % 7 == 0 else 0.3)
        k = int(rng.integers(1, n + 3))
        items, scores = ref_recommend(row[None, :], excluded[None, :], k)
        assert np.array_equal(items[0], brute_recommend(row, excluded, k)), (row, excluded, k)
        assert np.isneginf(scores[0][items[0] < 0]).all()


def test_user_item_csr_matches_the_loaders_lists():
    from invpref_kdd_2022_b200.dataloader import YahooImplicitBCELossDataLoader, user_item_csr
    rng = np.random.default_rng(1)
    n_users, n_items = 40, 90
    tr = np.stack([rng.integers(0, n_users, 800), rng.integers(0, n_items, 800), rng.integers(0, 2, 800)], 1)
    te = np.stack([rng.integers(0, n_users, 200), rng.integers(0, n_items, 200), np.ones(200, np.int64)], 1)
    tr[0, :] = (n_users - 1, n_items - 1, 1)
    loader = YahooImplicitBCELossDataLoader("", torch.device("cpu"), train=tr, test=te)
    pos = tr[tr[:, 2] > 0]
    for (off, items), (u, i) in (((loader.mask_off, loader.mask_items), (pos[:, 0], pos[:, 1])),
                                 ((loader.gt_off, loader.gt_items), (te[:, 0], te[:, 1]))):
        o2, i2 = user_item_csr(u, i, loader.user_num)
        assert np.array_equal(off, o2) and np.array_equal(items, i2)
        for user in range(loader.user_num):
            assert items[off[user]:off[user + 1]].tolist() == sorted(set(i[u == user].tolist()))
    off, items = user_item_csr(np.zeros(0, np.int64), np.zeros(0, np.int64), 3)
    assert off.tolist() == [0, 0, 0, 0] and items.size == 0


# ==== GPU: recommend ================================================================================================
def _size_cases():
    big = (1 << 20) + 3
    return [1, TI - 1, TI, TI + 1, SLICES * TI - 1, SLICES * TI, SLICES * TI + 1, 4099, big]


@gpu
@pytest.mark.parametrize("n_items", _size_cases())
def test_recommend_item_counts(n_items):
    """One item, partial / full / one-past item tiles, the smallest catalogue split over 8 slices and one item
    either side of it, and 2^20 + 3 items; one-hot tables with many equal scores, exclusion lists with entries
    outside [0, n_items), a duplicate user."""
    rng = np.random.default_rng(n_items)
    n_users = 6
    tab = one_hot(rng, n_users, n_items, 40, False)
    excl = random_lists(rng, n_users, n_items, min(300, max(1, n_items // 4)))
    ks = sorted({1, min(n_items, 37), min(n_items, 256)})
    run_recommend(tab, False, [0, 1, 4, 1, 5], ks, excl)


@gpu
@pytest.mark.parametrize("D", [1, 3, 17, 40, 64, 128, 256])
def test_recommend_dims(D):
    """Dense integer tables (|z| <= 32 * 32 * 256 < 2^24): float4 and scalar dims, one and several staged chunks."""
    rng = np.random.default_rng(D)
    n_users, n = 5, 3001
    tab = Tables(rng.integers(-32, 33, (n_users, D)), I=rng.integers(-32, 33, (n, D)))
    run_recommend(tab, False, np.arange(n_users), [1, 33, 256], random_lists(rng, n_users, n, 40))


@gpu
@pytest.mark.parametrize("k", [1, 2, 31, 32, 33, 255, 256])
def test_recommend_k(k):
    rng = np.random.default_rng(100 + k)
    n_users, n = 7, 20000
    tab = one_hot(rng, n_users, n, 8, False, a_range=20)
    run_recommend(tab, False, np.arange(n_users), [k], random_lists(rng, n_users, n, 50))


@gpu
@pytest.mark.parametrize("b", [1, TU - 1, TU, TU + 1, 65537])
def test_recommend_batch_sizes(b):
    """Partial, full and one-past user tiles, and 65 537 users (one slice per tile), duplicate users included."""
    rng = np.random.default_rng(b)
    n_users, n = 3000, 300 if b > 1000 else 5000
    tab = one_hot(rng, n_users, n, 8, False, a_range=30)
    users = rng.integers(0, n_users, b)
    if b > 1:
        users[-1] = users[0]
    run_recommend(tab, False, users, [40], random_lists(rng, n_users, n, 20))


@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
def test_recommend_nan_inf_and_signed_zero_scores(implicit):
    """NaN (any sign / payload) above +inf, -inf below every finite score, products that are -0.0 (summed from +0)."""
    rng = np.random.default_rng(11)
    n = 3000
    neg_nan = np.array([0xffc00000], dtype=np.uint32).view(np.float32)[0]
    a = rng.choice([0.0, 17.0, 30.0, -89.0, -200.0], n) if implicit else rng.integers(-50, 51, n).astype(np.float64)
    special = rng.choice(n, 60, replace=False)
    a[special[:15]], a[special[15:30]], a[special[30:40]] = np.inf, -np.inf, np.nan
    a = a.astype(np.float32)
    a[special[40:50]] = neg_nan
    a[special[50:]] = -0.0
    tab = Tables(np.array([[1.0], [0.0], [np.nan], [2.0 if implicit else -2.0]]), a=a, c=np.zeros(n, np.int64))
    excl = csr_of([np.sort(special[::3]), [], np.arange(0, n, 2), np.sort(special[1::4])])
    run_recommend(tab, implicit, [0, 1, 2, 3], [1, 25, 60, 256], excl)


def _stream(name, n):
    a = np.arange(n, dtype=np.float64)
    if name == "ascending":                  # every tile holds better scores than all before: a reduction per tile
        return a, None
    if name == "descending":
        return -a, None
    if name == "all_equal":                  # must return ids 0 .. k-1
        return np.full(n, 3.0), None
    a = np.random.default_rng(5).integers(-1000, 0, n).astype(np.float64)
    edge = TI * 37 if name == "tie_across_tile_edge" else slice_edges(n)[3]
    grp = np.arange(edge - 10, edge + 70)
    a[grp] = 50
    a[np.arange(10, 10 + 100 * 7, 7)] = 100 + np.arange(100)          # 100 items above the group
    return a, grp


@gpu
@pytest.mark.parametrize("name", ["ascending", "descending", "all_equal", "tie_across_tile_edge",
                                  "tie_across_slice_edge"])
def test_recommend_threshold_streams(name):
    """Streams that move the running threshold: ascending (every tile reduces), descending, 2^20 equal scores, a
    tie group at the k-th score straddling an item-tile edge and a cluster-slice edge (k = 130 keeps 30 of 80)."""
    n = (1 << 20) if name == "all_equal" else 200003
    a, grp = _stream(name, n)
    tab = Tables(np.array([[1.0], [2.0]]), a=a, c=np.zeros(n, np.int64))
    ks = [130] if grp is not None else [1, 50, 256]
    run_recommend(tab, False, [0, 1], ks)
    if name == "all_equal":
        hp = _hot(*tab.device(torch.device("cuda:0")), False)
        top, _ = hp.recommend(torch.zeros(1, dtype=torch.int64, device="cuda:0"), 256)
        assert top.cpu().numpy()[0].tolist() == list(range(256))


EXCL_CASES = ["empty_lists", "every_item", "fewer_than_k", "out_of_range", "long_lists_across_edges", "no_lists"]


@gpu
@pytest.mark.parametrize("case", EXCL_CASES)
def test_recommend_exclusion(case):
    rng = np.random.default_rng(EXCL_CASES.index(case))
    n_users, n, k = 5, 20011, 64
    tab = one_hot(rng, n_users, n, 8, False, a_range=30)
    excl = random_lists(rng, n_users, n, 40, out_of_range=False)
    if case == "empty_lists":
        excl = csr_of([np.zeros(0, np.int64)] * n_users)
    elif case == "every_item":                       # all -1 and -inf
        excl = csr_of([np.arange(n)] * n_users)
    elif case == "fewer_than_k":
        keep = [rng.choice(n, j, replace=False) for j in (0, 1, 3, 63, 10)]
        excl = csr_of([np.setdiff1d(np.arange(n), kp) for kp in keep])
    elif case == "out_of_range":
        excl = csr_of([np.concatenate([[-(2 ** 40), -5, -1], excl[1][excl[0][u]:excl[0][u + 1]], [n, n + 1, 2 ** 40]])
                       for u in range(n_users)])
    elif case == "long_lists_across_edges":         # runs over item-tile and slice edges, longer than a tile
        edges = [TI * 9] + slice_edges(n)
        excl = csr_of([np.unique(np.concatenate([np.arange(e - 300, e + 300) for e in edges[u % 3::2]]))
                       for u in range(n_users)])
    elif case == "no_lists":
        excl = None
    run_recommend(tab, False, np.arange(n_users), [1, k, 256], excl)


# ==== GPU: the evaluator on the same kernel at a large catalogue =====================================================
@gpu
@pytest.mark.parametrize("implicit", [False, True], ids=["explicit", "implicit"])
def test_eval_topk_at_2_pow_20_items(implicit):
    n = (1 << 20) + 3
    rng = np.random.default_rng(20 + implicit)
    if implicit:
        tab = Tables(np.array([[1.0], [1.0], [5.0]]), a=rng.choice([0.0, 20.0, -100.0], n), c=np.zeros(n, np.int64))
    else:
        tab = one_hot(rng, 3, n, 40, False)
    mask, pool, gt = (random_lists(rng, 3, n, 500) for _ in range(3))
    assert run_eval_topk(tab, implicit, [0, 1, 2], [1, 100, 256], mask, pool, gt) == 0


@gpu
@pytest.mark.parametrize("n", [2047, 2048, 2049])
def test_eval_topk_either_side_of_the_kernel_choice(n):
    """The evaluator runs one CTA per user below 2048 items and the streaming kernel from 2048 on: same results."""
    rng = np.random.default_rng(n)
    tab = one_hot(rng, 40, n, 40, False)
    mask, pool, gt = (random_lists(rng, 40, n, 60) for _ in range(3))
    users = rng.integers(0, 40, 37)
    assert run_eval_topk(tab, False, users, [1, 30, 256], mask, pool, gt) == 0


@gpu
def test_implicit_evaluator_metrics_at_60000_items():
    """ImplicitTestManager.evaluate() on the fused path against fp64_metrics: identity-like item table (one-hot
    rows e_c(i)) and per-user z on a 1/64 grid of distinct values, so no ties in the top k."""
    from invpref_kdd_2022_b200.dataloader import YahooImplicitBCELossDataLoader
    from invpref_kdd_2022_b200.evaluate import ImplicitTestManager
    from invpref_kdd_2022_b200.models import InvPrefImplicit
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(6)
    n_users, n, D = 70, 60000, 64
    tr = [(u, i, 1) for u in range(n_users) for i in rng.choice(n, 30, replace=False)]
    tr.append((n_users - 1, n - 1, 0))
    te = [(u, i, 1) for u in range(n_users) if u % 5 for i in rng.choice(n, int(rng.integers(1, 9)), replace=False)]
    loader = YahooImplicitBCELossDataLoader("", dev, train=np.array(tr, np.int64), test=np.array(te, np.int64))
    model = InvPrefImplicit(n_users, n, 2, D).to(dev)
    c = rng.integers(0, D, n)
    a = (rng.permutation(n) / 16384.0 - 1.8).astype(np.float32).astype(np.float64)   # distinct; U = +-1: exact z
    U = rng.choice([-1.0, 1.0], (n_users, D))
    with torch.no_grad():
        model.embed_user_invariant.weight.copy_(torch.from_numpy(U).float())
        It = torch.zeros((n, D))
        It[torch.arange(n), torch.from_numpy(c)] = torch.from_numpy(a).float()
        model.embed_item_invariant.weight.copy_(It)
    ks = [1, 5, 20, 50]
    got = ImplicitTestManager(model, loader, test_batch_size=32, top_k_list=ks).evaluate()
    users = np.asarray(loader.all_test_users_by_sorted_list)
    Z = a[None, :] * U[users][:, c]
    masked = dense_lists((loader.mask_off, loader.mask_items), users, n)
    want = fp64_metrics(Z, masked, np.zeros_like(masked), loader.get_sorted_all_test_users_ground_truth, ks)
    for m in want:
        for k in ks:
            assert abs(got[m][k] - want[m][k]) <= 1e-12, (m, k, got[m][k], want[m][k])


# ==== GPU: model API ================================================================================================
def _model(cls, dev, n_users=50, n_items=3000, D=16, seed=0):
    """Integer tables: exact z in any summation order; implicit |z| <= 16, where fp32 sigmoids of distinct
    integers stay distinct and ordered."""
    torch.manual_seed(seed)
    m = cls(n_users, n_items, 3, D).to(dev)
    rng = np.random.default_rng(seed)
    v = 1 if cls.implicit else 20
    with torch.no_grad():
        m.embed_user_invariant.weight.copy_(torch.from_numpy(rng.integers(-v, v + 1, (n_users, D))).float())
        m.embed_item_invariant.weight.copy_(torch.from_numpy(rng.integers(-v, v + 1, (n_items, D))).float())
    return m


@gpu
@pytest.mark.parametrize("which", ["explicit", "implicit"])
def test_model_recommend_matches_the_reference(which):
    from invpref_kdd_2022_b200.dataloader import user_item_csr
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    dev = torch.device("cuda:0")
    cls = InvPrefImplicit if which == "implicit" else InvPrefExplicit
    m = _model(cls, dev)
    rng = np.random.default_rng(3)
    pairs = np.stack([rng.integers(0, 50, 4000), rng.integers(0, 3000, 4000)], 1)
    off, items = user_item_csr(pairs[:, 0], pairs[:, 1], 50)
    users = np.array([3, 0, 49, 3, 17])
    for excl in (None, (off, items), (torch.from_numpy(off).to(dev), torch.from_numpy(items).to(dev))):
        top, sc = m.recommend(torch.from_numpy(users).to(dev), 20, exclude=excl)
        assert top.dtype == torch.int64 and sc.dtype == torch.float32 and top.shape == (5, 20)
        U = m.embed_user_invariant.weight.detach().cpu().numpy().astype(np.float64)
        I = m.embed_item_invariant.weight.detach().cpu().numpy().astype(np.float64)
        z = U[users] @ I.T
        ex = dense_lists(None if excl is None else (off, items), users, 3000)
        order = ref_order(z + 0.0)
        for r in range(len(users)):
            o = order[r][~ex[r, order[r]]][:20]
            assert top[r].cpu().numpy().tolist() == o.tolist()
        if which == "explicit":
            assert np.array_equal(sc.cpu().numpy(), np.take_along_axis(z, top.cpu().numpy(), 1).astype(np.float32))


@gpu
def test_model_recommend_after_lazy_steps_equals_flushed_tables():
    """After lazy-Adam train steps without a flush, recommend sees the caught-up user rows: it equals recommend on a
    copy of the flushed tables."""
    from invpref_kdd_2022_b200.models import InvPrefExplicit
    dev = torch.device("cuda:0")
    m = InvPrefExplicit(300, 2000, 2, 64).to(dev)
    hp = m.hot_path(lr=1e-2, lazy=True)
    assert hp.lazy
    rng = np.random.default_rng(4)
    for _ in range(4):
        B = 512
        t = lambda x: torch.from_numpy(x).to(dev)
        hp.train_step(t(rng.integers(0, 30, B)), t(rng.integers(0, 2000, B)), t(rng.random(B).astype(np.float32)),
                      t(rng.integers(0, 2, B)), t(np.ones(B, np.float32)), c_inv=1.0, c_ea=1.0, c_env=1.0, c_L2=0.0,
                      c_L1=0.0, alpha=1.0, use_class_rw=False, use_rec_rw=False)
    assert hp._dirty
    users = torch.arange(40, 300, 7, device=dev)                     # rows the batches did not touch
    top, sc = m.recommend(users, 30)
    assert not hp._dirty
    ref = _hot(hp.params["Uinv"].clone(), hp.params["Iinv"].clone(), False)
    top2, sc2 = ref.recommend(users, 30)
    assert torch.equal(top, top2) and torch.equal(sc.view(torch.int32), sc2.view(torch.int32))


@gpu
def test_model_recommend_rejects_bad_input():
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    dev = torch.device("cuda:0")
    m = _model(InvPrefImplicit, dev, n_items=100)
    with pytest.raises(IndexError):
        m.recommend(torch.tensor([0, 50], device=dev), 5)
    with pytest.raises(IndexError):
        m.recommend(torch.tensor([-1], device=dev), 5)
    for k in (0, 257, 101):                          # k = 101 > n_items
        with pytest.raises(RuntimeError, match="bad argument"):
            m.recommend(torch.tensor([0], device=dev), k)
    top, sc = m.recommend(torch.tensor([0], device=dev), 100)
    assert sorted(top[0].cpu().tolist()) == list(range(100))
    top, sc = m.recommend(torch.zeros(0, dtype=torch.int64, device=dev), 5)
    assert top.shape == (0, 5) and sc.shape == (0, 5)
    with pytest.raises(RuntimeError, match="exclude"):      # offsets shorter than n_users + 1
        m.recommend(torch.tensor([0], device=dev), 5, exclude=(np.zeros(10, np.int64), np.zeros(1, np.int64)))
    with pytest.raises(RuntimeError, match="exclude"):
        m.recommend(torch.tensor([0], device=dev), 5, exclude=(np.zeros(51, np.int32), np.zeros(1, np.int64)))
    cpu = InvPrefExplicit(10, 20, 2, 8)
    with pytest.raises(RuntimeError):
        cpu.recommend(torch.tensor([0]), 3)

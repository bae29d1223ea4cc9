"""CPU, needs a checkout of the original project at oracle/_ref (skips without it): the callers either side of the
hot path -- data loaders (SURVEY.md §8f rank 3) and evaluators (ranks 1 and 4) -- against the LIVE reference on the
datasets that ship with it.  Loaders: same table sizes, same arrays, same per-user mask / ground-truth / pool
sets.  Evaluators: same metric dictionaries when both sides score with the same stub model (the ranking logic,
masking, item-pool highlighting, NDCG / recall / precision and the MSE / RMSE / MAE formulas are what is compared;
the scores themselves are the hot path's business and are covered by the GPU suite)."""
import os

import numpy as np
import pytest
import torch

from oracle import ref_shim

DATA = os.path.join(ref_shim.REF_ROOT, "dataset")
pytestmark = pytest.mark.skipif(not (ref_shim.available() and os.path.isdir(DATA)),
                                reason="no checkout of the original project at oracle/_ref")


@pytest.fixture(scope="module")
def ref():
    with ref_shim.quiet():
        return ref_shim.load()


@pytest.mark.parametrize("name", ["Coat_explicit_all_data", "Yahoo_explicit_all_data"])
def test_explicit_loader_matches_reference(ref, name):
    from invpref_kdd_2022_b200.dataloader import ExplicitDataLoader
    cpu = torch.device("cpu")
    ours = ExplicitDataLoader(os.path.join(DATA, name), cpu, cache=False)
    theirs = ref.dataloader.ExplicitDataLoader(os.path.join(DATA, name), cpu)
    assert (ours.user_num, ours.item_num) == (theirs.user_num, theirs.item_num)
    assert (ours.train_data_len, ours.test_data_len) == (theirs.train_data_len, theirs.test_data_len)
    assert np.array_equal(ours.train_data_np, theirs.train_data_np)
    assert np.array_equal(ours.test_data_np, theirs.test_data_np)
    assert torch.equal(ours.all_test_pairs_tensor, theirs.all_test_pairs_tensor)
    assert torch.equal(ours.all_test_scores_tensor, theirs.all_test_scores_tensor)


@pytest.mark.parametrize("name,pool", [("Coat_all_data", True), ("Yahoo_all_data", True)])
def test_implicit_loader_matches_reference(ref, name, pool):
    from invpref_kdd_2022_b200.dataloader import YahooImplicitBCELossDataLoader
    cpu = torch.device("cpu")
    ours = YahooImplicitBCELossDataLoader(os.path.join(DATA, name), cpu, has_item_pool_file=pool, cache=False)
    theirs = ref.dataloader.YahooImplicitBCELossDataLoader(os.path.join(DATA, name), cpu, has_item_pool_file=pool)
    assert (ours.user_num, ours.item_num) == (theirs.user_num, theirs.item_num)
    assert np.array_equal(ours.train_data_np, theirs.train_data_np)
    assert ours.all_test_users_by_sorted_list == theirs.all_test_users_by_sorted_list
    assert torch.equal(ours.all_test_users_by_sorted_tensor, theirs.all_test_users_by_sorted_tensor)
    users = ours.all_test_users_by_sorted_list
    step = max(1, len(users) // 400)                       # every user on Coat, ~400 spread over Yahoo
    for u in users[::step]:
        assert ours.user_mask_items(u) == set(theirs.user_mask_items(u)), u
        assert ours.get_user_ground_truth(u) == set(theirs.get_user_ground_truth(u)), u
        if pool:
            assert ours.user_highlight_items(u) == set(theirs.user_highlight_items(u)), u
    gt_o, gt_t = ours.get_sorted_all_test_users_ground_truth, theirs.get_sorted_all_test_users_ground_truth
    assert len(gt_o) == len(gt_t) and all(a == set(b) for a, b in zip(gt_o[::step], gt_t[::step]))


class _StubImplicit(torch.nn.Module):
    """Scores every (user, item) pair with a fixed pseudo-random table: both evaluators see the same ratings."""

    def __init__(self, n_users, n_items, seed=3):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.table = torch.rand((n_users, n_items), generator=g)

    def predict(self, users_id):
        return self.table[users_id].clone()


class _StubExplicit(torch.nn.Module):
    def __init__(self, n_users, n_items, seed=4):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.table = 1.0 + 4.0 * torch.rand((n_users, n_items), generator=g)

    def predict(self, users_id, items_id):
        return self.table[users_id, items_id]


@pytest.mark.parametrize("use_pool", [False, True])
def test_implicit_evaluator_matches_reference(ref, use_pool):
    from invpref_kdd_2022_b200.dataloader import YahooImplicitBCELossDataLoader
    from invpref_kdd_2022_b200.evaluate import ImplicitTestManager
    cpu = torch.device("cpu")
    path = os.path.join(DATA, "Coat_all_data")
    ours_dl = YahooImplicitBCELossDataLoader(path, cpu, has_item_pool_file=True, cache=False)
    ref_dl = ref.dataloader.YahooImplicitBCELossDataLoader(path, cpu, has_item_pool_file=True)
    model = _StubImplicit(ours_dl.user_num, ours_dl.item_num)
    ks = [3, 5, 7]
    got = ImplicitTestManager(model, ours_dl, test_batch_size=97, top_k_list=list(ks), use_item_pool=use_pool).evaluate()
    with ref_shim.quiet():
        want = ref.evaluate.ImplicitTestManager(model, ref_dl, test_batch_size=97, top_k_list=list(ks),
                                                use_item_pool=use_pool).evaluate()
    assert set(got) == set(want) == {"ndcg", "recall", "precision"}
    for metric in want:
        assert list(got[metric]) == list(want[metric]) == ks
        for k in ks:
            assert abs(got[metric][k] - want[metric][k]) <= 1e-12, (metric, k, got[metric][k], want[metric][k])


def test_explicit_evaluator_matches_reference(ref):
    from invpref_kdd_2022_b200.dataloader import ExplicitDataLoader
    from invpref_kdd_2022_b200.evaluate import ExplicitTestManager
    cpu = torch.device("cpu")
    path = os.path.join(DATA, "Coat_explicit_all_data")
    ours_dl = ExplicitDataLoader(path, cpu, cache=False)
    ref_dl = ref.dataloader.ExplicitDataLoader(path, cpu)
    model = _StubExplicit(ours_dl.user_num, ours_dl.item_num)
    got = ExplicitTestManager(model, ours_dl).evaluate()
    with ref_shim.quiet():
        want = ref.evaluate.ExplicitTestManager(model, ref_dl).evaluate()
    assert set(got) == set(want) == {"mse", "rmse", "mae"}
    for k in want:
        assert abs(got[k] - want[k]) <= 1e-6 * abs(want[k]), (k, got[k], want[k])


@pytest.mark.parametrize("name", ["Yahoo_InvPref_Implicit", "MIND_InvPref", "MovieLens_InvPref"])
def test_driver_item_pool_flags_match_reference(name):
    """Which implicit drivers rank only the test item pool (reference <driver>.py: ImplicitTestManager(...,
    use_item_pool=...) and YahooImplicitBCELossDataLoader(..., has_item_pool_file=...))."""
    import importlib
    import re
    src = open(os.path.join(ref_shim.REF_ROOT, name + ".py")).read()
    use = re.search(r"use_item_pool=(True|False)", src).group(1) == "True"
    has = re.search(r"has_item_pool_file=(True|False)", src).group(1) == "True"
    drv = importlib.import_module("invpref_kdd_2022_b200.drivers." + name)
    assert (drv.USE_ITEM_POOL, drv.HAS_ITEM_POOL_FILE) == (use, has)
    for key in ("MODEL_CONFIG", "TRAIN_CONFIG", "EVALUATE_CONFIG"):
        blk = re.search(key + r"[^=]*=\s*(\{.*?\n\})", src, flags=re.S).group(1)
        assert getattr(drv, key) == eval(blk), key

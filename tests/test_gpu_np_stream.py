"""GPU: numpy's global stream drawn on the device (npstream.device_randint, invpref_mt_randint) is np.random.randint bit
for bit and leaves numpy's state where the host call would; the trainers' tie_break_rng="numpy_device" mode then
reproduces the "numpy" mode exactly."""
import numpy as np
import pytest
import torch

from _golden import CASES, Golden

pytestmark = pytest.mark.gpu

HIGHS = [1, 2, 6, 24, 120, 720, 5040, 40320, 2 ** 31 + 1, 2 ** 32]
POSES = [0, 1, 226, 227, 396, 623, 624]
NS = [0, 1, 623, 624, 625, 9000, 200_000]
DEV = torch.device("cuda:0")


def set_state(seed, pos):
    r = np.random.RandomState(seed)
    key = r.randint(0, 2 ** 32, 624, dtype=np.uint64).astype(np.uint32)
    np.random.set_state(("MT19937", key, pos, 0, 0.0))


def same_state(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3] and a[4] == b[4]


def check_draw(high, n, seed, pos):
    from invpref_kdd_2022_b200.npstream import device_randint
    set_state(seed, pos)
    want = np.random.randint(0, high, n)
    want_state = np.random.get_state()
    set_state(seed, pos)
    got = device_randint(high, n, DEV)
    assert got.dtype == torch.int64 and got.device == DEV and got.shape == (n,)
    assert np.array_equal(got.cpu().numpy(), want), (high, n, pos)
    assert same_state(np.random.get_state(), want_state), (high, n, pos)


@pytest.mark.parametrize("high", HIGHS)
def test_bit_equal_to_numpy_on_the_grid(high):
    for pos in POSES:
        for j, n in enumerate(NS):
            check_draw(high, n, 7 * pos + j + high % 1009, pos)


@pytest.mark.parametrize("high,n", [(720, 4_194_304), (24, 96_500_000), (6, 3_000_000), (40320, 1_000_000)])
def test_bit_equal_at_dataset_sizes(high, n):
    """MIND's tie-break draw (4 M from 6!), a C5-sized draw (96.5 M from 4!), and two more shapes."""
    for pos in (624, 17):
        check_draw(high, n, n % 1013 + pos, pos)


def test_consecutive_calls_and_gauss_cache():
    from invpref_kdd_2022_b200.npstream import device_randint
    calls = [(24, 70_000), (720, 3000), (2, 1), (6, 500_000), (1, 9), (40320, 1300), (2 ** 32, 2000)]
    for interleave in (False, True):
        np.random.seed(5)
        np.random.standard_normal()                             # has_gauss = 1 with a cached value
        got = []
        for high, n in calls:
            got.append(device_randint(high, n, DEV).cpu().numpy())
            if interleave:
                np.random.standard_normal()
        got_state = np.random.get_state()
        np.random.seed(5)
        np.random.standard_normal()
        for (high, n), g in zip(calls, got):
            assert np.array_equal(g, np.random.randint(0, high, n))
            if interleave:
                np.random.standard_normal()
        assert same_state(got_state, np.random.get_state())
        assert got_state[3] == (0 if interleave else 1)      # the device draws kept numpy's cached gaussian


def test_out_argument_and_bad_arguments():
    from invpref_kdd_2022_b200.npstream import device_randint, jump_table_bytes
    out = torch.full((1000,), -1, dtype=torch.int64, device=DEV)
    np.random.seed(3)
    r = device_randint(720, 1000, DEV, out=out)
    assert r is out
    np.random.seed(3)
    assert np.array_equal(out.cpu().numpy(), np.random.randint(0, 720, 1000))
    before = np.random.get_state()
    for bad in (0, -1, 2 ** 32 + 1):
        with pytest.raises(ValueError):
            device_randint(bad, 10, DEV)
    with pytest.raises(ValueError):
        device_randint(6, -1, DEV)
    assert same_state(before, np.random.get_state())
    assert jump_table_bytes(DEV) > 13 * 49_000_000


# ---------------------------------------------------------------------------------------------- trainers
def build(g, mode, epochs=1):
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    from invpref_kdd_2022_b200.train import ExplicitTrainManager, ImplicitTrainManager

    class NullEvaluator:
        def evaluate(self):
            return {"mse": 0.0}

    torch.manual_seed(g.seed)
    np.random.seed(g.seed)
    M = InvPrefImplicit if g.implicit else InvPrefExplicit
    T = ImplicitTrainManager if g.implicit else ExplicitTrainManager
    model = M(g.U, g.I, g.K, g.D, g.roe, g.ree).to(DEV)
    tm = T(model=model, evaluator=NullEvaluator(), device=DEV, training_data=torch.LongTensor(g.data).to(DEV),
           batch_size=g.B, epochs=epochs, cluster_interval=1, evaluate_interval=1, lr=g.lr,
           invariant_coe=g.coef["c_inv"], env_aware_coe=g.coef["c_ea"], env_coe=g.coef["c_env"],
           L2_coe=g.coef["c_L2"], L1_coe=g.coef["c_L1"], alpha=g.alpha, use_class_re_weight=g.crw,
           use_recommend_re_weight=g.rrw, tie_break_rng=mode)
    return model, tm


def run_epoch_cluster(g, mode):
    model, tm = build(g, mode)
    out = {"envs0": tm.envs.cpu().numpy(), "state0": np.random.get_state()}
    tm.stat_envs()
    tm.train_a_epoch()
    np.random.seed(g.seed + 1)
    out["diff"] = tm.cluster()
    out["cnt"] = tm.stat_envs()
    out["envs"] = tm.envs.cpu().numpy()
    out["sw"] = tm.sample_weights.cpu().numpy()
    out["cw"] = tm.class_weights.cpu().numpy()
    out["sd"] = {k: v.cpu().numpy() for k, v in model.state_dict().items()}
    out["state1"] = np.random.get_state()
    u, i, y = tm.users_tensor[:g.B], tm.items_tensor[:g.B], tm.scores_tensor[:g.B]
    out["batch"] = tm.cluster_a_batch(u, i, y).cpu().numpy()
    out["state2"] = np.random.get_state()
    return out


@pytest.mark.parametrize("case", CASES)
def test_trainer_numpy_device_equals_numpy(case):
    g = Golden(case)
    a, b = run_epoch_cluster(g, "numpy"), run_epoch_cluster(g, "numpy_device")
    assert np.array_equal(a["envs0"], g["envs0"]) and np.array_equal(b["envs0"], g["envs0"])
    for k in ("state0", "state1", "state2"):
        assert same_state(a[k], b[k]), k
    assert a["diff"] == b["diff"] and a["cnt"] == b["cnt"]
    for k in ("envs", "sw", "cw", "batch"):
        assert np.array_equal(a[k], b[k]), k
    for k in a["sd"]:
        assert np.array_equal(a["sd"][k], b["sd"][k]), k


@pytest.mark.parametrize("case", CASES)
def test_trainer_train_numpy_device_equals_numpy(case):
    g = Golden(case)
    res = []
    for mode in ("numpy", "numpy_device"):
        _, tm = build(g, mode, epochs=3)
        res.append((tm.train(silent=True, auto=True), np.random.get_state()))
    (ta, sa), (tb, sb) = res
    assert ta == tb
    assert same_state(sa, sb)


# ---------------------------------------------------------------------------------------------- sharded trainer
def sharded(g, world, rank, mode):
    from invpref_kdd_2022_b200.dist_train import ShardedExplicitTrainManager, ShardedImplicitTrainManager
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    from invpref_kdd_2022_b200.parallel import SimDriver
    torch.manual_seed(g.seed)
    M = InvPrefImplicit if g.implicit else InvPrefExplicit
    model = M(g.U, g.I, g.K, g.D, g.roe, g.ree).to(DEV)
    init = {k: p.data.clone() for k, p in model.named_hot_params().items()}
    np.random.seed(g.seed)
    T = ShardedImplicitTrainManager if g.implicit else ShardedExplicitTrainManager
    return T(g.U, g.I, g.K, g.D, torch.LongTensor(g.data), DEV, batch_size=g.B, epochs=2, cluster_interval=1,
             evaluate_interval=1, lr=g.lr, invariant_coe=g.coef["c_inv"], env_aware_coe=g.coef["c_ea"],
             env_coe=g.coef["c_env"], L2_coe=g.coef["c_L2"], L1_coe=g.coef["c_L1"], alpha=g.alpha,
             use_class_re_weight=g.crw, use_recommend_re_weight=g.rrw, reg_only_embed=g.roe, reg_env_embed=g.ree,
             init=init, driver=None if world == 1 else SimDriver(world), rank=rank, world=world, tie_break_rng=mode)


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("case", ["coat_explicit", "implicit_k6"])
def test_sharded_draws_numpy_device_equal_numpy(case, world):
    """Every rank of G = 2, 3: the same initial envs (its rows of the global draw) and the same tie-break rows of every
    global batch as the host path, with numpy's stream in the same place afterwards."""
    g = Golden(case)
    K_fact = len(g["eps_table"])
    for rank in range(world):
        a = sharded(g, world, rank, "numpy")
        sa = np.random.get_state()
        b = sharded(g, world, rank, "numpy_device")
        assert same_state(sa, np.random.get_state())
        assert torch.equal(a.envs, b.envs)
        assert np.array_equal(a.envs.cpu().numpy(), g["envs0"][a.rows.cpu().numpy()])
        np.random.seed(g.seed + 2)
        want = []
        for bi in range(a.batch_num):
            lo, hi = a._lo[bi], a._lo[bi + 1]
            cnt = min(g.N, (bi + 1) * g.B) - bi * g.B
            idx = torch.from_numpy(np.random.randint(0, K_fact, cnt)).to(DEV)
            want.append(idx[a.rows[lo:hi] - bi * g.B])
        sw = np.random.get_state()
        np.random.seed(g.seed + 2)
        for bi in range(b.batch_num):
            cnt = min(g.N, (bi + 1) * g.B) - bi * g.B
            assert torch.equal(b._global_draw(K_fact, bi, cnt, g.B), want[bi])
        assert same_state(sw, np.random.get_state())


@pytest.mark.parametrize("case", ["coat_explicit", "implicit_k6"])
def test_sharded_world1_cluster_numpy_device_equals_numpy(case):
    g = Golden(case)
    res = []
    for mode in ("numpy", "numpy_device"):
        tm = sharded(g, 1, 0, mode)
        tm.stat_envs()
        tm.train_a_epoch()
        np.random.seed(g.seed + 1)
        diff = tm.cluster()
        cnt = tm.stat_envs()
        res.append((diff, cnt, tm.envs.cpu().numpy(), tm.sample_weights.cpu().numpy(), np.random.get_state(),
                    tm.train(silent=True, auto=True)))
    (da, ca, ea, wa, sa, ta), (db, cb, eb, wb, sb, tb) = res
    assert da == db and ca == cb and np.array_equal(ea, eb) and np.array_equal(wa, wb) and same_state(sa, sb)
    assert ta == tb


def test_bad_mode():
    g = Golden("coat_explicit")
    with pytest.raises(ValueError):
        build(g, "numpy_host")
    with pytest.raises(ValueError):
        sharded(g, 1, 0, "device")

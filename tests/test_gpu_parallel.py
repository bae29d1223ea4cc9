"""GPU (one device): the multi-GPU step code run as G simulated ranks in one process (SimDriver executes the
collectives the step generators yield) must reproduce the single-GPU result on the same global batches:
losses, every table row, env assignments.  This is the "fake collective" test of SURVEY.md §4; the real NCCL
path runs the same generators under DistDriver (tests/test_dist_gloo.py covers the drivers on CPU)."""
import numpy as np
import pytest
import torch

from oracle import invpref_numpy as on

pytestmark = pytest.mark.gpu
TOL = 1e-5


def nerr(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = np.abs(b).max()
    return float(np.abs(a - b).max() / (den if den > 0 else 1.0))


def synth(U, I, N, K, D, implicit, seed):
    rng = np.random.default_rng(seed)
    u = np.floor(U * rng.random(N) ** 1.5).astype(np.int64)
    i = np.floor(I * rng.random(N) ** 3).astype(np.int64)
    y = (rng.integers(0, 2, N) if implicit else rng.integers(1, 6, N)).astype(np.float32)
    e = rng.integers(0, K, N).astype(np.int64)
    w = rng.random(N).astype(np.float32)
    p = {"Uinv": rng.normal(0, 0.1, (U, D)), "Iinv": rng.normal(0, 0.1, (I, D)), "Uenv": rng.normal(0, 0.3, (U, D)),
         "Ienv": rng.normal(0, 0.3, (I, D)), "E": rng.normal(0, 0.5, (K, D)), "W": rng.normal(0, 0.3, (K, D)),
         "b": rng.normal(0, 0.1, (K,))}
    return u, i, y, e, w, {k: v.astype(np.float32) for k, v in p.items()}


KW = dict(c_inv=0.8, c_ea=1.7, c_env=1.1, c_L2=0.6, c_L1=0.03, alpha=1.3, use_class_rw=True, use_rec_rw=True)


def single_gpu(p, batches, implicit, roe, ree, lr):
    from invpref_kdd_2022_b200.engine import HotPath
    dev = torch.device("cuda:0")
    hp = HotPath({k: torch.tensor(v, device=dev) for k, v in p.items()}, implicit, roe, ree, lr=lr)
    t = lambda a: torch.tensor(a, device=dev)
    losses = [hp.train_step(t(u), t(i), t(y), t(e), t(w), **KW).cpu().numpy().copy() for (u, i, y, e, w) in batches]
    return hp, np.asarray(losses)


@pytest.mark.parametrize("exchange", ["collective", "push"])
@pytest.mark.parametrize("lazy", [True, False])
@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("implicit,roe,ree", [(False, True, False), (True, False, True)])
def test_sharded_matches_single_gpu(world, implicit, roe, ree, lazy, exchange):
    from invpref_kdd_2022_b200.parallel import ShardedTrainer, SimDriver
    dev = torch.device("cuda:0")
    U, I, K, D, B = 1000, 203, 4, 64, 20000
    u, i, y, e, w, p = synth(U, I, 2 * B + 777, K, D, implicit, 5)
    bounds = on.mini_batch_bounds(len(u), B)                               # 3 batches, the last one short
    batches = [(u[a:b], i[a:b], y[a:b], e[a:b], w[a:b]) for a, b in bounds]
    ref, ref_losses = single_gpu(p, batches, implicit, roe, ree, 1e-2)
    init = {k: torch.tensor(v, device=dev) for k, v in p.items()}
    ranks = [ShardedTrainer(U, I, K, D, implicit, roe, ree, 1e-2, r, world, dev, cache_rows=I, init=init, lazy=lazy,
                            stage_rows=2 * I if exchange == "push" else 0) for r in range(world)]
    if exchange == "push":
        _wire_push(ranks)
    sim = SimDriver(world)
    t = lambda a: torch.tensor(a, device=dev)
    losses = []
    for (bu, bi, by, be, bw) in batches:
        sbs = sim.run_all([rk.prepare_gen(t(bu), t(bi), t(by)) for rk in ranks])
        assert sum(sb.sel.numel() for sb in sbs) == len(bu)
        outs = sim.run_all([rk.step_gen(sb, t(be)[sb.sel].contiguous(), t(bw)[sb.sel].contiguous(), **KW)
                            for rk, sb in zip(ranks, sbs)])
        for o in outs[1:]:
            assert torch.equal(o, outs[0])                                  # replicated results identical
        losses.append(outs[0].cpu().numpy().copy())
    assert np.abs(np.asarray(losses) - ref_losses).max() <= TOL * np.abs(ref_losses).max()
    full = {k: ref.params[k].cpu().numpy() for k in on.PARAM_ORDER}
    for r, rk in enumerate(ranks):
        loc = {k: v.cpu().numpy() for k, v in rk.local_tables().items()}
        # three Adam steps with a different (but fixed) summation order of the item partials: Adam's
        # g/(|g|+eps) amplification of tiny gradients allows ~1e-4 (BASELINE.md, multi-step drift)
        for k in ("Uinv", "Uenv", "Iinv", "Ienv"):
            assert nerr(loc[k], full[k][r::world]) <= 2e-4, (k, r)
        for k in ("E", "W", "b"):
            assert nerr(loc[k], full[k]) <= 2e-4, (k, r)
    # EM re-assignment on the last batch: the union of the ranks' results equals the single-GPU result
    bu, bi, by, be, bw = batches[-1]
    eps = torch.tensor(on.init_eps(K), device=dev)
    pidx = torch.tensor(np.random.default_rng(0).integers(0, eps.shape[0], len(bu)), device=dev)
    new_ref, hist_ref, diff_ref = ref.cluster(t(bu), t(bi), t(by), pidx, eps, t(be))
    res = sim.run_all([rk.cluster_gen(sb, pidx[sb.sel].contiguous(), eps, t(be)[sb.sel].contiguous())
                       for rk, sb in zip(ranks, sbs)])
    new = torch.empty_like(new_ref)
    for sb, (nv, hist, diff) in zip(sbs, res):
        new[sb.sel] = nv
    mism = (new != new_ref).cpu().numpy()
    dist = on.cluster_distances(full, bu, bi, by, on.Flags(implicit, roe, ree))
    assert not (mism & ~on.near_tie_mask(dist)).any()
    assert sum(int(h.sum()) for _, h, _ in res) == len(bu)


@pytest.mark.parametrize("world", [2, 4])
def test_replicated_matches_single_gpu(world):
    from invpref_kdd_2022_b200.parallel import ReplicatedTrainer, SimDriver
    dev = torch.device("cuda:0")
    U, I, K, D, B = 300, 120, 6, 40, 9000
    u, i, y, e, w, p = synth(U, I, 2 * B + 100, K, D, True, 9)
    bounds = on.mini_batch_bounds(len(u), B)
    batches = [(u[a:b], i[a:b], y[a:b], e[a:b], w[a:b]) for a, b in bounds]
    ref, ref_losses = single_gpu(p, batches, True, False, True, 1e-2)
    ranks = [ReplicatedTrainer({k: torch.tensor(v, device=dev) for k, v in p.items()}, True, False, True, 1e-2, r,
                               world) for r in range(world)]
    sim = SimDriver(world)
    t = lambda a: torch.tensor(a, device=dev)
    losses = []
    for (bu, bi, by, be, bw) in batches:
        gens = []
        for rk in ranks:
            a, b = rk.chunk(0, len(bu))
            gens.append(rk.step_gen(t(bu[a:b]), t(bi[a:b]), t(by[a:b]), t(be[a:b]), t(bw[a:b]), len(bu), **KW))
        outs = sim.run_all(gens)
        losses.append(outs[0].cpu().numpy().copy())
    assert np.abs(np.asarray(losses) - ref_losses).max() <= TOL * np.abs(ref_losses).max()
    for rk in ranks:
        assert torch.equal(rk.flat, ranks[0].flat)
        for k in on.PARAM_ORDER:
            assert nerr(rk.params[k].cpu().numpy(), ref.params[k].cpu().numpy()) <= 2e-4, k


def _wire_push(ranks):
    """Push exchange between simulated ranks: peer pointers = the other ranks' tensors on the same device."""
    for rk in ranks:
        rk.enable_push([[x.Iinv.data_ptr() for x in ranks], [x.Ienv.data_ptr() for x in ranks]],
                       [[[x.stage[par][t].data_ptr() for x in ranks] for t in range(2)] for par in range(2)],
                       [[x.cache[t].data_ptr() for x in ranks] for t in range(2)])


@pytest.mark.parametrize("lazy", [True, False])
def test_sharded_push_exchange_is_bitwise_the_collective_path(lazy):
    """Two exchanges of the item rows / partial item gradients, same arithmetic in the same (rank) order:
      collective  gather_rows -> all-to-all -> cache; gradients all-to-all back -> scatter_add per rank -> adam_dense
      push        the item pass stores its partials into the owners' staging buffers (invpref_push), the owner
                  reduces from local memory and stores the updated rows into the requesters' next-batch caches
                  (invpref_owner_adam_push)
    must give bit-identical losses, tables and moments over several steps (double-buffered staging: 5 steps)."""
    from invpref_kdd_2022_b200.parallel import ShardedTrainer, SimDriver
    dev = torch.device("cuda:0")
    world, U, I, K, D, B, S = 3, 700, 151, 4, 64, 12000, 5
    u, i, y, e, w, p = synth(U, I, S * B, K, D, False, 11)
    init = {k: torch.tensor(v, device=dev) for k, v in p.items()}
    t = lambda a: torch.tensor(a, device=dev)
    out = []
    for mode in ("collective", "push"):
        ranks = [ShardedTrainer(U, I, K, D, False, True, False, 1e-2, r, world, dev, cache_rows=I, init=init,
                                lazy=lazy, stage_rows=(2 * I if mode == "push" else 0)) for r in range(world)]
        if mode == "push":
            _wire_push(ranks)
        sim = SimDriver(world)
        losses = []
        sbs_all = []
        for s in range(S):
            sl = slice(s * B, (s + 1) * B)
            sbs_all.append(sim.run_all([rk.prepare_gen(t(u[sl]), t(i[sl]), t(y[sl])) for rk in ranks]))
        for s in range(S):
            sl = slice(s * B, (s + 1) * B)
            sbs = sbs_all[s]
            nxt = sbs_all[s + 1] if s + 1 < S else [None] * world
            res = sim.run_all([rk.step_gen(sb, t(e[sl])[sb.sel].contiguous(), t(w[sl])[sb.sel].contiguous(),
                                           next_sb=nx, **KW) for rk, sb, nx in zip(ranks, sbs, nxt)])
            losses.append(res[0].clone())
        # a re-assignment after training reads the item rows through a fresh fetch (peer-memory loads under push)
        eps = torch.tensor(on.init_eps(K), device=dev)
        sl = slice(0, B)
        cl = sim.run_all([rk.cluster_gen(sb, None, None, t(e[sl])[sb.sel].contiguous())
                          for rk, sb in zip(ranks, sbs_all[0])])
        out.append((losses, [{k: v.clone() for k, v in rk.local_tables().items()} for rk in ranks],
                    [c[0].clone() for c in cl]))
    for other in out[1:]:
        for a, b in zip(out[0][0], other[0]):
            assert torch.equal(a, b)
        for ta, tb in zip(out[0][1], other[1]):
            for k in ta:
                assert torch.equal(ta[k], tb[k]), k
        for a, b in zip(out[0][2], other[2]):
            assert torch.equal(a, b)


def _managers(g, world, rank, driver, epochs=2, **kw):
    """A single-GPU ExplicitTrainManager/ImplicitTrainManager and the sharded manager, same seeds, same init."""
    from invpref_kdd_2022_b200.dist_train import ShardedExplicitTrainManager, ShardedImplicitTrainManager
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    dev = torch.device("cuda:0")
    torch.manual_seed(g.seed)
    M = InvPrefImplicit if g.implicit else InvPrefExplicit
    model = M(g.U, g.I, g.K, g.D, g.roe, g.ree).to(dev)
    init = {k: p.data.clone() for k, p in model.named_hot_params().items()}
    np.random.seed(g.seed)
    T = ShardedImplicitTrainManager if g.implicit else ShardedExplicitTrainManager
    return T(g.U, g.I, g.K, g.D, torch.LongTensor(g.data), dev, batch_size=g.B, epochs=epochs, cluster_interval=1,
             evaluate_interval=1, lr=g.lr, invariant_coe=g.coef["c_inv"], env_aware_coe=g.coef["c_ea"],
             env_coe=g.coef["c_env"], L2_coe=g.coef["c_L2"], L1_coe=g.coef["c_L1"], alpha=g.alpha,
             use_class_re_weight=g.crw, use_recommend_re_weight=g.rrw, reg_only_embed=g.roe, reg_env_embed=g.ree,
             init=init, driver=driver, rank=rank, world=world, **kw)


@pytest.mark.parametrize("case", ["coat_explicit", "implicit_k6"])
def test_sharded_train_manager_world1_follows_the_golden_epoch(case):
    """The distributed trainer behind the reference API (dist_train.py), degenerate world = 1: one epoch, cluster(),
    stat_envs() against what the LIVE reference produced (tests/golden): same initial envs (numpy stream), same
    epoch losses, same env counts bookkeeping."""
    from _golden import Golden
    g = Golden(case)
    tm = _managers(g, 1, 0, None)
    assert np.array_equal(tm.envs.cpu().numpy(), g["envs0"])
    cnt = tm.stat_envs()
    assert sum(cnt.values()) == g.N
    assert np.array_equal(tm.sample_weights.cpu().numpy(), g["sample_weights0"])
    assert np.array_equal(tm.class_weights.cpu().numpy(), g["class_weights0"])
    mean_ld = tm.train_a_epoch()
    for j, k in enumerate(on.LOSS_KEYS):
        assert abs(mean_ld[k] - g["epoch_mean_loss"][j]) <= 1e-4 * abs(g["epoch_mean_loss"][j]), k
    loc = tm.trainer.local_tables()
    ep = g.group("epoch1")
    for k, sk in on.STATE_KEYS.items():
        assert nerr(loc[k].cpu().numpy(), ep[sk]) <= 5e-4, k
    np.random.seed(g.seed + 1)
    diff = tm.cluster()
    new = tm.envs.cpu().numpy()
    assert diff == int((new != g["envs0"]).sum())
    cnt = tm.stat_envs()
    assert [cnt[k] for k in range(g.K)] == np.bincount(new, minlength=g.K).tolist()
    assert np.array_equal(tm.sample_weights.cpu().numpy(), on.stat_envs(new, g.K, g.N)[2])
    (losses, ep_idx), _, (diffs, cnts, cl_ep) = tm.train(silent=True, auto=True)
    assert ep_idx == [2] and cl_ep == [2] and sum(cnts[0].values()) == g.N

"""bench.py's multi-GPU leg: one process per GPU under torchrun (NCCL), see parallel.py.

Fixed global workload (strong scaling): the same global batches as the 1-GPU run are split over the ranks.
Timed region: K steps between a barrier + synchronize on both sides, CUDA events on every rank, MAX over
ranks; value = K * global_batch / that time.

Legs of the one JSON line rank 0 prints:
  headline        C5 (10 M x 1 M, D 64, B 2^22), users + items row-sharded, item exchange over peer memory
                  (INVPREF_EXCHANGE = push (default) | nccl);
  parity_vs_1gpu  a reduced shape trained for a few steps by the N ranks (same exchange) AND by rank 0 alone: losses
                  and every gathered table compared (tolerance: the summation order of the item partials differs), plus
                  bit-equality of the peer-memory exchange with the NCCL all-to-all exchange on the real ranks;
  configs.c4      MIND-shaped config (BASELINE.json configs[3]: "data-parallel at 1/2/4/8 B200") on the same ranks.
"""
from __future__ import annotations

import json
import os
import time

import numpy as np
import torch
import torch.distributed as dist


def _exchange_mode():
    m = (os.environ.get("INVPREF_EXCHANGE") or "push").lower()
    if m not in ("push", "nccl"):
        raise ValueError(f"INVPREF_EXCHANGE must be 'push' or 'nccl', not {m!r}")
    return m


def make_sharded(w, U, I, Bg, rank, world, dev, mode, init=None, lazy=True, sync=None):
    """A ShardedTrainer wired for `mode` ("push" or "nccl"); falls back (all ranks together) to the NCCL exchange if
    symmetric memory is unavailable.  Returns (trainer, note, mode)."""
    from invpref_kdd_2022_b200.parallel import ShardedTrainer, SymmetricItemStorage
    K, D = w["K"], w["D"]
    cache_rows = min(I, Bg // world * 2 + 1024)
    stage_rows = min(2 * cache_rows, (I + world - 1) // world * world)
    store, why = None, "disabled (INVPREF_EXCHANGE=nccl)"
    peer_sync = os.environ.get("INVPREF_SYNC", "peer").lower() != "nccl" if sync is None else bool(sync)
    n_small = 2 * K * D + K + 6
    if mode == "push":
        try:
            store = SymmetricItemStorage(I, D, world, cache_rows, dev, dist.group.WORLD, stage_rows=stage_rows,
                                         sync_floats=n_small if peer_sync else 0)
            why = ""
        except Exception as ex:      # noqa: BLE001 -- any failure means "use NCCL"
            store, why = None, f"{type(ex).__name__}: {ex}"[:200]
    elif sync:      # NCCL row / gradient exchange, but the step's all-reduce + barriers over peer memory
        try:        # (parity_check: isolates the exchange path, same summation order of E / W / b)
            store = SymmetricItemStorage(I, D, world, cache_rows, dev, dist.group.WORLD, sync_floats=n_small)
        except Exception:            # noqa: BLE001
            store = None
    ok = torch.tensor([1 if (store is not None or not (mode == "push" or sync)) else 0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok.item()) == 0:
        store, mode = None, "nccl"
    tr = ShardedTrainer(U, I, K, D, w["implicit"], w["roe"], w["ree"], w["lr"], rank, world, dev,
                        cache_rows=cache_rows, init=init, lazy=lazy, store=store)
    if tr.push is not None:
        note = "peer memory (torch symmetric memory): item pass pushes partial gradients into the owners' " \
               "staging, owners push updated rows into the requesters' next-batch caches (posted NVLink writes)"
        if tr.sync is not None:
            note += "; E/W/b gradient all-reduce and both step barriers over peer memory too (invpref_peer_allreduce: " \
                    "no NCCL call in the step)"
    else:
        note = "NCCL all-to-all (" + (why or "a peer could not map symmetric memory") + ")"
    torch.cuda.synchronize()
    dist.barrier()                       # every shard initialised before anyone touches a peer's memory
    return tr, note, mode


def prepare_all(tr, drv, batches, dev):
    t = lambda a: torch.from_numpy(a).to(dev)
    prepared = []
    for (u, i, y, e) in batches:
        sb = drv.run(tr.prepare_gen(t(u), t(i), t(y)))
        ge = t(e)
        gw = tr.hot.stat_envs(ge, tr.hot.env_hist(ge))[1]          # sample weights of the GLOBAL batch (train.py:945-957)
        prepared.append((sb, ge[sb.sel].contiguous(), gw[sb.sel].contiguous()))
    return prepared


def parity_check(rank, world, dev, mode, drv):
    """A few steps of a reduced shape on the REAL ranks vs the same batches on rank 0 alone (1-GPU engine), and the
    peer-memory exchange vs the NCCL exchange bit for bit.  Returns a dict on rank 0."""
    import bench as B
    from invpref_kdd_2022_b200.engine import HotPath
    # Shape of C5 scaled down; coefficients and table scales of the simulated-rank tests (tests/test_gpu_parallel.py):
    # at the N(0, 0.01) init and the Yahoo coefficients the user-invariant gradients are ~1e-8 = Adam's eps, where
    # g / (|g| + eps) turns summation-order noise into +-lr steps (BASELINE.md) and no two orders agree to 2e-4.
    w = dict(B.WORKLOADS["c5"], U=400_000, I=60_000, B=1 << 18,
             coef=dict(c_inv=0.8, c_ea=1.7, c_env=1.1, c_L2=0.6, c_L1=0.03))
    steps = 4
    U, I, Bg, batches = B.synth_batches(w, steps, seed=77)
    kw = dict(alpha=1.3, use_class_rw=w["crw"], use_rec_rw=w["rrw"], **w["coef"])
    init = B.make_tables(w, dev, U=U, I=I, seed=123)                 # same seed on every rank: identical tables
    for k, sc in (("Uinv", 10.0), ("Iinv", 10.0), ("Uenv", 30.0), ("Ienv", 30.0), ("E", 50.0), ("W", 3.0)):
        init[k] *= sc
    res = {}
    used_sync = None
    for m in dict.fromkeys((mode, "nccl")):
        # the NCCL-exchange twin uses the same synchronisation primitive as the main leg: what is compared bit for
        # bit is the item exchange (rows + partial gradients), not the summation order of an NCCL all-reduce
        tr, _, got = make_sharded(w, U, I, Bg, rank, world, dev, m, init=init, sync=used_sync)
        if used_sync is None:
            used_sync = tr.sync is not None
        prep = prepare_all(tr, drv, batches, dev)
        losses = []
        for s in range(steps):
            sb, le, sw = prep[s]
            nxt = prep[s + 1][0] if s + 1 < steps else None
            losses.append(drv.run(tr.step_gen(sb, le, sw, next_sb=nxt, **kw)).clone())
        tr.flush()
        torch.cuda.synchronize()
        tr.check_sync()
        dist.barrier()
        res[m] = (torch.stack(losses), {k: v.clone() for k, v in tr.local_tables().items()}, got)
        del tr, prep
        torch.cuda.empty_cache()
    # (1) exchange paths bit-identical on every rank
    same = 1
    if mode != "nccl" and res[mode][2] == mode:
        a, b = res[mode], res["nccl"]
        same = int(torch.equal(a[0], b[0]) and all(torch.equal(a[1][k], b[1][k]) for k in a[1]))
    flag = torch.tensor([same], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    # (2) against one GPU: gather the shards on rank 0
    losses, loc, _ = res[mode]
    out = None
    gathered = {}
    for k in ("Uinv", "Uenv", "Iinv", "Ienv"):
        rows = (U if k[0] == "U" else I)
        per = (rows + world - 1) // world
        pad = torch.zeros((per, w["D"]), device=dev)
        pad[:loc[k].shape[0]] = loc[k]
        bufs = [torch.zeros_like(pad) for _ in range(world)] if rank == 0 else None
        dist.gather(pad, bufs, dst=0)
        if rank == 0:
            full = torch.zeros((per * world, w["D"]), device=dev)
            for r in range(world):
                full[r::world] = bufs[r]
            gathered[k] = full[:rows]
    if rank == 0:
        hp = HotPath({k: v.clone() for k, v in init.items()}, w["implicit"], w["roe"], w["ree"], lr=w["lr"], lazy=True)
        ref_losses = []
        for (u, i, y, e) in batches:
            u, i, y, e = (torch.from_numpy(a).to(dev) for a in (u, i, y, e))
            sw = hp.stat_envs(e, hp.env_hist(e))[1]
            ref_losses.append(hp.train_step(u, i, y, e, sw, **kw).clone())
        hp.flush()
        ref_losses = torch.stack(ref_losses)
        nerr = lambda a, b: float((a - b).abs().max() / b.abs().max())
        terr = {k: nerr(gathered[k], hp.params[k]) for k in gathered}
        terr.update({k: nerr(loc[k], hp.params[k]) for k in ("E", "W", "b")})
        lerr = float(((losses - ref_losses).abs() / ref_losses.abs()).max())
        out = {"shape": f"U={U} I={I} D={w['D']} K={w['K']} B={Bg}, {steps} steps, exchange={res[mode][2]}",
               "max_rel_loss_err": lerr, "max_table_err": max(terr.values()), "table_err": terr,
               "tolerance": {"loss": 1e-5, "tables": 2e-4,
                             "why": "the item partials of a row are summed per rank, then across ranks in rank order: "
                                    "a different (fixed) order than the single-GPU sorted order"},
               "pass": bool(lerr <= 1e-5 and max(terr.values()) <= 2e-4),
               "peer_memory_bitwise_equals_nccl": bool(int(flag.item())),
               "sync": "invpref_peer_allreduce (both legs)" if used_sync else "NCCL all-reduce"}
        del hp
    del res, gathered
    torch.cuda.empty_cache()
    dist.barrier()
    return out


def timed_sharded(args, w, rank, world, dev, mode, drv, nb, steps, warmup, want_e2e=True):
    """Times `steps` sharded steps of workload `w`; returns the pieces of the JSON line (rank 0) or None."""
    import bench as B
    from invpref_kdd_2022_b200 import _lib
    K, D = w["K"], w["D"]
    U, I, Bg, batches = B.synth_batches(w, nb)
    P = 2 * (U + I) * D + 2 * K * D + K
    kw = dict(alpha=1.0, use_class_rw=w["crw"], use_rec_rw=w["rrw"], **w["coef"])
    tr, note, mode = make_sharded(w, U, I, Bg, rank, world, dev, mode)
    prepared = prepare_all(tr, drv, batches, dev)

    def step(s):
        sb, le, sw = prepared[s % nb]
        return drv.run(tr.step_gen(sb, le, sw, next_sb=prepared[(s + 1) % nb][0], **kw))

    for s in range(warmup):
        step(s)
    tr.flush()
    torch.cuda.synchronize()
    tr.phase_events = []
    clocks = B.ClockSampler(dev.index)
    if rank == 0:
        clocks.start()
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    torch.cuda.synchronize()
    ev0.record()
    for s in range(warmup, warmup + steps):
        loss = step(s)
    tr.flush()            # lazy Adam: every local user row brought up to date inside the timed region
    ev1.record()
    torch.cuda.synchronize()
    dist.barrier()
    launches = _lib.launch_count() - l0
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item()) / steps
    assert torch.isfinite(loss).all()
    clk = clocks.stop() if rank == 0 else None
    phases = {}
    evs = tr.phase_events
    for (n0, e0), (n1, e1) in zip(evs[:-1], evs[1:]):
        if n1 != "start":
            phases[n1] = phases.get(n1, 0.0) + e0.elapsed_time(e1) / steps
    tr.phase_events = None
    phases["cache_rows"], phases["local_batch"] = prepared[0][0].route.n_cache, int(prepared[0][0].users.numel())
    # bytes one rank moves over NVLink per step (either direction): partial gradients out + updated rows in/out
    xrows = float(np.mean([sb.route.n_cache - sb.route.recv_splits[rank] for sb, _, _ in prepared]))
    nvl = {"rows_per_rank_per_direction": xrows, "bytes_per_rank_per_direction": xrows * D * 4 * 2}
    ex_ms = phases.get("item_adam", 0.0) + phases.get("prefetch_next", 0.0) + phases.get("grad_a2a", 0.0) + \
        phases.get("small", 0.0)
    nvl["exchange_ms_rank0"] = ex_ms
    if ex_ms > 0:
        nvl["achieved_GBs_per_direction"] = 2 * nvl["bytes_per_rank_per_direction"] / (ex_ms * 1e-3) / 1e9
        nvl["frac_of_900"] = nvl["achieved_GBs_per_direction"] / 900.0
        nvl["note"] = "gradients out + rows in, over the time of everything after the local step (barriers included); " \
                      "in push mode most gradient bytes move DURING the item pass and are not on this clock"
    e2e = None
    if want_e2e:
        # e2e at N GPUs: per step every rank copies its share's ids (local user rows, item cache slots), scores, envs
        # and sample weights from pinned host memory and rebuilds the sort-segment plan of its share on a loader
        # stream (as the 1-GPU e2e leg does); the item ROUTE (which rows come from which owner) is static per batch
        # and stays resident.  The six losses go back to the host every step and are read one step later.
        host = [tuple(x.cpu().pin_memory() for x in (sb.users, sb.route.slots, sb.scores, le, sw))
                for sb, le, sw in prepared[:min(nb, 4)]]
        nh = len(host)
        loader = torch.cuda.Stream(device=dev)
        plan_bufs = [torch.empty(tr.hot.plan_bytes(max(int(sb.users.numel()) for sb, _, _ in prepared) + 1),
                                 dtype=torch.uint8, device=dev) for _ in range(2)]
        h_loss = torch.empty((2, 6)).pin_memory()
        read_back = [torch.cuda.Event(), torch.cuda.Event()]
        e2e_steps = max(3, min(steps, 32))
        ready = [torch.cuda.Event(), torch.cuda.Event()]
        seen = []

        def issue(s):
            j = s % nh
            sb, le, sw = prepared[j]
            with torch.cuda.stream(loader):
                for dst, src in zip((sb.users, sb.route.slots, sb.scores, le, sw), host[j]):
                    dst.copy_(src, non_blocking=True)
                if sb.users.numel():
                    sb.plan = tr.hot.new_plan(sb.users, sb.route.slots, out=plan_bufs[s % 2])
                ready[s % 2].record(loader)

        def e2e_step(s, first, last):
            if not last:
                issue(s + 1)
            torch.cuda.current_stream().wait_event(ready[s % 2])
            sb, le, sw = prepared[s % nh]
            out = drv.run(tr.step_gen(sb, le, sw, next_sb=prepared[(s + 1) % nh][0], **kw))
            loader.wait_stream(torch.cuda.current_stream())
            h_loss[s % 2].copy_(out, non_blocking=True)      # this step's six losses -> pinned host memory
            read_back[s % 2].record()
            if not first:                                     # the host reads step s-1's losses while step s runs (as the
                read_back[(s - 1) % 2].synchronize()          # 1-GPU leg does): every step's result is read
                seen.append(float(h_loss[(s - 1) % 2][5]))

        issue(0)
        e2e_step(0, True, False)
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in range(1, e2e_steps + 1):
            e2e_step(s, s == 1, s == e2e_steps)
        read_back[e2e_steps % 2].synchronize()
        seen.append(float(h_loss[e2e_steps % 2][5]))
        tr.flush()
        torch.cuda.synchronize()
        dist.barrier()
        assert len(seen) == e2e_steps and all(np.isfinite(seen))
        e2e_ms = torch.tensor([(time.perf_counter() - t0) / e2e_steps * 1e3], device=dev)
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
        h2d = torch.tensor([sum(t_.numel() * t_.element_size() for t_ in host[0])], device=dev, dtype=torch.float64)
        dist.all_reduce(h2d)
        e2e = {"value": Bg / (float(e2e_ms.item()) * 1e-3), "unit": "interactions/s", "ms_per_step": float(e2e_ms.item()),
               "h2d_bytes_per_step": int(h2d.item()), "d2h_bytes_per_step": 24 * world, "steps": e2e_steps,
               "note": "per step every rank copies its share (local user rows, item cache slots, scores, envs, sample "
                       "weights) from pinned host memory and rebuilds its sort-segment plan on a loader stream under "
                       "the previous step, runs the step, copies the six losses D2H; the host reads them one step later (while the "
                       "next step runs), as in the 1-GPU leg.  Unlike the "
                       "1-GPU leg the interactions arrive already routed to their user's owner and the item route "
                       "(which rows from which owner) is resident: building it needs a collective per batch"}
    del tr, prepared
    torch.cuda.empty_cache()
    return dict(ms=ms, Bg=Bg, P=P, D=D, K=K, note=note, mode=mode, launches=launches, clk=clk, phases=phases, nvl=nvl,
                e2e=e2e, loss=float(loss[5]))


def timed_replicated(w, rank, world, dev, drv, nb, steps, warmup):
    """SURVEY.md 8e "replicated tables": every rank holds all tables, takes a contiguous 1/world chunk of each global
    batch, exports its partial dense gradients; ONE all-reduce of the flat gradient (+ loss sums) per step, then the
    same dense Adam everywhere (parallel.ReplicatedTrainer).  Returns (ms per step, launches per step, final loss)."""
    import bench as B
    from invpref_kdd_2022_b200 import _lib
    from invpref_kdd_2022_b200.parallel import ReplicatedTrainer
    U, I, Bg, batches = B.synth_batches(w, nb)
    kw = dict(alpha=1.0, use_class_rw=w["crw"], use_rec_rw=w["rrw"], **w["coef"])
    init = B.make_tables(w, dev, U=U, I=I, seed=123)                  # same seed on every rank: identical replicas
    tr = ReplicatedTrainer(init, w["implicit"], w["roe"], w["ree"], w["lr"], rank, world)
    t = lambda a: torch.from_numpy(a).to(dev)
    prepared = []
    for (u, i, y, e) in batches:
        lo, hi = tr.chunk(0, Bg)
        ge = t(e)
        gw = tr.hot.stat_envs(ge, tr.hot.env_hist(ge))[1]
        cu, ci = t(u[lo:hi]), t(i[lo:hi])
        prepared.append((cu, ci, t(y[lo:hi]), ge[lo:hi].contiguous(), gw[lo:hi].contiguous(), tr.hot.new_plan(cu, ci)))

    def step(s):
        cu, ci, cy, ce, cw, plan = prepared[s % nb]
        return drv.run(tr.step_gen(cu, ci, cy, ce, cw, Bg, plan=plan, **kw))

    for s in range(warmup):
        step(s)
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    dist.barrier()
    torch.cuda.synchronize()
    ev0.record()
    for s in range(warmup, warmup + steps):
        loss = step(s)
    ev1.record()
    torch.cuda.synchronize()
    dist.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    assert torch.isfinite(loss).all()
    out = float(ms.item()) / steps, (_lib.launch_count() - l0) / steps, float(loss[5]), Bg, tr.flat.numel()
    del tr, prepared
    torch.cuda.empty_cache()
    return out


def config_leg_sharded(name, rank, world, dev, mode):
    """A dataset-scale config through the PUBLIC distributed trainer API (dist_train.Sharded*TrainManager), like
    bench.config_leg does on one GPU: one synthetic epoch of the config's shape, wall clock over whole
    train_a_epoch() calls (per-epoch loss read-back included), max over ranks.  With the push exchange every epoch
    after the first is one CUDA-graph launch per rank (no NCCL call inside)."""
    import bench as B
    from invpref_kdd_2022_b200 import _lib
    from invpref_kdd_2022_b200.dataloader import synthetic_interactions
    from invpref_kdd_2022_b200.dist_train import ShardedExplicitTrainManager, ShardedImplicitTrainManager
    w = B.WORKLOADS[name]
    U, I, N, Bg, K, D = w["U"], w["I"], w["N"], w["B"], w["K"], w["D"]
    data = synthetic_interactions(U, I, N, w["implicit"])
    torch.manual_seed(17373331)
    np.random.seed(17373331)
    T = ShardedImplicitTrainManager if w["implicit"] else ShardedExplicitTrainManager
    c = w["coef"]
    tm = T(U, I, K, D, torch.LongTensor(data), dev, batch_size=Bg, epochs=1, cluster_interval=1, evaluate_interval=1,
           lr=w["lr"], invariant_coe=c["c_inv"], env_aware_coe=c["c_ea"], env_coe=c["c_env"], L2_coe=c["c_L2"],
           L1_coe=c["c_L1"], alpha=None, use_class_re_weight=w["crw"], use_recommend_re_weight=w["rrw"],
           reg_only_embed=w["roe"], reg_env_embed=w["ree"], exchange=mode)
    tm.stat_envs()
    for _ in range(3):                       # first epoch builds routes and plans, second captures the graph
        ld = tm.train_a_epoch()
    epochs = max(4, 60 // max(1, tm.batch_num))
    torch.cuda.synchronize()
    dist.barrier()
    l0 = _lib.launch_count()
    t0 = time.perf_counter()
    for _ in range(epochs):
        ld = tm.train_a_epoch()
    torch.cuda.synchronize()
    wall = torch.tensor([(time.perf_counter() - t0) / epochs * 1e3], device=dev)
    dist.all_reduce(wall, op=dist.ReduceOp.MAX)
    wall = float(wall.item())
    assert np.isfinite(ld["loss"])
    tc0 = time.perf_counter()
    for _ in range(2):
        tm.cluster()
        tm.stat_envs()
    torch.cuda.synchronize()
    cl = torch.tensor([(time.perf_counter() - tc0) / 2 * 1e3], device=dev)
    dist.all_reduce(cl, op=dist.ReduceOp.MAX)
    graph = bool(tm._graph is not None and len(tm._graph.handles) > 0)
    leg = {"workload": w["name"], "interactions_per_epoch": N, "steps_per_epoch": tm.batch_num, "global_batch": Bg,
           "value": N / (wall * 1e-3), "unit": "interactions/s", "ms_per_step": wall / tm.batch_num,
           "ms_per_epoch": wall, "scaling": "strong", "final_loss": float(ld["loss"]),
           "launches_per_step": (_lib.launch_count() - l0) / (epochs * tm.batch_num),
           "cuda_graph_epochs": graph, "peer_sync": tm.trainer.sync is not None, "exchange": tm.exchange,
           "timing": "wall clock over %d train_a_epoch() calls of the distributed trainer incl. the per-epoch loss "
                     "read-back, max over ranks" % epochs,
           "cluster": {"value": N / (float(cl.item()) * 1e-3), "unit": "samples/s", "ms": float(cl.item())},
           "parallelism": f"row-sharded over {world} ranks through dist_train.Sharded*TrainManager"}
    del tm
    torch.cuda.empty_cache()
    return leg


def run(args, w):
    from invpref_kdd_2022_b200.parallel import DistDriver
    import bench as B

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    # stdout carries exactly one JSON line: NCCL's version banner / debug log goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    dist.init_process_group("nccl", device_id=dev)
    drv = DistDriver()
    mode = _exchange_mode()
    nb = max(1, min(args.nbatch or 8, args.steps + args.warmup))
    parity = None
    if not args.no_parity:
        try:
            parity = parity_check(rank, world, dev, mode, drv)
        except Exception as ex:      # noqa: BLE001 -- reported, never fatal for the timing line
            parity = {"pass": False, "error": f"{type(ex).__name__}: {ex}"[:300]}
    r = timed_sharded(args, w, rank, world, dev, mode, drv, nb, args.steps, args.warmup)
    legs = {}
    if not args.no_config_legs and args.workload == "c5":
        w4 = B.WORKLOADS["c4"]
        try:
            r4 = timed_sharded(args, w4, rank, world, dev, mode, drv, 16, max(args.steps, 32), args.warmup,
                               want_e2e=False)
            legs["c4"] = {"workload": w4["name"], "value": r4["Bg"] / (r4["ms"] * 1e-3), "unit": "interactions/s",
                          "ms_per_step": r4["ms"], "global_batch": r4["Bg"], "distinct_batches": 16,
                          "parallelism": f"row-sharded over {world} ranks, {r4['note']}",
                          "launches_per_step": r4["launches"] / max(args.steps, 32), "rank0_phase_ms": r4["phases"],
                          "final_loss": r4["loss"]}
        except Exception as ex:      # noqa: BLE001
            legs["c4"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
        try:
            legs["c4_trainer"] = config_leg_sharded("c4", rank, world, dev, r["mode"])
        except Exception as ex:      # noqa: BLE001
            legs["c4_trainer"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
        try:
            ms_r, l_r, loss_r, bg_r, p_r = timed_replicated(w4, rank, world, dev, drv, 16, max(args.steps, 32),
                                                            args.warmup)
            legs["c4_replicated"] = {"workload": w4["name"], "value": bg_r / (ms_r * 1e-3), "unit": "interactions/s",
                                     "ms_per_step": ms_r, "global_batch": bg_r, "scaling": "strong",
                                     "launches_per_step": l_r, "final_loss": loss_r,
                                     "all_reduce_bytes_per_step": 4 * (p_r + 8),
                                     "parallelism": f"tables replicated on {world} ranks, contiguous batch chunks, one "
                                     "NCCL all-reduce of the flat dense gradient per step, dense Adam on every rank "
                                     "(SURVEY.md 8e, replicated-tables row)"}
        except Exception as ex:      # noqa: BLE001
            legs["c4_replicated"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
        # The same config as the reference driver scales it: MIND_InvPref.py:51,206 trains one independent model per
        # entry of RANDOM_SEED_LIST, one after the other.  Here every rank trains its own seed at the same time
        # through the single-GPU trainer API (no collective on the path): weak scaling, "replicas only" (DESIGN.md 5).
        try:
            dist.barrier()
            leg = B.config_leg("c4", dev, with_eager=False, seed=17373331 + 90 * rank, quick=True)
            v = torch.tensor([leg["value"]], device=dev, dtype=torch.float64)
            vs = [torch.zeros_like(v) for _ in range(world)]
            dist.all_gather(vs, v)
            vs = [float(x.item()) for x in vs]
            legs["c4_replicas"] = {"workload": w4["name"], "value": world * min(vs), "unit": "interactions/s",
                                   "scaling": "weak", "per_rank_value": vs, "ms_per_step_slowest_rank":
                                   leg["global_batch"] / min(vs) * 1e3, "launches_per_step": leg["launches_per_step"],
                                   "parallelism": f"{world} independent seeds, one single-GPU trainer per rank "
                                   "(train_a_epoch as one CUDA-graph launch), no collective; value = ranks x the slowest "
                                   "rank's interactions/s"}
        except Exception as ex:      # noqa: BLE001
            legs["c4_replicas"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
    peak, peak_src = B.measured_peaks()
    if rank == 0:
        Bg, P, D, K, ms = r["Bg"], r["P"], r["D"], r["K"], r["ms"]
        sbytes = B.step_bytes(Bg, D, K, P)
        mode_s = f"users+items row-sharded (mod {world}), interactions routed to the user's owner, item rows/grads " \
                 f"exchanged over {r['note']}, E/W/b all-reduce"
        line = {"metric": "train interactions/sec (fwd+bwd+Adam)", "value": Bg / (ms * 1e-3),
                "unit": "interactions/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": w["name"], "global_batch": Bg, "params": P, "distinct_batches": nb,
                           "l2": "inputs larger than L2" if P * 4 > 2.5e8 else "tables fit in L2 (no flush)",
                           "parallelism": mode_s, "exchange": r["mode"]},
                "roofline": {"bound": "hbm", "kernel": "fused train step (all kernels, all ranks), SURVEY.md 8d bytes",
                             "achieved": sbytes / (ms * 1e-3) / 1e9, "peak": peak * world,
                             "peak_source": peak_src + f" x {world} GPUs", "unit": "GB/s",
                             "frac": None, "traffic": None,
                             "note": "8d convention bytes / time; with lazy Adam the step moves fewer bytes than the "
                                     "convention, so no fraction is claimed here (see the 1-GPU line)"},
                "nvlink": r["nvl"], "e2e": r["e2e"], "gpu_launches": int(r["launches"]), "clocks": r["clk"],
                "final_loss": r["loss"], "rank0_phase_ms": r["phases"], "parity_vs_1gpu": parity}
        if legs:
            line["configs"] = legs
        print(json.dumps(line), flush=True)
    dist.barrier()
    dist.destroy_process_group()

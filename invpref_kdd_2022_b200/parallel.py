"""Multi-GPU InvPref: one process per GPU (``torch.distributed``, NCCL over NVLink/NVSwitch).

The reference is single-GPU; this layer is new (SURVEY.md §8e).  Interactions of every global batch are
partitioned across ranks -- the loss is a mean over the global batch, so any partition is semantically
free once every 1/B factor uses the GLOBAL batch size (``invpref_hyper.global_batch``).

``ReplicatedTrainer``  dataset-scale tables (C1-C4): tables replicated, each rank takes a contiguous chunk
                       of the batch, exports its partial dense gradients, ONE all-reduce over the flat
                       gradient buffer (+ the six loss partial sums), then the same dense Adam everywhere.
``ShardedTrainer``     10M-user scale (C5): user rows and item rows are mod-sharded over the ranks together
                       with their Adam state.  An interaction is routed to the rank that owns its USER row,
                       so user rows never cross NVLink: the fused segment-reduce -> Adam runs locally on the
                       user shard.  Item rows are fetched from their owners per step (all-to-all of rows into
                       a compact per-batch cache; the routing is static per batch and built once), the
                       per-rank partial item gradients go back the same way, the owner adds them in rank
                       order (deterministic) and applies dense Adam to its item shard.  E / W / b are
                       replicated; their gradients and the loss partial sums are all-reduced (a few KB).

Every collective is issued by a small driver from a generator (`yield ("all_to_all", ...)`), so the same step
code runs under ``torch.distributed`` (``DistDriver``) and under ``SimDriver``, which runs G simulated ranks
in ONE process on one GPU -- that is how the 1-GPU test-suite checks the sharded arithmetic against the
single-GPU result without a multi-GPU box.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List

import torch

from . import _lib
from .engine import HotPath

SMALL = ("E", "W", "b")


# ================================ collectives =====================================================
class DistDriver:
    """Executes the collectives a step generator yields with torch.distributed (NCCL on GPU, gloo on CPU)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist, self.group = dist, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)

    def run(self, gen):
        dist = self.dist
        try:
            req = next(gen)
            while True:
                op = req[0]
                if op == "all_reduce":
                    dist.all_reduce(req[1], group=self.group)
                elif op == "all_to_all":
                    _, out, inp, out_splits, in_splits = req
                    self._a2a(out, inp, out_splits, in_splits)
                else:
                    raise ValueError(op)
                req = gen.send(None)
        except StopIteration as stop:
            return stop.value

    def _a2a(self, out, inp, out_splits, in_splits):
        dist = self.dist
        try:
            dist.all_to_all_single(out, inp, list(out_splits), list(in_splits), group=self.group)
        except RuntimeError:
            # gloo builds without alltoall: emulate with all_gather (host-side tests only)
            sizes = [torch.zeros(1, dtype=torch.int64) for _ in range(self.world)]
            dist.all_gather(sizes, torch.tensor([inp.shape[0]], dtype=torch.int64), group=self.group)
            mx = int(max(s.item() for s in sizes))
            pad = torch.zeros((mx,) + tuple(inp.shape[1:]), dtype=inp.dtype)
            pad[:inp.shape[0]] = inp
            bufs = [torch.zeros_like(pad) for _ in range(self.world)]
            dist.all_gather(bufs, pad, group=self.group)
            splits = [torch.zeros(self.world, dtype=torch.int64) for _ in range(self.world)]
            dist.all_gather(splits, torch.tensor(list(in_splits), dtype=torch.int64), group=self.group)
            o = 0
            for p in range(self.world):
                sp = splits[p].tolist()
                start = sum(sp[:self.rank])
                out[o:o + sp[self.rank]] = bufs[p][start:start + sp[self.rank]]
                o += sp[self.rank]


class LocalDriver:
    """world = 1: every collective is the identity (all_reduce) or a local copy (all_to_all).  Lets the sharded
    trainers run in a single process without a process group."""
    world, rank = 1, 0

    def run(self, gen):
        try:
            req = next(gen)
            while True:
                if req[0] == "all_to_all":
                    _, out, inp, _, _ = req
                    out.copy_(inp)
                elif req[0] != "all_reduce":
                    raise ValueError(req[0])
                req = gen.send(None)
        except StopIteration as stop:
            return stop.value


class SimDriver:
    """Runs the generators of G simulated ranks in lockstep inside one process (tests / debugging)."""

    def __init__(self, world):
        self.world = world

    def run_all(self, gens: List):
        G = self.world
        reqs, done, results = [None] * G, [False] * G, [None] * G
        for k in range(G):
            try:
                reqs[k] = next(gens[k])
            except StopIteration as stop:        # no collective at all (e.g. peer-memory fetch only)
                done[k], results[k] = True, stop.value
        if all(done):
            return results
        assert not any(done), "ranks finished at different points"
        while True:
            op = reqs[0][0]
            assert all(r[0] == op for r in reqs), "ranks diverged"
            if op == "all_reduce":
                tot = reqs[0][1].clone()
                for r in reqs[1:]:
                    tot += r[1]
                for r in reqs:
                    r[1].copy_(tot)
            elif op == "all_to_all":
                for dst in range(G):
                    _, out, _, out_splits, _ = reqs[dst]
                    o = 0
                    for src in range(G):
                        _, _, inp, _, in_splits = reqs[src]
                        start = sum(in_splits[:dst])
                        n = in_splits[dst]
                        assert n == out_splits[src]
                        out[o:o + n] = inp[start:start + n]
                        o += n
            for k in range(G):
                try:
                    reqs[k] = gens[k].send(None)
                except StopIteration as stop:
                    done[k], results[k] = True, stop.value
            if all(done):
                return results
            assert not any(done), "ranks finished at different points"


# ================================ replicated tables ===============================================
class ReplicatedTrainer:
    """Tables replicated; batch chunked over ranks; one all-reduce of the flat gradient per step."""

    def __init__(self, params: Dict[str, torch.Tensor], implicit, reg_only_embed, reg_env_embed, lr, rank, world):
        dev = params["Uinv"].device
        self.rank, self.world = rank, world
        sizes = [params[k].numel() for k in _lib.PARAM_FIELDS]
        pad = [(-n) % 4 for n in sizes]                       # keep every view 16-byte aligned
        total = sum(n + p for n, p in zip(sizes, pad))
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.gflat = torch.zeros(total + 8, dtype=torch.float32, device=dev)     # + six loss partial sums
        self.mflat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.vflat = torch.zeros(total, dtype=torch.float32, device=dev)
        self.params, self.grads = {}, {}
        o = 0
        for k, n, p in zip(_lib.PARAM_FIELDS, sizes, pad):
            self.flat[o:o + n].copy_(params[k].reshape(-1))
            self.params[k] = self.flat[o:o + n].view(params[k].shape)
            self.grads[k] = self.gflat[o:o + n].view(params[k].shape)
            o += n + p
        self.loss = self.gflat[total:total + 6]
        self.hot = HotPath(self.params, implicit, reg_only_embed, reg_env_embed, lr=lr)
        # every group is exported, so the step never touches per-tensor Adam state: Adam runs on the flat
        # buffers below (adam_dense); the library still wants valid pointers
        self.hot.m = self.grads
        self.hot.v = self.grads
        self.flags = _lib.EXPORT_USER_GRADS | _lib.EXPORT_ITEM_GRADS | _lib.EXPORT_SMALL_GRADS | \
            (0 if rank == 0 else _lib.SKIP_PARAM_REG)

    def chunk(self, lo, hi):
        """Contiguous chunk of the global batch rows [lo, hi) for this rank."""
        n = hi - lo
        per = (n + self.world - 1) // self.world
        a = min(lo + self.rank * per, hi)
        return a, min(a + per, hi)

    def step_gen(self, users, items, scores, envs, weights, global_batch, plan=None, **kw):
        """users..weights: this rank's chunk (may be empty).  Yields collectives; returns the loss tensor."""
        self.gflat.zero_()
        # hot.m / hot.v alias the gradient buffer: safe only while EVERY group is exported (the step then never
        # touches per-tensor Adam state)
        all_exported = _lib.EXPORT_USER_GRADS | _lib.EXPORT_ITEM_GRADS | _lib.EXPORT_SMALL_GRADS
        assert self.flags & all_exported == all_exported, "ReplicatedTrainer: m/v are aliased, every group must be exported"
        if users.numel() > 0:
            self.hot.train_step(users, items, scores, envs, weights, plan=plan, loss_out=self.loss,
                                grads_out=self.grads, global_batch=global_batch, flags=self.flags, **kw)
        else:
            self.hot.step += 1
        yield ("all_reduce", self.gflat)
        self.hot.adam_dense(self.flat, self.mflat, self.vflat, self.gflat[:self.flat.numel()])
        return self.loss


# ================================ row-sharded tables ==============================================
class ItemRoute:
    """Static routing of one local batch: which item rows this rank needs from which owner, and which of
    its own rows every peer needs.  Built once per batch (the batch slicing is fixed, utils.py:12-19)."""

    def __init__(self):
        self.slots = None          # int64 [b]   cache slot of every local interaction's item
        self.n_cache = 0           # rows in the cache (= unique items of the local batch)
        self.recv_splits = None    # list[G]     cache rows coming from each owner
        self.send_splits = None    # list[G]     rows of my shard going to each requester
        self.send_rows = None      # int64 [sum(send_splits)] owner-local row indices, grouped by requester
        # push exchange over peer memory (ShardedTrainer.enable_push).  Rows: a requester loads cache slot c from
        # owner slot_owner[c]'s shard (first fetch), and owners store their updated rows into the requesters' caches
        # at pos.  Gradients: owners keep a staging buffer laid out like send_rows (grouped by requester); a
        # requester stores the partial gradient of cache slot c into owner slot_owner[c]'s staging at push_index[c]
        self.slot_owner = None     # int32 [n_cache] owner rank of every cache slot
        self.want_rows = None      # int64 [n_cache] owner-local row of every cache slot
        self.peer_first = None     # list[G]     first slot, in requester p's cache, of the rows it wants from me
        self.pos = None            # int32 [G, I_loc] slot of my row j in rank p's row cache, or -1
        self.peer_off = None       # list[G]     first staging row, at owner o, of the block of rows I want from o
        self.push_index = None     # int32 [n_cache] row in the owner's staging buffer of every cache slot
        self.spos = None           # int32 [G, I_loc] row in MY staging buffer of rank p's partial for my row j, or -1
        self.n_stage = 0           # rows of my staging buffer in use (= len(send_rows))


def build_route_gen(items_global: torch.Tensor, world: int, route: ItemRoute):
    """Generator: builds `route` for the local interactions' GLOBAL item ids (collectives are yielded)."""
    dev = items_global.device
    uniq, inverse = torch.unique(items_global, sorted=True, return_inverse=True)
    owner = uniq % world
    order = torch.sort(owner, stable=True).indices               # cache order: grouped by owner, id ascending
    slot_of_uniq = torch.empty_like(order)
    slot_of_uniq[order] = torch.arange(order.numel(), device=dev)
    route.slots = slot_of_uniq[inverse].contiguous()
    route.n_cache = int(uniq.numel())
    counts = torch.bincount(owner, minlength=world)
    route.recv_splits = [int(c) for c in counts.tolist()]
    want_rows = (uniq[order] // world).contiguous()               # owner-local rows, in cache order
    send_counts = torch.zeros(world, dtype=torch.int64, device=dev)
    yield ("all_to_all", send_counts, counts.to(torch.int64), [1] * world, [1] * world)
    route.send_splits = [int(c) for c in send_counts.tolist()]
    route.send_rows = torch.empty(sum(route.send_splits), dtype=torch.int64, device=dev)
    yield ("all_to_all", route.send_rows, want_rows, route.send_splits, route.recv_splits)
    # where, in every requester's cache, the block of rows it wants from me starts (peer-memory exchange)
    route.slot_owner = owner[order].to(torch.int32).contiguous()
    route.want_rows = want_rows
    first = torch.cumsum(counts, 0) - counts                     # my cache: first slot of each owner's block
    peer_first = torch.zeros(world, dtype=torch.int64, device=dev)
    yield ("all_to_all", peer_first, first.to(torch.int64).contiguous(), [1] * world, [1] * world)
    route.peer_first = [int(c) for c in peer_first.tolist()]
    # push exchange: where, in every OWNER's staging buffer (laid out like its send_rows), my block starts
    send_off = torch.cumsum(send_counts, 0) - send_counts        # my staging: first row of each requester's block
    peer_off = torch.zeros(world, dtype=torch.int64, device=dev)
    yield ("all_to_all", peer_off, send_off.to(torch.int64).contiguous(), [1] * world, [1] * world)
    route.peer_off = [int(c) for c in peer_off.tolist()]
    slot = torch.arange(route.n_cache, device=dev)
    own = route.slot_owner.to(torch.int64)
    route.push_index = (peer_off[own] + slot - first[own]).to(torch.int32).contiguous()
    route.n_stage = int(route.send_rows.numel())
    return route


def build_slot_table(route: ItemRoute, world: int, n_local_rows: int, first) -> torch.Tensor:
    """t[p, j] = first[p] + k if my item row j is the k-th row rank p asked me for, -1 if rank p did not ask for it.
    ``first = route.peer_first``: the slot of row j in rank p's row cache (route.pos).  ``first[p] =
    sum(send_splits[:p])``: the row of my staging buffer, laid out like send_rows, that holds rank p's partial gradient
    of row j (route.spos)."""
    dev = route.send_rows.device
    tab = torch.full((world, max(n_local_rows, 1)), -1, dtype=torch.int32, device=dev)
    o = 0
    for p in range(world):
        n = route.send_splits[p]
        if n:
            tab[p, route.send_rows[o:o + n]] = (first[p] + torch.arange(n, device=dev)).to(torch.int32)
        o += n
    return tab


class SymmetricItemStorage:
    """Peer-visible storage of one rank: ONE torch symmetric-memory buffer with the same layout on every rank, so that
    a peer's section is `buffer_ptrs[rank] + offset`.  ``ShardedTrainer(store=...)`` takes its buffers from it.
    Raises if symmetric memory is unavailable."""

    def __init__(self, n_items, dim, world, cache_rows, device, group, stage_rows=0, sync_floats=0):
        """``stage_rows`` > 0: the sections of the push exchange -- the item shard [Iinv | Ienv], the peer-written row
        caches and the double-buffered gradient staging of that many rows.  ``sync_floats`` > 0: the slot / flag
        arrays of ``invpref_peer_allreduce`` (``ShardedTrainer.enable_peer_sync``) for vectors of up to that many
        floats.  Either may be absent."""
        import torch.distributed._symmetric_memory as symm
        rows_max = (n_items + world - 1) // world
        pad = lambda n: (n + 63) // 64 * 64                      # 256-byte aligned sections
        sizes = []
        self.stage_rows = int(stage_rows)
        if self.stage_rows:
            sizes += [("Iinv", pad(rows_max * dim)), ("Ienv", pad(rows_max * dim)),
                      ("cache0", pad(cache_rows * dim)), ("cache1", pad(cache_rows * dim))]
            sizes += [(f"stage{par}{t}", pad(self.stage_rows * dim)) for par in range(2) for t in range(2)]
        self.sync_floats = pad(int(sync_floats)) if sync_floats else 0
        if self.sync_floats:
            sizes += [("sync_slots", 2 * world * self.sync_floats), ("sync_flags", pad(world))]
        self.offsets, self.sizes, o = {}, dict(sizes), 0
        for k, n in sizes:
            self.offsets[k] = o
            o += n
        self.buf = symm.empty(o, dtype=torch.float32, device=device)
        self.buf.zero_()
        self.hdl = symm.rendezvous(self.buf, group)
        self.base = [int(p) for p in self.hdl.buffer_ptrs]
        if len(self.base) != world:
            raise RuntimeError("symmetric memory: unexpected number of peer buffers")

    def alloc(self, name, shape):
        n = 1
        for d in shape:
            n *= int(d)
        if n > self.sizes[name]:
            raise ValueError(f"symmetric memory section {name}: {tuple(shape)} does not fit")
        o = self.offsets[name]
        return self.buf[o:o + n].view(tuple(shape))

    def ptrs(self, name):
        return [b + 4 * self.offsets[name] for b in self.base]


class ShardedBatch:
    """One rank's share of one global batch, prepared once."""

    def __init__(self):
        self.sel = None       # int64 [b] positions inside the global batch (order preserved)
        self.users = None     # int64 [b] LOCAL user rows (u // G)
        self.route = ItemRoute()
        self.scores = None
        self.plan = None
        self.global_batch = 0


class ShardedTrainer:
    """User and item tables mod-sharded by row over `world` ranks (row r of rank g holds id r*world + g)."""

    def __init__(self, n_users, n_items, n_envs, dim, implicit, reg_only_embed, reg_env_embed, lr, rank, world,
                 device, cache_rows, init=None, seed=17373331, lazy=True, store=None, stage_rows=0):
        """``store``: a ``SymmetricItemStorage``.  With its push sections, the item shard, the row caches and the
        gradient staging live there (``stage_rows`` is then the store's) and the push exchange is wired
        (``enable_push``); with its sync arrays, ``enable_peer_sync`` is wired too.  Without a store every buffer is
        an ordinary device tensor: the NCCL exchange, or simulated ranks in one process, whose caller may wire
        ``enable_push`` to the other ranks' tensors (``stage_rows`` > 0)."""
        self.rank, self.world, self.dev = rank, world, device
        self.U, self.I, self.K, self.D = n_users, n_items, n_envs, dim
        self.U_loc = (n_users - rank + world - 1) // world
        self.I_loc = (n_items - rank + world - 1) // world
        self.cache_rows = max(int(cache_rows), 1)
        f32 = dict(dtype=torch.float32, device=device)
        # owned shards
        if init is not None:      # init: full tables (tests) -> take my rows
            uinv, uenv = init["Uinv"][rank::world].clone(), init["Uenv"][rank::world].clone()
            self.Iinv, self.Ienv = init["Iinv"][rank::world].clone(), init["Ienv"][rank::world].clone()
            small = [init[k].reshape(-1).clone() for k in SMALL]
        else:
            g = torch.Generator(device=device).manual_seed(seed + rank)
            uinv = torch.randn((self.U_loc, dim), generator=g, **f32) * 0.01
            uenv = torch.randn((self.U_loc, dim), generator=g, **f32) * 0.01
            self.Iinv = torch.randn((self.I_loc, dim), generator=g, **f32) * 0.01
            self.Ienv = torch.randn((self.I_loc, dim), generator=g, **f32) * 0.01
            g0 = torch.Generator(device=device).manual_seed(seed)          # replicated tensors: same on all ranks
            small = [torch.randn(n, generator=g0, **f32) * s for n, s in
                     ((n_envs * dim, 0.01), (n_envs * dim, 0.1), (n_envs, 0.1))]
        peer = store is not None and store.stage_rows > 0       # the push exchange's buffers live in the store
        if peer:
            self.Iinv = store.alloc("Iinv", self.Iinv.shape).copy_(self.Iinv)
            self.Ienv = store.alloc("Ienv", self.Ienv.shape).copy_(self.Ienv)
        self.mI = [torch.zeros_like(self.Iinv), torch.zeros_like(self.Ienv)]
        self.vI = [torch.zeros_like(self.Iinv), torch.zeros_like(self.Ienv)]
        self.gI = [torch.zeros_like(self.Iinv), torch.zeros_like(self.Ienv)]
        # replicated small tensors in one flat buffer [E | W | b], gradients + six loss sums likewise
        KD = n_envs * dim
        self.small = torch.cat(small)
        self.gsmall = torch.zeros(2 * KD + n_envs + 6, **f32)
        self.msmall, self.vsmall = torch.zeros_like(self.small), torch.zeros_like(self.small)
        views = lambda t: {"E": t[:KD].view(n_envs, dim), "W": t[KD:2 * KD].view(n_envs, dim),
                           "b": t[2 * KD:2 * KD + n_envs]}
        self.loss = self.gsmall[2 * KD + n_envs:]
        mk = (lambda name, shape: store.alloc(name, shape).zero_()) if peer else \
            (lambda name, shape: torch.zeros(shape, **f32))
        # per-batch item cache (what the local kernels see as "the item tables") and its gradient (read by the
        # collective path only: with the push exchange the item pass stores its partials into the owners' staging)
        self.cache = [mk(f"cache{t}", (self.cache_rows, dim)) for t in range(2)]
        self.gcache = [torch.zeros((self.cache_rows, dim), **f32) for _ in range(2)]
        # push exchange: double-buffered staging of the ranks' partial item gradients, [parity][table]
        self.stage_rows = store.stage_rows if store is not None else int(stage_rows)
        self.stage = None
        if self.stage_rows:
            self.stage = [[mk(f"stage{par}{t}", (self.stage_rows, dim)) for t in range(2)] for par in range(2)]
        params = {"Uinv": uinv, "Uenv": uenv, "Iinv": self.cache[0], "Ienv": self.cache[1]}
        params.update(views(self.small))
        # lazy: the local user shard uses lazy dense Adam (bit-identical, see HotPath), so there is no dense
        # sweep at all; otherwise the sweep runs on a side stream under the NVLink exchange
        self.lazy = bool(lazy)
        self.hot = HotPath(params, implicit, reg_only_embed, reg_env_embed, lr=lr, lazy=self.lazy)
        self.hot.m = {"Uinv": torch.zeros_like(uinv), "Uenv": torch.zeros_like(uenv), "Iinv": self.cache[0],
                      "Ienv": self.cache[1]}
        self.hot.v = {"Uinv": torch.zeros_like(uinv), "Uenv": torch.zeros_like(uenv), "Iinv": self.cache[0],
                      "Ienv": self.cache[1]}
        self.hot.m.update(views(self.msmall))
        self.hot.v.update(views(self.vsmall))
        self.grads = {"Uinv": uinv, "Uenv": uenv, "Iinv": self.gcache[0], "Ienv": self.gcache[1]}   # U*: unused
        self.grads.update(views(self.gsmall))
        self.flags = _lib.EXPORT_ITEM_GRADS | _lib.EXPORT_SMALL_GRADS | (0 if rank == 0 else _lib.SKIP_PARAM_REG)
        self.send_buf = None
        self.recv_g = None
        self._fetched = None                      # batch whose item rows are currently in the cache
        self.side = torch.cuda.Stream(device=device)
        self.phase_events = None                  # set to [] to record (name, event) marks per step (bench)
        self.push = None                          # push exchange state once enable_push() ran
        self.bar = torch.zeros(1, **f32)          # payload of the barrier all-reduce (peer-memory mode)
        self.sync = None                          # peer-memory all-reduce / barrier state once enable_peer_sync() ran
        self.store = store                        # the mapped buffer outlives every pointer into it
        if peer:
            self.enable_push([store.ptrs("Iinv"), store.ptrs("Ienv")],
                             [[store.ptrs(f"stage{par}{t}") for t in range(2)] for par in range(2)],
                             [store.ptrs(f"cache{t}") for t in range(2)])
        if store is not None and store.sync_floats:
            self.enable_peer_sync(store.ptrs("sync_slots"), store.ptrs("sync_flags"), store.sync_floats)

    def enable_push(self, table_ptrs, stage_ptrs, cache_ptrs):
        """Push exchange over peer memory (NVLink stores instead of NCCL all-to-alls): ``table_ptrs[t][rank]`` /
        ``stage_ptrs[parity][t][rank]`` / ``cache_ptrs[t][rank]`` = device address IN THIS PROCESS of rank `rank`'s
        shard / staging buffer / row cache of item table t (own rank included).  The item pass stores its partial
        gradients straight into the owners' staging buffers and the owners, after Adam, store the updated rows into
        the requesters' caches for the next batch.  The shards are read only where no owner has pushed the rows: the
        first fetch of a loop or epoch and cluster_gen."""
        G = self.world
        assert self.stage is not None
        flat = lambda ptrs: [int(x) for t in range(2) for x in ptrs[t]]
        assert all(len(flat(p)) == 2 * G for p in [table_ptrs, cache_ptrs] + list(stage_ptrs))
        self.push = {"tables": (C.c_void_p * (2 * G))(*flat(table_ptrs)),
                     "base": [torch.tensor(flat(stage_ptrs[par]), dtype=torch.int64, device=self.dev)
                              for par in range(2)],
                     "caches": (C.c_void_p * (2 * G))(*flat(cache_ptrs)), "step": 0}

    def enable_peer_sync(self, slot_ptrs, flag_ptrs, n_max):
        """The two rank-wide synchronisation points of a step (the all-reduce of the E / W / b gradients + loss sums,
        and the barrier after the owners' row pushes) as ``invpref_peer_allreduce`` over peer memory instead of NCCL
        all-reduces: ``slot_ptrs[rank]`` / ``flag_ptrs[rank]`` = device address IN THIS PROCESS of rank `rank`'s slot
        array (2 * world * n_max floats) and flag array (world uint32, zeroed, and a barrier passed since), own rank
        included.  The sum runs in rank order on every rank.  With it the step issues no NCCL call at all."""
        G = self.world
        assert len(slot_ptrs) == len(flag_ptrs) == G and n_max >= self.gsmall.numel()
        self.sync = {"slots": (C.c_void_p * G)(*[int(x) for x in slot_ptrs]),
                     "flags": (C.c_void_p * G)(*[int(x) for x in flag_ptrs]), "n_max": int(n_max),
                     "ctr": torch.zeros(1, dtype=torch.int32, device=self.dev),
                     "status": torch.zeros(1, dtype=torch.int32, device=self.dev)}

    def _peer_allreduce(self, t):
        """In-place sum of `t` (or, with None, just the barrier) over the ranks through peer memory."""
        sy = self.sync
        _lib.check(self.hot.lib.invpref_peer_allreduce(
            _lib.ptr(t) if t is not None else None, t.numel() if t is not None else 0, sy["n_max"], self.world,
            self.rank, sy["slots"], sy["flags"], _lib.ptr(sy["ctr"], torch.int32), _lib.ptr(sy["status"], torch.int32),
            _lib.stream_ptr()), "peer_allreduce")

    def check_sync(self):
        """Raises if a peer failed to arrive at a peer-memory synchronisation point (synchronises the device)."""
        if self.sync is not None and int(self.sync["status"].item()) != 0:
            raise RuntimeError("invpref_peer_allreduce: a rank did not arrive within the spin limit")

    def _mark(self, name):
        if self.phase_events is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.phase_events.append((name, ev))

    # ---- setup -------------------------------------------------------------------------------------
    def prepare_gen(self, users_g, items_g, scores_g):
        """Generator: this rank's share of a global batch (GLOBAL ids, full batch given on every rank)."""
        sb = ShardedBatch()
        sb.global_batch = int(users_g.numel())
        sb.sel = torch.nonzero(users_g % self.world == self.rank).reshape(-1)
        sb.users = (users_g[sb.sel] // self.world).contiguous()
        sb.scores = scores_g[sb.sel].contiguous()
        yield from build_route_gen(items_g[sb.sel], self.world, sb.route)
        if sb.route.n_cache > self.cache_rows:
            raise RuntimeError(f"item cache too small: {sb.route.n_cache} > {self.cache_rows}")
        if self.stage_rows and sb.route.n_stage > self.stage_rows:
            raise RuntimeError(f"gradient staging too small: {sb.route.n_stage} > {self.stage_rows}")
        sb.plan = self.hot.new_plan(sb.users, sb.route.slots)      # also for an empty share (sweep needs it)
        return sb

    def _buf(self, name, rows):
        cur = getattr(self, name)
        if cur is None or cur[0].shape[0] < rows:
            cur = [torch.empty((max(rows, 1), self.D), dtype=torch.float32, device=self.dev) for _ in range(2)]
            setattr(self, name, cur)
        return cur

    def _gather(self, table, rows, out):
        _lib.check(self.hot.lib.invpref_gather_rows(_lib.ptr(table), _lib.ptr(rows), rows.numel(), self.D,
                                                    _lib.ptr(out), _lib.stream_ptr()), "gather_rows")

    def _scatter_add(self, src, rows, table):
        _lib.check(self.hot.lib.invpref_scatter_add_rows(_lib.ptr(src), _lib.ptr(rows), rows.numel(), self.D,
                                                         _lib.ptr(table), _lib.stream_ptr()), "scatter_add_rows")

    def fetch_gen(self, sb: ShardedBatch):
        """All-to-all of item rows: owners pack the requested rows, requesters receive them as the cache."""
        r = sb.route
        if self.push is not None:
            # one kernel: every cache row is loaded straight from its owner's shard (the caller has made sure,
            # with a barrier, that all owners finished their last update)
            if r.n_cache:
                _lib.check(self.hot.lib.invpref_fetch_rows_p2p(
                    self.push["tables"], self.world, _lib.ptr(r.slot_owner, torch.int32),
                    _lib.ptr(r.want_rows, torch.int64), r.n_cache, self.D, _lib.ptr(self.cache[0]), _lib.ptr(self.cache[1]), _lib.stream_ptr()),
                    "fetch_rows_p2p")
            return
        ns = int(r.send_rows.numel())
        send = self._buf("send_buf", ns)
        for t, (table, buf) in enumerate(zip((self.Iinv, self.Ienv), send)):
            if ns:
                self._gather(table, r.send_rows, buf)
            yield ("all_to_all", self.cache[t][:r.n_cache], buf[:ns], r.recv_splits, r.send_splits)

    # ---- train step -----------------------------------------------------------------------------------
    def step_gen(self, sb: ShardedBatch, envs, weights, next_sb: ShardedBatch = None, dyn=None, **kw):
        """envs / weights: this rank's slices (aligned with sb.sel).  Returns the loss tensor (global values
        after the all-reduce).  ``dyn``: device address of this step's ``invpref_dyn`` record: every kernel of the step
        reads Adam's bias corrections, alpha and the step number from it (CUDA-graph capture of an epoch; push
        exchange with ``enable_peer_sync`` only, where the step issues nothing but library kernels).

        Overlap: the dense Adam sweep over the local user rows without a gradient (the largest local kernel,
        pure HBM streaming) runs on a side stream while the main stream exchanges the item gradients over
        NVLink, updates the item shard and the replicated tensors, and already fetches the item rows of
        `next_sb` (the batch order is fixed, so the next batch is known)."""
        r = sb.route
        self._mark("start")
        if self._fetched is not sb:
            yield from self.fetch_gen(sb)
        self._fetched = None
        self._mark("fetch")
        self.gsmall.zero_()
        main = torch.cuda.current_stream()
        push, par = None, 0
        if self.push is not None:
            par = self.push["step"] & 1
            if r.n_cache:
                push = _lib.Push(_lib.ptr(self.push["base"][par], torch.int64), _lib.ptr(r.slot_owner, torch.int32),
                                 _lib.ptr(r.push_index, torch.int32), self.world, 0)
        if self.lazy:
            if sb.users.numel() > 0:
                self.hot.train_step(sb.users, r.slots, sb.scores, envs, weights, plan=sb.plan, loss_out=self.loss,
                                    grads_out=self.grads, global_batch=sb.global_batch, flags=self.flags, push=push,
                                    dyn=dyn, **kw)
            else:   # no interaction routed here: the local rows just fall one more step behind
                assert dyn is None, "graph capture needs a non-empty share of every batch"
                self.hot._ensure_state(())
                self.hot._ensure_lazy()
                self.hot.step += 1
                self.hot._dirty = True
                self.hot.write_sched()
            self._mark("local_step")
        else:
            self.hot._ensure_state(("Uinv", "Uenv"))
            if sb.users.numel() > 0:
                self.hot.train_step(sb.users, r.slots, sb.scores, envs, weights, plan=sb.plan, loss_out=self.loss,
                                    grads_out=self.grads, global_batch=sb.global_batch,
                                    flags=self.flags | _lib.DEFER_USER_SWEEP, push=push, **kw)
            else:       # no interaction routed here: every local user row still moves by momentum
                self.hot.step += 1
                for k in ("Uinv", "Uenv"):
                    self.hot.params[k], self.hot.shadow[k] = self.hot.shadow[k], self.hot.params[k]
            self._mark("local_step")
            self.side.wait_stream(main)
            with torch.cuda.stream(self.side):
                self.hot.user_sweep(sb.plan, sb.users.numel())
        if self.push is not None:
            # PUSH exchange.  The item pass above already stored this rank's partial item gradients into the owners'
            # staging buffers (parity `par`).  Barrier 1 = the all-reduce of the replicated tensors' gradients: when
            # it returns every rank's item pass -- and with it every posted NVLink write -- has completed.  Then ONE
            # kernel per rank reduces its rows from LOCAL memory in rank order, applies Adam and stores the updated
            # rows into the requesters' caches for the next batch.
            if self.sync is not None:
                self._peer_allreduce(self.gsmall)
            else:
                yield ("all_reduce", self.gsmall)
            self._mark("grad_a2a")
            if r.spos is None:
                r.spos = build_slot_table(r, self.world, self.I_loc,
                                          [sum(r.send_splits[:p]) for p in range(self.world)])
            npos = None
            if next_sb is not None:
                nr = next_sb.route
                if nr.pos is None:
                    nr.pos = build_slot_table(nr, self.world, self.I_loc, nr.peer_first)
                npos = nr.pos
            hyper = _lib.Hyper(0, 0, 0, 0, 0, 0, self.hot.lr, self.hot.betas[0], self.hot.betas[1], self.hot.eps,
                               int(self.hot.step), 0, 0, 0, 0, 0, dyn)
            _lib.check(self.hot.lib.invpref_owner_adam_push(
                _lib.ptr(self.Iinv), _lib.ptr(self.Ienv), _lib.ptr(self.mI[0]), _lib.ptr(self.mI[1]),
                _lib.ptr(self.vI[0]), _lib.ptr(self.vI[1]), self.I_loc, self.D, self.world,
                _lib.ptr(self.stage[par][0]), _lib.ptr(self.stage[par][1]), _lib.ptr(r.spos, torch.int32),
                self.push["caches"] if npos is not None else None,
                _lib.ptr(npos, torch.int32) if npos is not None else None, C.byref(hyper), _lib.stream_ptr()),
                "owner_adam_push")
            self._mark("item_adam")
            n_small = self.small.numel()
            self.hot.adam_dense(self.small, self.msmall, self.vsmall, self.gsmall[:n_small], dyn=dyn)
            # Barrier 2: every owner's pushes have landed before anyone's next local step reads its cache.  (The
            # staging buffers need no barrier of their own: they alternate, and barrier 1 of the NEXT step already
            # orders this step's owner kernels before the item pass of the step after it.)
            if self.sync is not None:
                self._peer_allreduce(None)
            else:
                yield ("all_reduce", self.bar)
            self._mark("small")
            if next_sb is not None:
                self._fetched = next_sb
            self._mark("prefetch_next")
            if not self.lazy:                # the side stream carries the dense user sweep only
                main.wait_stream(self.side)
            self._mark("sweep_wait")
            self.push["step"] += 1
            return self.loss
        # partial item gradients back to the owners (reverse routing)
        ns = int(r.send_rows.numel())
        recv = self._buf("recv_g", ns)
        for t in range(2):
            yield ("all_to_all", recv[t][:ns], self.gcache[t][:r.n_cache], r.send_splits, r.recv_splits)
        self._mark("grad_a2a")
        # owner: add the peers' partials in rank order (deterministic), then dense Adam on the shard
        for t, (m, v, table) in enumerate(zip(self.mI, self.vI, (self.Iinv, self.Ienv))):
            self.gI[t].zero_()
            o = 0
            for p in range(self.world):
                n = r.send_splits[p]
                if n:
                    self._scatter_add(recv[t][o:o + n], r.send_rows[o:o + n], self.gI[t])
                o += n
            self.hot.adam_dense(table.view(-1), m.view(-1), v.view(-1), self.gI[t].view(-1))
        self._mark("item_adam")
        # replicated E / W / b: all-reduce of a few KB (gradients + loss partial sums), same Adam on every rank
        if self.sync is not None:
            self._peer_allreduce(self.gsmall)
        else:
            yield ("all_reduce", self.gsmall)
        n_small = self.small.numel()
        self.hot.adam_dense(self.small, self.msmall, self.vsmall, self.gsmall[:n_small])
        self._mark("small")
        if next_sb is not None:       # the cache is free again: fetch the next batch's item rows now
            yield from self.fetch_gen(next_sb)
            self._fetched = next_sb
        self._mark("prefetch_next")
        main.wait_stream(self.side)
        self._mark("sweep_wait")
        return self.loss

    # ---- EM re-assignment -------------------------------------------------------------------------------
    def flush(self):
        """Lazy mode: bring the local user shard up to the last completed step."""
        self.hot.flush()

    def cluster_gen(self, sb: ShardedBatch, perm_idx, eps_table, old_envs):
        """train.py:846-879 on this rank's share of a batch; hist / diff are all-reduced by the caller."""
        yield from self.fetch_gen(sb)
        self._fetched = None
        if sb.users.numel() == 0:
            z = torch.zeros(0, dtype=torch.int64, device=self.dev)
            return z, torch.zeros(self.K, dtype=torch.int64, device=self.dev), torch.zeros(1, dtype=torch.int64,
                                                                                           device=self.dev)
        return self.hot.cluster(sb.users, sb.route.slots, sb.scores, perm_idx, eps_table, old_envs, trusted=True)

    # ---- inspection (tests) -----------------------------------------------------------------------------
    def local_tables(self):
        self.hot.flush()
        return {"Uinv": self.hot.params["Uinv"], "Uenv": self.hot.params["Uenv"], "Iinv": self.Iinv,
                "Ienv": self.Ienv, "E": self.hot.params["E"], "W": self.hot.params["W"], "b": self.hot.params["b"]}

"""Multi-GPU InvPref trainers behind the reference's trainer API (one process per GPU, ``torch.distributed``).

``ShardedExplicitTrainManager`` / ``ShardedImplicitTrainManager`` keep the method surface of the reference's
``ExplicitTrainManager`` / ``ImplicitTrainManager`` (train.py:693-1019 / 16-342) -- ``train()``, ``train_a_epoch()``,
``cluster()``, ``stat_envs()``, the loss dictionaries and the return triple of ``train()`` -- on tables that are
row-sharded over the ranks (``parallel.ShardedTrainer``: user and item rows mod-sharded with their Adam state, an
interaction handled by the rank that owns its user row, item rows / partial item gradients exchanged over NVLink peer
memory).  The reference is single-GPU, so what is kept is its semantics on the GLOBAL data:

  * global batch s is rows [s B, (s+1) B) of the training set, unshuffled (utils.py:12-19); every rank takes the rows
    of that slice whose user it owns (any partition of a batch is free: the losses are means over the global batch);
  * the initial environments and the per-cluster-batch tie-break indices are drawn from numpy's global stream exactly
    as train.py:711 / 870-871 do (every rank draws the same arrays from the same seed and keeps its share), so a run
    on G ranks assigns the same environments as the single-GPU trainer except for fp32 near-ties;
  * ``cluster()``: per-rank re-assignment of the local share, then ONE all-reduce of the K-bin histogram and the
    diff count (SURVEY.md 8e); ``stat_envs()``: class weights from the global histogram (train.py:945-957);
  * every rank returns the same (global) loss dictionaries and counts.

Each rank may be given only ITS share of the training set (``local_rows`` = global row indices of ``training_data``),
so no rank has to hold the whole interaction file; with ``local_rows=None`` the full set is given and filtered here.
"""
from __future__ import annotations

import itertools
import math

import numpy as np
import torch

from ._lib import LOSS_KEYS
from .npstream import device_randint
from .parallel import DistDriver, ShardedBatch, ShardedTrainer, build_route_gen
from .utils import _mean_merge_dict_func, merge_dict, transfer_loss_dict_to_line_str


class _ShardedInvPrefTrainManager:
    implicit = False

    def __init__(self, user_num: int, item_num: int, env_num: int, factor_num: int, training_data: torch.Tensor,
                 device: torch.device, batch_size: int, epochs: int, cluster_interval: int, evaluate_interval: int,
                 lr: float, invariant_coe: float, env_aware_coe: float, env_coe: float, L2_coe: float, L1_coe: float,
                 alpha: float = None, use_class_re_weight: bool = False, test_begin_epoch: int = 0,
                 begin_cluster_epoch: int = None, stop_cluster_epoch: int = None, cluster_use_random_sort: bool = True,
                 use_recommend_re_weight: bool = True, reg_only_embed: bool = False, reg_env_embed: bool = True,
                 evaluator=None, group=None, local_rows: torch.Tensor = None, total_rows: int = None,
                 init: dict = None, seed: int = 17373331, exchange: str = "push", lazy_adam: bool = True,
                 driver=None, rank: int = None, world: int = None, peer_sync: bool = True, use_graph: bool = True,
                 tie_break_rng: str = "numpy"):
        """Model arguments (``user_num .. factor_num``, ``reg_*``) are those of ``InvPrefExplicit/Implicit``
        (models.py:415-418): the sharded tables live in this object, not in an ``nn.Module``.  ``training_data``:
        int64 ``[n, 3]`` (user, item, score) -- the whole training set, or, with ``local_rows`` (their global row
        numbers, ascending) and ``total_rows``, only the rows whose user this rank owns.  ``init``: optional full
        tables (tests).  ``exchange``: "push" (peer memory, needs torch symmetric memory) | "nccl".
        ``peer_sync``: with the push exchange, also run the step's small all-reduce and barriers over peer
        memory (``invpref_peer_allreduce``) instead of NCCL.  ``use_graph``: with push + peer_sync (a step is then
        nothing but library kernels) every epoch after the first is replayed as ONE CUDA-graph launch per rank.
        ``driver`` / ``rank`` / ``world``: for simulated ranks (tests); default: torch.distributed.
        ``tie_break_rng``: "numpy" draws the initial environments and the tie-break rows from numpy's global stream on
        the host, "numpy_device" draws the same values on the GPU (npstream.py), one global batch at a time."""
        if tie_break_rng not in ("numpy", "numpy_device"):
            raise ValueError("tie_break_rng must be 'numpy' or 'numpy_device'")
        if exchange not in ("push", "nccl"):
            raise ValueError("exchange must be 'push' or 'nccl'")
        self.tie_break_rng = tie_break_rng
        if driver is None and world == 1:
            from .parallel import LocalDriver
            driver = LocalDriver()                                    # one rank: no process group needed
        self.drv = driver if driver is not None else DistDriver(group)
        self.rank = rank if rank is not None else self.drv.rank
        self.world = world if world is not None else self.drv.world
        if self.world == 1:
            exchange = "nccl"                                         # nothing to exchange: plain local copies
        self.device, self.group = device, group
        self.user_num, self.item_num, self.envs_num, self.factor_num = user_num, item_num, env_num, factor_num
        data = training_data.to(device)
        if local_rows is None:
            N = int(data.shape[0])
            rows = torch.nonzero(data[:, 0] % self.world == self.rank).reshape(-1)
            data = data[rows]
        else:
            N = int(total_rows)
            rows = local_rows.to(device)
            assert bool((data[:, 0] % self.world == self.rank).all()), "local share holds users of another rank"
        self.N, self.rows = N, rows                                   # global row numbers of the local share
        self.users_tensor = data[:, 0].contiguous()                   # GLOBAL ids of the local share
        self.items_tensor = data[:, 1].contiguous()
        self.scores_tensor = data[:, 2].float().contiguous()
        bounds = torch.arange(0, N + batch_size, batch_size, device=device).clamp_(max=N)
        self._lo = torch.searchsorted(rows, bounds).tolist()          # local slice of every global batch
        # train.py:711: the global draw, identical on every rank; the local share keeps its rows
        if tie_break_rng == "numpy_device":
            self.envs = torch.cat([self._global_draw(env_num, b, min(N, (b + 1) * batch_size) - b * batch_size,
                                                     batch_size) for b in range(len(self._lo) - 1)])
        else:
            envs_all = np.random.randint(0, self.envs_num, N)
            self.envs = torch.from_numpy(envs_all).to(device)[rows].contiguous()
        self.cluster_interval, self.evaluate_interval = cluster_interval, evaluate_interval
        self.batch_size, self.epochs, self.lr = batch_size, epochs, lr
        self.invariant_coe, self.env_aware_coe, self.env_coe = invariant_coe, env_aware_coe, env_coe
        self.L2_coe, self.L1_coe = L2_coe, L1_coe
        self.epoch_cnt = 0
        self.batch_num = math.ceil(N / batch_size)
        self.each_env_count = dict()
        if alpha is None:                                                                      # train.py:740-745
            self.alpha, self.update_alpha = 0., True
        else:
            self.alpha, self.update_alpha = alpha, False
        self.use_class_re_weight = use_class_re_weight
        self.use_recommend_re_weight = use_recommend_re_weight
        self.sample_weights = torch.zeros(rows.numel(), dtype=torch.float32, device=device)
        self.class_weights = torch.zeros(self.envs_num, dtype=torch.float32, device=device)
        self.test_begin_epoch = test_begin_epoch
        self.begin_cluster_epoch, self.stop_cluster_epoch = begin_cluster_epoch, stop_cluster_epoch
        base = torch.Tensor([1e-10 * (1e-1 ** idx) for idx in range(self.envs_num)])          # train.py:763-769
        self.eps_random_tensor = torch.Tensor(list(itertools.permutations(base))).to(device)
        self.cluster_use_random_sort = cluster_use_random_sort
        self.evaluator = evaluator
        # ---- the sharded engine ----
        per_rank = max(self._lo[b + 1] - self._lo[b] for b in range(self.batch_num))
        if driver is None and self.world > 1:
            # the symmetric-memory buffer must have the same layout (hence the same size) on every rank: size the
            # caches for the largest share any rank has of any batch
            import torch.distributed as dist
            t = torch.tensor([per_rank], dtype=torch.int64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
            per_rank = int(t.item())
        cache_rows = min(item_num, per_rank + 1024)
        stage_rows = min(2 * cache_rows + 1024, ((item_num + self.world - 1) // self.world) * self.world) \
            if exchange == "push" else 0
        self.exchange = exchange
        store = None
        if exchange == "push" and driver is None:
            from .parallel import SymmetricItemStorage
            import torch.distributed as dist
            store = SymmetricItemStorage(item_num, factor_num, self.world, cache_rows, device,
                                         group if group is not None else dist.group.WORLD, stage_rows=stage_rows,
                                         sync_floats=(2 * env_num * factor_num + env_num + 6) if peer_sync else 0)
        self.trainer = ShardedTrainer(user_num, item_num, env_num, factor_num, self.implicit, reg_only_embed,
                                      reg_env_embed, lr, self.rank, self.world, device, cache_rows=cache_rows, init=init,
                                      seed=seed, lazy=lazy_adam, store=store, stage_rows=stage_rows)
        if store is not None:
            torch.cuda.synchronize()
            dist.barrier(group)
        self.engine = self.trainer.hot
        self.engine.check_ids(self.users_tensor // self.world, None, self.envs, sync=False)
        bad = torch.tensor([int(self.items_tensor.numel() and (int(self.items_tensor.max()) >= item_num or
                                                               int(self.items_tensor.min()) < 0))], device=device)
        self.engine.raise_if_bad_ids()
        if int(bad.item()):
            raise IndexError("index out of range in self: item id outside its embedding table")
        self._batches = None
        self.use_graph = bool(use_graph)
        self._graph = None
        self._loss_rows = None

    # ---- setup: this rank's share of every global batch, routed and planned once (the slicing is fixed) ----
    def _prepare(self):
        if self._batches is not None:
            return
        tr, out = self.trainer, []
        for b in range(self.batch_num):
            lo, hi = self._lo[b], self._lo[b + 1]
            sb = ShardedBatch()
            sb.global_batch = min(self.batch_size, self.N - b * self.batch_size)
            sb.sel = torch.arange(lo, hi, device=self.device)         # positions inside the LOCAL share
            sb.users = (self.users_tensor[lo:hi] // self.world).contiguous()
            sb.scores = self.scores_tensor[lo:hi]
            self.drv.run(build_route_gen(self.items_tensor[lo:hi], self.world, sb.route))
            if sb.route.n_cache > tr.cache_rows:
                raise RuntimeError(f"item cache too small: {sb.route.n_cache} > {tr.cache_rows}")
            if tr.stage_rows and sb.route.n_stage > tr.stage_rows:
                raise RuntimeError(f"gradient staging too small: {sb.route.n_stage} > {tr.stage_rows}")
            sb.plan = tr.hot.new_plan(sb.users, sb.route.slots)
            out.append(sb)
        self._batches = out

    def _all_reduce(self, t):
        def gen():
            yield ("all_reduce", t)
        self.drv.run(gen())
        return t

    # ---- train ------------------------------------------------------------------------------------------
    def _alpha_at(self, b: int) -> float:
        if self.update_alpha:                                                     # train.py:891-894
            p = float(b + (self.epoch_cnt + 1) * self.batch_num) / float((self.epoch_cnt + 1) * self.batch_num)
            self.alpha = 2. / (1. + np.exp(-10. * p)) - 1.
        return self.alpha

    def _loss_kw(self):
        return dict(c_inv=self.invariant_coe, c_ea=self.env_aware_coe, c_env=self.env_coe, c_L2=self.L2_coe,
                    c_L1=self.L1_coe, use_class_rw=self.use_class_re_weight, use_rec_rw=self.use_recommend_re_weight)

    def _graph_epoch(self) -> bool:
        """One epoch as ONE CUDA-graph launch per rank (the sharded twin of train.py's ``_graph_epoch``).  Applies to
        the push exchange with peer-memory synchronisation, where a step is a fixed sequence of library kernels on
        fixed buffers -- item pass with NVLink pushes, ``invpref_peer_allreduce``, owner reduce + Adam + row push,
        Adam on E / W / b, ``invpref_peer_allreduce`` -- and what changes between epochs (Adam's bias corrections,
        alpha, the step number, the synchronisation sequence number) is read from device memory."""
        tr, n = self.trainer, self.batch_num
        if not (self.use_graph and self.epoch_cnt >= 1 and tr.sync is not None and tr.push is not None and tr.lazy
                and tr.hot.m is not None and n <= 256 and all(sb.users.numel() > 0 for sb in self._batches)):
            return False
        from .engine import StepGraph
        if self._graph is None:
            self._graph = StepGraph(tr.hot, n)
            self._g_envs = torch.empty_like(self.envs)
            self._g_sw = torch.empty_like(self.sample_weights)
        g = self._graph
        tr.hot.reserve_steps(n)
        g.valid()
        main = torch.cuda.current_stream()
        g.stream.wait_stream(main)
        with torch.cuda.stream(g.stream):
            self._g_envs.copy_(self.envs)              # cluster() / stat_envs() re-bind these: stable copies
            self._g_sw.copy_(self.sample_weights)
            for b in range(n):
                g.fill(b, tr.hot.step + 1 + b, self._alpha_at(b))
            g.upload()
            key = tr.push["step"] & 1                  # which staging buffer the first step of the epoch uses
            if key not in g.handles:
                saved = (tr.hot.host_state(), tr.push["step"], tr._fetched)
                kw = self._loss_kw()

                def issue():
                    for b, sb in enumerate(self._batches):
                        lo, hi = self._lo[b], self._lo[b + 1]
                        nxt = self._batches[b + 1] if b + 1 < n else None
                        loss = self.drv.run(tr.step_gen(sb, self._g_envs[lo:hi], self._g_sw[lo:hi], next_sb=nxt,
                                                        alpha=0.0, dyn=g.record_ptr(b), **kw))
                        self._loss_rows[b].copy_(loss)
                    tr.hot.flush(dyn=g.record_ptr(n - 1))

                try:
                    g.capture(key, issue)
                finally:                               # capture records, it does not run: undo the host bookkeeping
                    tr.hot.restore_host_state(saved[0])
                    tr.push["step"], tr._fetched = saved[1], saved[2]
            g.launch(key)
            tr.hot.step += n                           # (no buffer swaps here: user tables in place, item rows exported)
            tr.hot._dirty = False                      # the captured epoch ends with the flush
            tr.push["step"] += n
            tr._fetched = None
        main.wait_stream(g.stream)
        return True

    def train_a_epoch(self) -> dict:
        """train.py:881-910 on the global batches; returns the same mean loss dictionary on every rank."""
        self._prepare()
        tr = self.trainer
        if self._loss_rows is None:
            self._loss_rows = torch.zeros((self.batch_num, 6), dtype=torch.float32, device=self.device)
        rows = self._loss_rows
        if not self._graph_epoch():
            kw = self._loss_kw()
            for b, sb in enumerate(self._batches):
                alpha = self._alpha_at(b)
                lo, hi = self._lo[b], self._lo[b + 1]
                nxt = self._batches[b + 1] if b + 1 < self.batch_num else None
                loss = self.drv.run(tr.step_gen(sb, self.envs[lo:hi], self.sample_weights[lo:hi], next_sb=nxt,
                                                alpha=alpha, **kw))
                rows[b].copy_(loss)
            tr.flush()
        self.epoch_cnt += 1
        vals = rows.cpu().tolist()
        tr.check_sync()
        return merge_dict([dict(zip(LOSS_KEYS, r)) for r in vals], _mean_merge_dict_func)

    # ---- EM re-assignment ---------------------------------------------------------------------------------
    def cluster(self) -> int:
        """train.py:912-936: every rank re-assigns its share; ONE all-reduce of [K-bin histogram | diff]."""
        self._prepare()
        tr = self.trainer
        tr.flush()
        if tr.store is not None:
            import torch.distributed as dist
            torch.cuda.synchronize()
            dist.barrier(self.group)          # every owner's rows are final before anyone fetches them
        new_envs = torch.empty_like(self.envs)
        acc = torch.zeros(self.envs_num + 1, dtype=torch.int64, device=self.device)
        for b, sb in enumerate(self._batches):
            lo, hi = self._lo[b], self._lo[b + 1]
            perm = None
            if self.cluster_use_random_sort and self.tie_break_rng == "numpy_device":
                perm = self._global_draw(self.eps_random_tensor.shape[0], b, sb.global_batch, self.batch_size)
            elif self.cluster_use_random_sort:        # the global draw of train.py:870-871, this rank's rows of it
                idx = np.random.randint(0, self.eps_random_tensor.shape[0], sb.global_batch)
                g_lo = b * self.batch_size
                perm = torch.from_numpy(idx.astype(np.int64)).to(self.device)[self.rows[lo:hi] - g_lo].contiguous()
            nv, hist, diff = self.drv.run(tr.cluster_gen(sb, perm, self.eps_random_tensor if perm is not None else None,
                                                         self.envs[lo:hi].contiguous()))
            new_envs[lo:hi] = nv
            acc[:self.envs_num] += hist
            acc[self.envs_num] += diff.reshape(-1)[0]
        self._all_reduce(acc)
        self.envs = new_envs
        self._hist = acc[:self.envs_num].clone()
        return int(acc[self.envs_num].item())

    def _global_draw(self, high: int, b: int, count: int, batch_size: int) -> torch.Tensor:
        """np.random.randint(0, high, count) for global batch b, drawn on the device; this rank's rows of it."""
        d = device_randint(high, count, self.device)
        lo, hi = self._lo[b], self._lo[b + 1]
        return d[self.rows[lo:hi] - b * batch_size].contiguous()

    def stat_envs(self) -> dict:
        """train.py:945-957 with the GLOBAL histogram (one all-reduce of K counters)."""
        hist = self.engine.env_hist(self.envs) if self.envs.numel() else \
            torch.zeros(self.envs_num, dtype=torch.int64, device=self.device)
        self._all_reduce(hist)
        from . import _lib
        cw = torch.empty(self.envs_num, dtype=torch.float32, device=self.device)
        # class weights from the GLOBAL counts and the GLOBAL N (library arithmetic: double -> fp32 as train.py:950-955);
        # the sample weights of the local rows are a plain look-up
        _lib.check(self.engine.lib.invpref_stat_envs(None, self.N, self.envs_num, _lib.ptr(hist, torch.int64),
                                                     _lib.ptr(cw), None, _lib.stream_ptr()), "stat_envs")
        self.class_weights, self.sample_weights = cw, cw[self.envs].contiguous()
        return {k: int(c) for k, c in enumerate(hist.cpu().tolist())}

    def update_each_env_count(self):
        self.each_env_count.update(self.stat_envs())

    # ---- tables -----------------------------------------------------------------------------------------
    def gather_state_dict(self, dst: int = 0):
        """The full model tables on rank ``dst`` under the reference's state_dict keys (None elsewhere): what an
        evaluator or a checkpoint needs.  Collective: call it on every rank."""
        import torch.distributed as dist
        from .models import _PARAM_PATHS
        loc = self.trainer.local_tables()
        out = {}
        for k in ("Uinv", "Iinv", "Uenv", "Ienv"):
            n = self.user_num if k[0] == "U" else self.item_num
            per = (n + self.world - 1) // self.world
            pad = torch.zeros((per, self.factor_num), device=self.device)
            pad[:loc[k].shape[0]] = loc[k]
            bufs = [torch.zeros_like(pad) for _ in range(self.world)] if self.rank == dst else None
            dist.gather(pad, bufs, dst=dst, group=self.group)
            if self.rank == dst:
                full = torch.zeros((per * self.world, self.factor_num), device=self.device)
                for r in range(self.world):
                    full[r::self.world] = bufs[r]
                out[".".join(_PARAM_PATHS[k])] = full[:n]
        if self.rank != dst:
            return None
        for k in ("E", "W", "b"):
            out[".".join(_PARAM_PATHS[k])] = loc[k].clone()
        return out

    # ---- epoch loop (train.py:959-1019) ------------------------------------------------------------------
    def train(self, silent: bool = False, auto: bool = False):
        test_result_list, test_epoch_list = [], []
        cluster_diff_num_list, cluster_epoch_list, envs_cnt_list = [], [], []
        loss_result_list, train_epoch_index_list = [], []
        verbose = not silent and not auto and self.rank == 0

        def evaluate():
            if self.evaluator is None:
                return
            res = self.evaluator.evaluate()
            test_result_list.append(res)
            test_epoch_list.append(self.epoch_cnt)
            if verbose:
                print('test at epoch:', self.epoch_cnt)
                print(transfer_loss_dict_to_line_str(res))

        evaluate()
        self.stat_envs()
        while self.epoch_cnt < self.epochs:
            loss_dict = self.train_a_epoch()
            train_epoch_index_list.append(self.epoch_cnt)
            loss_result_list.append(loss_dict)
            if verbose:
                print('train epoch:', self.epoch_cnt)
                print(transfer_loss_dict_to_line_str(loss_dict))
            if (self.epoch_cnt % self.evaluate_interval) == 0 and self.epoch_cnt >= self.test_begin_epoch:
                evaluate()
            if (self.epoch_cnt % self.cluster_interval) == 0:
                window = (self.begin_cluster_epoch is None or self.begin_cluster_epoch <= self.epoch_cnt) \
                    and (self.stop_cluster_epoch is None or self.stop_cluster_epoch > self.epoch_cnt)
                diff_num = self.cluster() if window else 0
                cluster_diff_num_list.append(diff_num)
                envs_cnt = self.stat_envs()
                cluster_epoch_list.append(self.epoch_cnt)
                envs_cnt_list.append(envs_cnt)
                if verbose:
                    print('cluster at epoch:', self.epoch_cnt)
                    print('diff num:', diff_num)
                    print(transfer_loss_dict_to_line_str(envs_cnt))
        return (loss_result_list, train_epoch_index_list), \
               (test_result_list, test_epoch_list), \
               (cluster_diff_num_list, envs_cnt_list, cluster_epoch_list)


class ShardedExplicitTrainManager(_ShardedInvPrefTrainManager):
    """Multi-GPU counterpart of the reference's ExplicitTrainManager (train.py:693-1019)."""
    implicit = False


class ShardedImplicitTrainManager(_ShardedInvPrefTrainManager):
    """Multi-GPU counterpart of the reference's ImplicitTrainManager (train.py:16-342)."""
    implicit = True

"""InvPref trainers with the reference's constructor and method signatures (reference
``train.py:16-342`` ImplicitTrainManager, ``train.py:693-1019`` ExplicitTrainManager); every batch is
ONE call into ``libinvpref_b200.so`` instead of ~250 ATen ops, and ``cluster()`` is one kernel over the
whole dataset instead of K forwards per batch.

Kept from the reference, because results depend on them:
  * batches are the sequential, unshuffled slices of ``utils.mini_batch`` (utils.py:12-19);
  * the initial environments come from ``np.random.randint`` at construction (train.py:711) and the
    tie-break indices from one ``np.random.randint(0, K!, b)`` per cluster batch (train.py:870-871), drawn
    from numpy's global stream in the reference's order -- on the host, or with ``tie_break_rng="numpy_device"``
    the same values on the GPU (npstream.py);
  * alpha schedule (train.py:891-894), stat_envs weighting (train.py:945-957), loss-dict keys and the
    per-epoch ``np.mean`` of per-batch python floats (utils.py:181-183).
"""
from __future__ import annotations

import itertools
import math

import numpy as np
import torch

from ._lib import LOSS_KEYS
from .npstream import device_randint
from .utils import _mean_merge_dict_func, merge_dict, mini_batch, transfer_loss_dict_to_line_str


class _InvPrefTrainManager:
    implicit = False

    def __init__(
            self, model, evaluator, device: torch.device, training_data: torch.Tensor, batch_size: int,
            epochs: int, cluster_interval: int, evaluate_interval: int, lr: float,
            invariant_coe: float, env_aware_coe: float, env_coe: float, L2_coe: float, L1_coe: float,
            alpha: float = None, use_class_re_weight: bool = False, test_begin_epoch: int = 0,
            begin_cluster_epoch: int = None, stop_cluster_epoch: int = None, cluster_use_random_sort: bool = True,
            use_recommend_re_weight: bool = True, cache_plans: bool = True, lazy_adam: bool = True,
            use_graph: bool = True, plan_cache_bytes: int = 16 << 30, sorted_cluster: bool = False,
            tie_break_rng: str = "numpy"
    ):
        if tie_break_rng not in ("numpy", "device", "numpy_device"):
            raise ValueError("tie_break_rng must be 'numpy' (the reference's host stream, train.py:870-871), "
                             "'numpy_device' (the same stream drawn on the GPU) or 'device'")
        self.tie_break_rng = tie_break_rng
        self.model = model
        self.evaluator = evaluator
        self.envs_num: int = model.env_num
        self.device = device
        n = training_data.shape[0]
        # contiguous copies of the three columns (the reference keeps stride-3 views, train.py:708-710)
        self.users_tensor = training_data[:, 0].contiguous().to(device)
        self.items_tensor = training_data[:, 1].contiguous().to(device)
        self.scores_tensor = training_data[:, 2].float().contiguous().to(device)
        if tie_break_rng == "numpy_device":
            self.envs = device_randint(self.envs_num, n, device)                                 # train.py:711
        else:
            self.envs = torch.LongTensor(np.random.randint(0, self.envs_num, n)).to(device)   # train.py:711
        self.cluster_interval, self.evaluate_interval = cluster_interval, evaluate_interval
        self.batch_size, self.epochs = batch_size, epochs
        self.lr = lr
        self.invariant_coe, self.env_aware_coe, self.env_coe = invariant_coe, env_aware_coe, env_coe
        self.L2_coe, self.L1_coe = L2_coe, L1_coe
        self.epoch_cnt: int = 0
        self.batch_num = math.ceil(n / batch_size)
        self.each_env_count = dict()
        if alpha is None:                                                                      # train.py:740-745
            self.alpha, self.update_alpha = 0., True
        else:
            self.alpha, self.update_alpha = alpha, False
        self.use_class_re_weight = use_class_re_weight
        self.use_recommend_re_weight = use_recommend_re_weight
        self.sample_weights = torch.zeros(n, dtype=torch.float32, device=device)
        self.class_weights = torch.zeros(self.envs_num, dtype=torch.float32, device=device)
        self.test_begin_epoch = test_begin_epoch
        self.begin_cluster_epoch, self.stop_cluster_epoch = begin_cluster_epoch, stop_cluster_epoch
        self.eps_random_tensor = self._init_eps().to(device)
        self.cluster_use_random_sort = cluster_use_random_sort
        self.const_env_tensor_list = [torch.full((n,), k, dtype=torch.int64, device=device)
                                      for k in range(self.envs_num)]                           # train.py:758-761
        # fused engine bound to the model's parameter storages; holds the Adam state (train.py:718)
        # lazy_adam: user rows outside a batch are updated lazily (the same arithmetic as dense torch.optim.Adam; one-ulp
        # exceptions from FMA contraction, DESIGN.md); train_a_epoch flushes at the end of the epoch, train_a_batch after
        # every call
        self.engine = model.hot_path(lr=lr, lazy=lazy_adam)
        self.engine.lr = float(lr)
        # the reference's nn.Embedding raises IndexError on an id outside its table; validate the whole training
        # set once here (the kernels below then take these tensors as trusted)
        self.engine.check_ids(self.users_tensor, self.items_tensor, self.envs)
        self.optimizer = self.engine           # exposes .m / .v / .step (exp_avg, exp_avg_sq, step)
        self.cache_plans = cache_plans
        self._plans = {}
        # Plans are cached while they fit `plan_cache_bytes` (a plan is ~80 bytes per interaction: the 239 batches of a
        # 10^9-interaction epoch would take 79 GB).  Batches beyond the budget get their plan rebuilt every epoch into
        # one of two rotating buffers on a loader stream, one step ahead of the step that consumes it (a plan build is
        # a 2 x 32-bit radix sort of the batch: ~1 ms for 4 M interactions, hidden under the 4.6 ms step).
        self.plan_cache_bytes = int(plan_cache_bytes)
        self._plan_bytes_used = 0
        self._ring = None
        self._consumed_slot = None
        # cluster() walks the whole dataset; optionally over a user-sorted view (built once: ids never change) in which
        # the two user rows of consecutive samples come out of L2 instead of HBM (invpref_cluster_sorted; identical
        # results).  Off by default: measured on the B200 it moves fewer DRAM bytes but is SLOWER (4.9 vs 5.8 G samples/s
        # at 96 M samples) -- the scattered tie-break / old / new environment accesses through the permutation cost more
        # than the user rows save, and the unsorted kernel already runs at 0.95 of the HBM roofline.
        # train_a_batch (the reference's public per-batch call) leaves every parameter current, as torch.optim.Adam does:
        # with lazy Adam that is a sweep over the user rows that are behind.  Callers that drive their own batch loop
        # and read the tables only through this package (forward / predict / cluster / state_dict flush on demand) can
        # set this to False and keep the lazy saving.
        self.flush_after_batch = True
        self.sorted_cluster = bool(sorted_cluster)
        self._cl_view = None
        self._scratch_busy_on_main = False      # a plan was built on the main stream since the loader last synced
        self._loss_rows = None
        # CUDA-graph replay of the epoch (train.py:881-910 issues 3-31 steps per epoch on the dataset configs, every
        # one of them a fixed sequence of launches on fixed buffers): from the second epoch on, one graph launch per
        # epoch instead of ~10 launches + their host-side marshalling per step.  Bit-identical to the plain loop.
        self.use_graph = bool(use_graph) and cache_plans and self.batch_num <= 256
        self._graph = None
        self._g_envs = None
        self._g_sw = None

    def _init_eps(self) -> torch.Tensor:
        """train.py:763-769, same torch expression so the fp32 table is bit-identical."""
        base_eps = 1e-10
        eps_list = [base_eps * (1e-1 ** idx) for idx in range(self.envs_num)]
        temp = torch.Tensor(eps_list)
        return torch.Tensor(list(itertools.permutations(temp)))

    # ---- train ----------------------------------------------------------------------------------
    def _plan_for(self, key, users, items):
        if not self.cache_plans or key is None:
            return None
        plan = self._plans.get(key)
        if plan is None:
            nbytes = self.engine.plan_bytes(users.numel())
            if self._plan_bytes_used + nbytes > self.plan_cache_bytes:
                return self._streamed_plan(key)
            plan = self.engine.new_plan(users, items)
            self._scratch_busy_on_main = True
            self.engine.plan_status(plan, users.numel())       # IndexError on an out-of-range id (once per batch)
            self._plans[key] = plan
            self._plan_bytes_used += nbytes
        return plan

    # ---- plans that do not fit the cache: built one step ahead on a loader stream, two rotating buffers ----
    def _ring_state(self):
        if self._ring is None:
            nbytes = self.engine.plan_bytes(self.batch_size)
            self._ring = {"buf": [torch.empty(nbytes, dtype=torch.uint8, device=self.device) for _ in range(2)],
                          "ready": [torch.cuda.Event(), torch.cuda.Event()],
                          "consumed": [torch.cuda.Event(), torch.cuda.Event()],
                          "stream": torch.cuda.Stream(device=self.device), "holds": [None, None], "turn": 0}
            self.engine.workspace(self.batch_size)             # allocated before two streams share it
            self._scratch_busy_on_main = True
            for ev in self._ring["consumed"]:
                ev.record()
        return self._ring

    def _prefetch_plan(self, key):
        """Starts building the plan of batch `key` (if it is a streamed one) on the loader stream."""
        if not self.cache_plans or key >= self.batch_num or key in self._plans:
            return
        if self._plan_bytes_used + self.engine.plan_bytes(self.batch_size) <= self.plan_cache_bytes:
            return                                             # will be cached when its step comes
        r = self._ring_state()
        if key in r["holds"]:
            return
        slot = r["turn"]
        r["turn"] ^= 1
        lo = key * self.batch_size
        u, i = self.users_tensor[lo:lo + self.batch_size], self.items_tensor[lo:lo + self.batch_size]
        if self._scratch_busy_on_main:                         # the sort scratch was last used on the main stream
            r["stream"].wait_stream(torch.cuda.current_stream())
            self._scratch_busy_on_main = False
        with torch.cuda.stream(r["stream"]):
            r["stream"].wait_event(r["consumed"][slot])        # the step that last read this buffer is done
            self.engine.new_plan(u, i, out=r["buf"][slot])
            r["ready"][slot].record(r["stream"])
        r["holds"][slot] = key

    def _streamed_plan(self, key):
        r = self._ring_state()
        if key not in r["holds"]:
            self._prefetch_plan(key)
        slot = r["holds"].index(key)
        torch.cuda.current_stream().wait_event(r["ready"][slot])
        self._consumed_slot = slot
        return r["buf"][slot]

    def _check_engine(self):
        if self.model._hot is not self.engine:
            raise RuntimeError("the model's parameter storages were re-allocated (.to() / .float() / load into new "
                               "tensors) after this trainer was built: its Adam state belongs to the old storages; "
                               "move the model first, then construct the trainer")

    def _step(self, users, items, scores, envs, weights, alpha, loss_out=None, plan_key=None):
        self._check_engine()
        users, items, envs = users.contiguous(), items.contiguous(), envs.contiguous()
        assert users.shape == items.shape == scores.shape == envs.shape          # train.py:789-790
        return self.engine.train_step(
            users, items, scores.contiguous(), envs, weights.contiguous() if weights is not None else None,
            c_inv=self.invariant_coe, c_ea=self.env_aware_coe, c_env=self.env_coe, c_L2=self.L2_coe,
            c_L1=self.L1_coe, alpha=alpha, use_class_rw=self.use_class_re_weight,
            use_rec_rw=self.use_recommend_re_weight, plan=self._plan_for(plan_key, users, items), loss_out=loss_out)

    def train_a_batch(self, batch_users_tensor, batch_items_tensor, batch_scores_tensor, batch_envs_tensor,
                      batch_sample_weights, alpha) -> dict:
        """train.py:771-844.  One fused step; returns the six losses as python floats (one sync)."""
        self.engine.check_ids(batch_users_tensor.contiguous(), batch_items_tensor.contiguous(),
                              batch_envs_tensor.contiguous(), sync=False)
        out = self._step(batch_users_tensor, batch_items_tensor, batch_scores_tensor, batch_envs_tensor,
                         batch_sample_weights, alpha)
        if self.flush_after_batch:
            self.engine.flush()
        vals = out.cpu().tolist()
        self.engine.raise_if_bad_ids()
        return dict(zip(LOSS_KEYS, vals))

    def _alpha_at(self, batch_index: int) -> float:
        if self.update_alpha:                                                     # train.py:891-894
            p = float(batch_index + (self.epoch_cnt + 1) * self.batch_num) / float(
                (self.epoch_cnt + 1) * self.batch_num)
            self.alpha = 2. / (1. + np.exp(-10. * p)) - 1.
        return self.alpha

    def _graph_epoch(self) -> bool:
        """One epoch as ONE CUDA-graph launch.  Returns False (nothing done) when the graph path does not apply yet:
        the first epoch runs launch by launch (it builds and validates the plans and allocates every buffer)."""
        eng, n = self.engine, self.batch_num
        if not (self.use_graph and self.epoch_cnt >= 1 and len(self._plans) == n and eng.m is not None):
            return False
        from .engine import StepGraph
        N = self.users_tensor.shape[0]
        if self._graph is None or self._graph.hot is not eng:
            self._graph = StepGraph(eng, n)
            self._g_envs = torch.empty(N, dtype=torch.int64, device=self.device)
            self._g_sw = torch.empty(N, dtype=torch.float32, device=self.device)
        g = self._graph
        eng.reserve_steps(n)
        g.valid()
        main = torch.cuda.current_stream()
        g.stream.wait_stream(main)
        with torch.cuda.stream(g.stream):
            # cluster() / stat_envs() re-bind self.envs / self.sample_weights to new tensors (as the reference does):
            # the captured kernels read these stable copies
            self._g_envs.copy_(self.envs)
            self._g_sw.copy_(self.sample_weights)
            for b in range(n):
                g.fill(b, eng.step + 1 + b, self._alpha_at(b))
            g.upload()
            key = eng.parity
            if key not in g.handles:
                saved = eng.host_state()

                def issue():
                    for b, (u, i, y, e, w) in enumerate(mini_batch(
                            self.batch_size, self.users_tensor, self.items_tensor, self.scores_tensor, self._g_envs,
                            self._g_sw)):
                        eng.train_step(u, i, y, e, w, c_inv=self.invariant_coe, c_ea=self.env_aware_coe,
                                       c_env=self.env_coe, c_L2=self.L2_coe, c_L1=self.L1_coe, alpha=0.0,
                                       use_class_rw=self.use_class_re_weight, use_rec_rw=self.use_recommend_re_weight,
                                       plan=self._plans[b], loss_out=self._loss_rows[b], dyn=g.record_ptr(b))
                    eng.flush(dyn=g.record_ptr(n - 1))

                try:
                    g.capture(key, issue)
                finally:
                    eng.restore_host_state(saved)     # capture records, it does not run: undo the host bookkeeping
            g.launch(key)
            eng.advance(n, flushed=True)
        main.wait_stream(g.stream)
        return True

    def train_a_epoch(self) -> dict:
        """train.py:881-910.  Losses stay on the device until the end of the epoch (one sync per epoch
        instead of six per batch); the returned dict is the same np.mean of per-batch floats."""
        self.model.train()
        self._check_engine()
        if self._loss_rows is None or self._loss_rows.shape[0] != self.batch_num:
            self._loss_rows = torch.zeros((self.batch_num, 6), dtype=torch.float32, device=self.device)
            if self._graph is not None:
                self._graph.drop()
        if self._graph_epoch():
            self.epoch_cnt += 1
            rows = self._loss_rows.cpu().tolist()
            return merge_dict([dict(zip(LOSS_KEYS, r)) for r in rows], _mean_merge_dict_func)
        for batch_index, (u, i, y, e, w) in enumerate(mini_batch(
                self.batch_size, self.users_tensor, self.items_tensor, self.scores_tensor, self.envs,
                self.sample_weights)):
            self._consumed_slot = None
            self._step(u, i, y, e, w, self._alpha_at(batch_index), loss_out=self._loss_rows[batch_index],
                       plan_key=batch_index)
            if self._consumed_slot is not None:                 # a streamed plan: its buffer is free after this step
                self._ring["consumed"][self._consumed_slot].record()
                self._ring["holds"][self._consumed_slot] = None
            self._prefetch_plan(batch_index + 1)
        self.epoch_cnt += 1
        self.engine.flush()
        rows = self._loss_rows.cpu().tolist()
        return merge_dict([dict(zip(LOSS_KEYS, r)) for r in rows], _mean_merge_dict_func)

    # ---- EM re-assignment ---------------------------------------------------------------------------
    def cluster_a_batch(self, batch_users_tensor, batch_items_tensor, batch_scores_tensor) -> torch.Tensor:
        """train.py:846-879 for one batch (draws its tie-break indices like the reference)."""
        perm = None
        if self.cluster_use_random_sort and self.tie_break_rng == "numpy_device":
            perm = device_randint(self.eps_random_tensor.shape[0], batch_users_tensor.shape[0], self.device)
        elif self.cluster_use_random_sort:
            idx = np.random.randint(0, self.eps_random_tensor.shape[0], batch_users_tensor.shape[0])
            perm = torch.from_numpy(idx.astype(np.int64)).to(self.device)
        new_envs, _, _ = self.engine.cluster(batch_users_tensor.contiguous(), batch_items_tensor.contiguous(),
                                             batch_scores_tensor.contiguous(), perm,
                                             self.eps_random_tensor if perm is not None else None, None)
        return new_envs

    def cluster(self) -> int:
        """train.py:912-936.  The host draws one randint per cluster batch, in order (so the numpy stream
        advances exactly as in the reference); the device does the whole dataset in one launch."""
        self.model.eval()
        n = self.users_tensor.shape[0]
        perm = None
        if self.cluster_use_random_sort and self.tie_break_rng == "device":
            # NOT the reference's stream: the tie-break rows are drawn by torch's device generator.  The draws only
            # decide between environments whose distances agree to ~1e-10 (train.py:763-769), but numpy's sequential
            # Mersenne-Twister stream costs ~10 ns per sample on the host -- 40 of the 53 ms of a MIND-sized cluster()
            perm = torch.randint(0, self.eps_random_tensor.shape[0], (n,), device=self.device)
        elif self.cluster_use_random_sort and self.tie_break_rng == "numpy_device":
            # the per-batch draws concatenate into one draw of n: the same values, numpy's state advanced the same
            perm = device_randint(self.eps_random_tensor.shape[0], n, self.device)
        elif self.cluster_use_random_sort:
            draws = [np.random.randint(0, self.eps_random_tensor.shape[0], min(self.batch_size, n - lo))
                     for lo in range(0, n, self.batch_size)]
            perm = torch.from_numpy(np.concatenate(draws)).to(self.device)       # randint draws int64 already
        eps = self.eps_random_tensor if perm is not None else None
        if self.sorted_cluster:
            if self._cl_view is None:
                self._cl_view = self.engine.sorted_view(self.users_tensor, self.items_tensor, self.scores_tensor)
            new_envs, hist, diff = self.engine.cluster_sorted(self._cl_view, perm, eps, self.envs)
        else:
            new_envs, hist, diff = self.engine.cluster(self.users_tensor, self.items_tensor, self.scores_tensor, perm,
                                                       eps, self.envs, trusted=True)
        self.envs = new_envs
        self._hist = hist
        return int(diff.item())

    def update_each_env_count(self):
        cnt = self.engine.env_hist(self.envs).cpu().tolist()
        self.each_env_count.update({k: c for k, c in enumerate(cnt)})

    def stat_envs(self) -> dict:
        """train.py:945-957: histogram, class_weights (frequency, float64 -> fp32), sample_weights."""
        hist = self.engine.env_hist(self.envs)
        self.class_weights, self.sample_weights = self.engine.stat_envs(self.envs, hist)
        return {k: int(c) for k, c in enumerate(hist.cpu().tolist())}

    # ---- epoch loop -----------------------------------------------------------------------------------
    def train(self, silent: bool = False, auto: bool = False):
        """train.py:959-1019; returns the same triple of (results, epochs) tuples."""
        test_result_list, test_epoch_list = [], []
        cluster_diff_num_list, cluster_epoch_list, envs_cnt_list = [], [], []
        loss_result_list, train_epoch_index_list = [], []
        verbose = not silent and not auto

        def evaluate():
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


class ExplicitTrainManager(_InvPrefTrainManager):
    """reference train.py:693-1019 (MSE recommend loss / MSE cluster distance)."""
    implicit = False


class ImplicitTrainManager(_InvPrefTrainManager):
    """reference train.py:16-342 (BCE recommend loss / BCE cluster distance)."""
    implicit = True

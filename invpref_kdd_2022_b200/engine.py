"""Host-side driver of the C ABI: owns the double-buffered tables, Adam state, workspace and plans.

The arithmetic lives in ``libinvpref_b200.so``; this module only holds torch tensors (device memory)
and marshals pointers.  One ``HotPath`` per model per process (= per GPU).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import torch

from . import _lib

PARAM_FIELDS = _lib.PARAM_FIELDS
TABLES = ("Uinv", "Iinv", "Uenv", "Ienv")


class HotPath:
    """Fused train step / EM re-assignment / forward for one set of InvPref parameters.

    ``params``: dict ``{Uinv, Iinv, Uenv, Ienv, E, W, b}`` of fp32 CUDA tensors (the nn.Parameter
    ``.data`` of the model, so the model sees every update).  The four tables are double-buffered
    (``invpref_train_step`` reads one set and writes the other); after each step ``params`` holds
    the NEW tensors and ``on_swap`` (if given) is called so the owner can re-point its Parameters.
    """

    def __init__(self, params: Dict[str, torch.Tensor], implicit: bool, reg_only_embed: bool, reg_env_embed: bool,
                 lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, on_swap=None, lazy: bool = False):
        """``lazy``: lazy dense Adam for the user tables (``invpref_adam.user_last_step`` in the header): rows
        that are not in a batch are not touched in memory; the skipped zero-gradient steps are replayed,
        bit-identically, when the row is next used or by ``flush()``.  Every method of this class that reads
        the user tables flushes first; code that reads ``params`` directly must call ``flush()``."""
        self.lib = _lib.load()
        for k in PARAM_FIELDS:
            t = params[k]
            if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
                raise RuntimeError(f"parameter {k} must be a contiguous fp32 CUDA tensor (no CPU fallback)")
        self.params = dict(params)
        self.device = params["Uinv"].device
        n_users, dim = params["Uinv"].shape
        n_items = params["Iinv"].shape[0]
        n_envs = params["E"].shape[0]
        self.n_users, self.n_items, self.n_envs, self.dim = n_users, n_items, n_envs, dim
        self.implicit = bool(implicit)
        self.desc = _lib.make_desc(n_users, n_items, n_envs, dim, implicit, reg_only_embed, reg_env_embed)
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.step = 0
        self.on_swap = on_swap
        self.shadow = None           # allocated on the first train step
        self.m = None
        self.v = None
        self._ws = None
        self._ws_batch = -1
        self.loss_buf = torch.zeros(6, dtype=torch.float32, device=self.device)
        # lazy Adam needs the fused user pass; shapes that only have the unfused path (K * D too large for the
        # per-CTA dE/dW slices) run plain dense Adam -- same results, more HBM traffic
        self.lazy_supported = self.lib.invpref_upass_supported(C.byref(self.desc)) == 1
        self.lazy_requested = bool(lazy)
        self.lazy = bool(lazy) and self.lazy_supported
        self.id_flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.generation = 0          # bumped whenever a buffer a captured CUDA graph may name is re-allocated
        self.parity = 0              # number of double-buffer swaps so far, mod 2
        self.last_step = None        # int32 [n_users]
        self.sched = None            # fp32 [cap, 2]
        self._dirty = False          # some user rows are behind self.step

    def _adam_struct(self):
        a = _lib.Adam(_lib.make_params(self.m), _lib.make_params(self.v), None, None, 0)
        if self.lazy:
            if self.last_step is None:
                raise RuntimeError("internal: lazy state not initialised")
            self.reserve_steps(1)
            a.user_last_step = _lib.ptr(self.last_step, torch.int32)
            a.sched = _lib.ptr(self.sched, torch.float32)
            a.sched_cap = self.sched.shape[0]
        return a

    def reserve_steps(self, n: int):
        """Lazy mode: room in the schedule table for the next ``n`` steps (grows it: re-allocation)."""
        if self.lazy and self.sched is not None and self.step + n + 2 >= self.sched.shape[0]:
            cap = self.sched.shape[0]
            while self.step + n + 2 >= cap:
                cap *= 4
            grown = torch.zeros((cap, 2), dtype=torch.float32, device=self.device)
            grown[:self.sched.shape[0]] = self.sched
            self.sched = grown
            self.generation += 1

    def _ensure_lazy(self):
        """Called with self.step == number of COMPLETED steps: every row is current at that step."""
        if self.lazy and self.last_step is None:
            self.last_step = torch.full((self.n_users,), int(self.step), dtype=torch.int32, device=self.device)
            cap = 1 << 14
            while cap <= self.step + 2:
                cap *= 4
            self.sched = torch.zeros((cap, 2), dtype=torch.float32, device=self.device)
            self.generation += 1

    def write_sched(self):
        """Lazy mode, a step without a local batch (multi-GPU: nothing routed here): only record the step's
        Adam scalars so that later replays find them."""
        import math
        t = int(self.step)
        self._adam_struct()
        bc1, bc2 = 1.0 - self.betas[0] ** t, 1.0 - self.betas[1] ** t
        self.sched[t, 0] = self.lr / bc1
        self.sched[t, 1] = 1.0 / math.sqrt(bc2)

    def set_lazy(self, lazy: bool):
        self.lazy_requested = bool(lazy)
        lazy = bool(lazy) and self.lazy_supported
        if bool(lazy) == self.lazy:
            return
        self.flush()
        self.lazy = bool(lazy)
        self.last_step = None
        self.sched = None
        self.generation += 1

    def flush(self, dyn: Optional[int] = None):
        """Lazy mode: bring every user row up to the last completed step (no-op otherwise).  ``dyn``: device
        address of the ``invpref_dyn`` record of that step (CUDA-graph capture, see ``StepGraph``)."""
        if not (self.lazy and self._dirty):
            return
        hyper = _lib.Hyper(0, 0, 0, 0, 0, 0, self.lr, self.betas[0], self.betas[1], self.eps, int(self.step), 0, 0,
                           0, 0, 0, dyn)
        p = _lib.make_params(self.params)
        adam = self._adam_struct()
        _lib.check(self.lib.invpref_flush_users(C.byref(self.desc), C.byref(p), C.byref(adam), C.byref(hyper),
                                                _lib.stream_ptr()), "flush_users")
        self._dirty = False

    # ---- the slice of the torch.optim.Optimizer surface callers of `trainer.optimizer` use (train.py:718) -------
    def zero_grad(self, set_to_none: bool = True):
        """No-op: gradients are never materialised (the segment reductions feed Adam in registers)."""

    def state_dict(self):
        """torch.optim.Adam-shaped: per-parameter step / exp_avg / exp_avg_sq in model.parameters() order."""
        self.flush()
        self._ensure_state(())
        state = {i: {"step": torch.tensor(float(self.step)), "exp_avg": self.m[k], "exp_avg_sq": self.v[k]}
                 for i, k in enumerate(PARAM_FIELDS)}
        group = {"lr": self.lr, "betas": self.betas, "eps": self.eps, "weight_decay": 0, "amsgrad": False,
                 "params": list(range(len(PARAM_FIELDS)))}
        return {"state": state, "param_groups": [group]}

    def load_state_dict(self, sd):
        self.flush()
        self._ensure_state(())
        for i, k in enumerate(PARAM_FIELDS):
            st = sd["state"][i]
            self.m[k].copy_(st["exp_avg"])
            self.v[k].copy_(st["exp_avg_sq"])
            self.step = int(st["step"])
        g = sd["param_groups"][0]
        self.lr, self.betas, self.eps = float(g["lr"]), (float(g["betas"][0]), float(g["betas"][1])), float(g["eps"])
        if self.lazy and self.last_step is not None:
            self.last_step.fill_(self.step)            # every row is current at the loaded step
        self.generation += 1

    # ---- buffers -------------------------------------------------------------------------
    def _ensure_state(self, shadow_for=TABLES):
        if self.m is None:
            self.m = {k: torch.zeros_like(self.params[k]) for k in PARAM_FIELDS}
            self.v = {k: torch.zeros_like(self.params[k]) for k in PARAM_FIELDS}
            self.generation += 1
        if self.shadow is None:
            self.shadow = {}
        for k in shadow_for:
            if k not in self.shadow:
                self.shadow[k] = self.params[k].clone()
                self.generation += 1

    def adam_dense(self, theta, m, v, grad, step=None, dyn: Optional[int] = None):
        """``invpref_adam_dense``: in-place Adam on flat fp32 tensors with a materialised gradient (``dyn``: device
        address of the step's ``invpref_dyn`` record, CUDA-graph capture)."""
        hyper = _lib.Hyper(0, 0, 0, 0, 0, 0, self.lr, self.betas[0], self.betas[1], self.eps,
                           int(step if step is not None else self.step), 0, 0, 0, 0, 0, dyn)
        _lib.check(self.lib.invpref_adam_dense(_lib.ptr(theta, torch.float32), _lib.ptr(m, torch.float32),
                                               _lib.ptr(v, torch.float32), _lib.ptr(grad, torch.float32),
                                               theta.numel(), C.byref(hyper), _lib.stream_ptr()), "adam_dense")

    def workspace(self, batch: int) -> torch.Tensor:
        if self._ws is None or batch > self._ws_batch:
            n = _lib.workspace_bytes(self.desc, batch)
            self._ws = torch.empty(n, dtype=torch.uint8, device=self.device)
            self._ws_batch = batch
            self.generation += 1
        return self._ws

    def new_plan(self, users: torch.Tensor, items: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Sort-segment plan of one batch (``invpref_build_plan``); reusable while (users, items) are fixed.

        Runs on the current stream and touches only the sort scratch of the workspace, which a ``train_step``
        that is GIVEN a plan never uses: the plan of the next batch can be built on a side stream while the
        current step runs (``out``: caller-owned buffer of at least ``plan_bytes`` bytes to build into)."""
        B = users.numel()
        n = _lib.plan_bytes(self.desc, B)
        if out is None:
            plan = torch.empty(n, dtype=torch.uint8, device=self.device)
        else:
            if not (out.is_cuda and out.dtype == torch.uint8 and out.is_contiguous() and out.numel() >= n):
                raise RuntimeError("new_plan(out=...): need a contiguous uint8 CUDA buffer of plan_bytes() bytes")
            plan = out
        ws = self.workspace(B)
        _lib.check(self.lib.invpref_build_plan(C.byref(self.desc), _lib.ptr(users, torch.int64),
                                               _lib.ptr(items, torch.int64), B, _lib.ptr(plan), plan.numel(),
                                               _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "build_plan")
        return plan

    def plan_bytes(self, batch: int) -> int:
        return _lib.plan_bytes(self.desc, batch)

    def plan_status(self, plan: torch.Tensor, B: int) -> None:
        """Raises IndexError if a user / item id of the batch the plan was built for is outside its table
        (``invpref_plan_status``; synchronises -- call it once per cached plan, not per step)."""
        _lib.check(self.lib.invpref_plan_status(C.byref(self.desc), _lib.ptr(plan), int(B), _lib.stream_ptr()),
                   "plan_status")

    def check_ids(self, users=None, items=None, envs=None, sync: bool = True) -> None:
        """``invpref_check_ids``: the reference's nn.Embedding raises on an id outside its table; here the ids are
        validated by one small kernel.  ``sync=True`` reads the flag back and raises IndexError; ``sync=False``
        only accumulates into ``self.id_flag`` (read it later with ``raise_if_bad_ids``)."""
        B = next(t.numel() for t in (users, items, envs) if t is not None)
        _lib.check(self.lib.invpref_check_ids(
            C.byref(self.desc), _lib.ptr(users, torch.int64) if users is not None else None,
            _lib.ptr(items, torch.int64) if items is not None else None,
            _lib.ptr(envs, torch.int64) if envs is not None else None, B, _lib.ptr(self.id_flag, torch.int32),
            _lib.stream_ptr()), "check_ids")
        if sync:
            self.raise_if_bad_ids()

    def raise_if_bad_ids(self) -> None:
        f = int(self.id_flag.item())
        if f:
            self.id_flag.zero_()
            what = [n for b, n in ((1, "user"), (2, "item"), (4, "env")) if f & b]
            raise IndexError(f"index out of range in self: {' / '.join(what)} id outside its embedding table "
                             f"(users {self.n_users}, items {self.n_items}, envs {self.n_envs})")

    # ---- fused train step ---------------------------------------------------------------------
    def train_step(self, users, items, scores, envs, weights, *, c_inv, c_ea, c_env, c_L2, c_L1, alpha,
                   use_class_rw, use_rec_rw, plan: Optional[torch.Tensor] = None,
                   loss_out: Optional[torch.Tensor] = None, grads_out: Optional[Dict[str, torch.Tensor]] = None,
                   global_batch: int = 0, flags: int = 0, dyn: Optional[int] = None, push=None):
        """train.py:771-844 in one library call.  Returns the device tensor holding the six losses.

        ``dyn``: device address of an ``invpref_dyn`` record; the kernels then read Adam's bias corrections,
        alpha and the step number from it instead of from the launch arguments (CUDA-graph replay).
        ``push``: an ``_lib.Push`` (``invpref_push``): exported item gradients go to peer memory.

        ``flags`` / ``global_batch``: data-parallel use, see ``invpref_hyper`` in the header; tables of an
        exported group are neither updated nor swapped."""
        self._ensure_state([k for k in TABLES
                            if not (flags & (_lib.EXPORT_USER_GRADS if k[0] == "U" else _lib.EXPORT_ITEM_GRADS))
                            and not (self.lazy and k[0] == "U")])
        B = users.numel()
        ws = self.workspace(B)
        self._ensure_lazy()
        self.step += 1
        hyper = _lib.Hyper(float(c_inv), float(c_ea), float(c_env), float(c_L2), float(c_L1), float(alpha), self.lr,
                           self.betas[0], self.betas[1], self.eps, self.step, int(bool(use_class_rw)),
                           int(bool(use_rec_rw)), int(global_batch), int(flags), 0, dyn,
                           C.cast(C.pointer(push), C.c_void_p) if push is not None else None)
        p_in = _lib.make_params(self.params)
        out = dict(self.params)
        swap = [k for k in TABLES if not (flags & (_lib.EXPORT_USER_GRADS if k[0] == "U" else _lib.EXPORT_ITEM_GRADS))
                and not (self.lazy and k[0] == "U")]           # lazy user tables are updated in place
        out.update({k: self.shadow[k] for k in swap})
        p_out = _lib.make_params(out)
        adam = self._adam_struct()
        batch = _lib.Batch(_lib.ptr(users, torch.int64), _lib.ptr(items, torch.int64), _lib.ptr(envs, torch.int64),
                           _lib.ptr(scores, torch.float32), _lib.ptr(weights, torch.float32), B)
        if loss_out is None:
            loss_out = self.loss_buf
        g = _lib.make_params(grads_out) if grads_out is not None else None
        rc = self.lib.invpref_train_step(C.byref(self.desc), C.byref(p_in), C.byref(p_out), C.byref(adam),
                                         C.byref(batch), C.byref(hyper), _lib.ptr(plan), _lib.ptr(loss_out),
                                         C.byref(g) if g is not None else None, _lib.ptr(ws), ws.numel(),
                                         _lib.stream_ptr())
        if rc != 0:
            self.step -= 1
        _lib.check(rc, "train_step")
        self._dirty = self.lazy
        # the updated rows are in the other buffer set: swap
        for k in swap:
            self.params[k], self.shadow[k] = self.shadow[k], self.params[k]
        if swap:
            self.parity ^= 1
        if self.on_swap is not None:
            self.on_swap(self.params)
        return loss_out

    # ---- host-side bookkeeping of a captured / replayed sequence of steps (StepGraph) ----------------
    def host_state(self):
        return (self.step, dict(self.params), dict(self.shadow or {}), self._dirty, self.parity)

    def restore_host_state(self, st):
        self.step, self.params, shadow, self._dirty, self.parity = st[0], dict(st[1]), dict(st[2]), st[3], st[4]
        if self.shadow is not None:
            self.shadow = shadow
        if self.on_swap is not None:
            self.on_swap(self.params)

    def advance(self, n_steps: int, flushed: bool):
        """What ``n_steps`` plain (no export flags) train steps do to the host-side state: the step counter and
        the double-buffer roles.  Called after a graph replay that ran those steps on the device."""
        self.step += int(n_steps)
        if n_steps % 2:
            for k in TABLES:
                if not (self.lazy and k[0] == "U"):
                    self.params[k], self.shadow[k] = self.shadow[k], self.params[k]
            self.parity ^= 1
            if self.on_swap is not None:
                self.on_swap(self.params)
        self._dirty = self.lazy and not flushed

    def user_sweep(self, plan: torch.Tensor, B: int):
        """The deferred dense sweep of the step that just ran with ``DEFER_USER_SWEEP`` (call it after
        ``train_step`` returned, i.e. after the buffer swap: it reads the old set and writes the current one)."""
        hyper = _lib.Hyper(0, 0, 0, 0, 0, 0, self.lr, self.betas[0], self.betas[1], self.eps, int(self.step), 0, 0,
                           0, 0, 0)
        old = dict(self.params)
        old.update({k: self.shadow[k] for k in ("Uinv", "Uenv")})
        p_in, p_out = _lib.make_params(old), _lib.make_params(self.params)
        adam = self._adam_struct()
        _lib.check(self.lib.invpref_user_sweep(C.byref(self.desc), C.byref(p_in), C.byref(p_out), C.byref(adam),
                                               C.byref(hyper), _lib.ptr(plan), int(B), _lib.stream_ptr()),
                   "user_sweep")

    # ---- forward / backward (autograd-compatible path) ----------------------------------------
    def forward(self, users, items, envs, want_logp=True, trusted=False):
        """``trusted``: the ids were validated before (e.g. the trainer's own tensors, checked at construction);
        otherwise they are checked first and an IndexError is raised like the reference's embedding lookup."""
        if not trusted and users.numel():
            self.check_ids(users, items, envs)
        self.flush()
        B = users.numel()
        s_inv = torch.empty(B, dtype=torch.float32, device=self.device)
        s_env = torch.empty(B, dtype=torch.float32, device=self.device)
        logp = torch.empty((B, self.n_envs), dtype=torch.float32, device=self.device) if want_logp else None
        p = _lib.make_params(self.params)
        _lib.check(self.lib.invpref_forward(C.byref(self.desc), C.byref(p), _lib.ptr(users, torch.int64),
                                            _lib.ptr(items, torch.int64), _lib.ptr(envs, torch.int64), B,
                                            _lib.ptr(s_inv), _lib.ptr(s_env), _lib.ptr(logp), _lib.stream_ptr()),
                   "forward")
        return s_inv, s_env, logp

    def predict(self, users, items, trusted=False):
        if not trusted and users.numel():
            self.check_ids(users, items, None)
        self.flush()
        B = users.numel()
        out = torch.empty(B, dtype=torch.float32, device=self.device)
        p = _lib.make_params(self.params)
        _lib.check(self.lib.invpref_predict(C.byref(self.desc), C.byref(p), _lib.ptr(users, torch.int64),
                                            _lib.ptr(items, torch.int64), B, _lib.ptr(out), _lib.stream_ptr()),
                   "predict")
        return out

    def backward(self, users, items, envs, alpha, g_s_inv, g_s_env, g_logp, grads: Dict[str, torch.Tensor], plan=None):
        """Accumulates the autograd gradients of ``forward`` into ``grads`` (dense, deterministic)."""
        self.flush()
        B = users.numel()
        ws = self.workspace(B)
        p = _lib.make_params(self.params)
        g = _lib.make_params(grads)
        batch = _lib.Batch(_lib.ptr(users, torch.int64), _lib.ptr(items, torch.int64), _lib.ptr(envs, torch.int64),
                           None, None, B)
        _lib.check(self.lib.invpref_backward(C.byref(self.desc), C.byref(p), C.byref(batch), float(alpha),
                                             _lib.ptr(g_s_inv), _lib.ptr(g_s_env), _lib.ptr(g_logp), _lib.ptr(plan),
                                             C.byref(g), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "backward")

    # ---- EM re-assignment -------------------------------------------------------------------------
    def cluster(self, users, items, scores, perm_idx, eps_table, old_envs, trusted=False, out=None):
        """train.py:846-879 over a whole slice.  Returns (new_envs int64[B], hist int64[K], diff int64[1]).
        ``out``: optional int64 [B] tensor to write the new environments into (no allocation in the call)."""
        if not trusted and users.numel():
            self.check_ids(users, items, None)
        self.flush()
        B = users.numel()
        new_envs = out if out is not None else torch.empty(B, dtype=torch.int64, device=self.device)
        hist = torch.zeros(self.n_envs, dtype=torch.int64, device=self.device)
        diff = torch.zeros(1, dtype=torch.int64, device=self.device)
        p = _lib.make_params(self.params)
        _lib.check(self.lib.invpref_cluster(C.byref(self.desc), C.byref(p), _lib.ptr(users, torch.int64),
                                            _lib.ptr(items, torch.int64), _lib.ptr(scores, torch.float32),
                                            _lib.ptr(perm_idx, torch.int64) if perm_idx is not None else None,
                                            _lib.ptr(eps_table, torch.float32) if eps_table is not None else None,
                                            _lib.ptr(old_envs, torch.int64) if old_envs is not None else None, B,
                                            _lib.ptr(new_envs), _lib.ptr(hist),
                                            _lib.ptr(diff) if old_envs is not None else None, _lib.stream_ptr()),
                   "cluster")
        return new_envs, hist, diff

    def sorted_view(self, users, items, scores):
        """User-sorted view of a dataset for ``cluster_sorted``: (perm int32, users int32, items int32, scores fp32).
        Built once per dataset (ids never change): a stable sort by user id."""
        perm = build_segments(users, int(self.desc.n_users))[0]            # the library's own stable radix sort
        return (perm.to(torch.int32).contiguous(), users[perm].to(torch.int32).contiguous(),
                items[perm].to(torch.int32).contiguous(), scores[perm].contiguous())

    def cluster_sorted(self, view, perm_idx, eps_table, old_envs, out=None):
        """``invpref_cluster_sorted``: the re-assignment of ``cluster`` over the user-sorted ``view`` of the dataset
        (``sorted_view``); identical results, the user rows of consecutive samples come out of L2."""
        self.flush()
        perm, us, its, ys = view
        N = perm.numel()
        new_envs = out if out is not None else torch.empty(N, dtype=torch.int64, device=self.device)
        hist = torch.zeros(self.n_envs, dtype=torch.int64, device=self.device)
        diff = torch.zeros(1, dtype=torch.int64, device=self.device)
        p = _lib.make_params(self.params)
        _lib.check(self.lib.invpref_cluster_sorted(
            C.byref(self.desc), C.byref(p), _lib.ptr(perm, torch.int32), _lib.ptr(us, torch.int32),
            _lib.ptr(its, torch.int32), _lib.ptr(ys, torch.float32),
            _lib.ptr(perm_idx, torch.int64) if perm_idx is not None else None,
            _lib.ptr(eps_table, torch.float32) if eps_table is not None else None,
            _lib.ptr(old_envs, torch.int64) if old_envs is not None else None, N, _lib.ptr(new_envs), _lib.ptr(hist),
            _lib.ptr(diff) if old_envs is not None else None, _lib.stream_ptr()), "cluster_sorted")
        return new_envs, hist, diff

    def env_hist(self, envs):
        hist = torch.zeros(self.n_envs, dtype=torch.int64, device=self.device)
        _lib.check(self.lib.invpref_env_hist(_lib.ptr(envs, torch.int64), envs.numel(), self.n_envs, _lib.ptr(hist),
                                             _lib.stream_ptr()), "env_hist")
        return hist

    def stat_envs(self, envs, hist, out=None):
        """train.py:945-957 -> (class_weights fp32[K], sample_weights fp32[N]).  ``out``: optional fp32 [N] tensor
        for the sample weights."""
        N = envs.numel()
        cw = torch.empty(self.n_envs, dtype=torch.float32, device=self.device)
        sw = out if out is not None else torch.empty(N, dtype=torch.float32, device=self.device)
        _lib.check(self.lib.invpref_stat_envs(_lib.ptr(envs, torch.int64), N, self.n_envs, _lib.ptr(hist, torch.int64),
                                              _lib.ptr(cw), _lib.ptr(sw), _lib.stream_ptr()), "stat_envs")
        return cw, sw


class StepGraph:
    """A CUDA graph over a fixed sequence of library calls (``invpref_graph_*``) plus the device records
    (``invpref_dyn``) through which the captured kernels see what changes between replays: Adam's bias corrections,
    alpha, the step number.  Replaying costs one H2D copy of the records and one graph launch, instead of ~10
    kernel launches and their host-side marshalling per step."""

    def __init__(self, hot: HotPath, n_records: int):
        self.hot, self.n = hot, int(n_records)
        self.dyn_dev = torch.zeros((self.n, 4), dtype=torch.float32, device=hot.device)
        self.dyn_host = torch.zeros((self.n, 4), dtype=torch.float32).pin_memory()
        self.stream = torch.cuda.Stream(device=hot.device)
        self.handles = {}            # start parity of the double buffers -> graph handle
        self.generation = hot.generation

    def record_ptr(self, j: int) -> int:
        return self.dyn_dev.data_ptr() + 16 * int(j)

    def fill(self, j: int, step: int, alpha: float):
        h = self.hot
        hyper = _lib.Hyper(0, 0, 0, 0, 0, float(alpha), h.lr, h.betas[0], h.betas[1], h.eps, int(step), 0, 0, 0, 0, 0)
        rec = C.cast(C.c_void_p(self.dyn_host.data_ptr() + 16 * int(j)), C.POINTER(_lib.Dyn))
        _lib.check(h.lib.invpref_dyn_fill(C.byref(hyper), rec), "dyn_fill")

    def upload(self):
        self.dyn_dev.copy_(self.dyn_host, non_blocking=True)

    def valid(self) -> bool:
        if self.generation != self.hot.generation:
            self.drop()
            self.generation = self.hot.generation
        return True

    def capture(self, key, fn):
        """Records the library calls ``fn()`` issues on the current stream (must be ``self.stream``)."""
        lib = self.hot.lib
        _lib.check(lib.invpref_graph_begin(_lib.stream_ptr()), "graph_begin")
        try:
            fn()
        finally:
            out = C.c_void_p()
            rc = lib.invpref_graph_end(_lib.stream_ptr(), C.byref(out))
        _lib.check(rc, "graph_end")
        self.handles[key] = out

    def launch(self, key):
        _lib.check(self.hot.lib.invpref_graph_launch(self.handles[key], _lib.stream_ptr()), "graph_launch")

    def launches(self, key) -> int:
        return int(self.hot.lib.invpref_graph_launches(self.handles[key]))

    def drop(self):
        for h in self.handles.values():
            self.hot.lib.invpref_graph_destroy(h)
        self.handles = {}

    def __del__(self):
        try:
            self.drop()
        except Exception:
            pass


def build_segments(ids: torch.Tensor, n_rows: int):
    """``invpref_build_segments``: (perm, seg_row, seg_off) as int64 tensors, trimmed to n_seg."""
    lib = _lib.load()
    B = ids.numel()
    dev = ids.device
    desc = _lib.make_desc(n_rows, n_rows, 2, 4, 0, 0, 0)
    ws = torch.empty(_lib.workspace_bytes(desc, B), dtype=torch.uint8, device=dev)
    S = min(max(B, 1), n_rows)
    perm = torch.empty(max(B, 1), dtype=torch.int64, device=dev)
    seg_row = torch.empty(S, dtype=torch.int64, device=dev)
    seg_off = torch.zeros(S + 1, dtype=torch.int64, device=dev)
    n_seg = torch.zeros(1, dtype=torch.int64, device=dev)
    _lib.check(lib.invpref_build_segments(_lib.ptr(ids, torch.int64) if B else None, B, n_rows, _lib.ptr(perm),
                                          _lib.ptr(seg_row), _lib.ptr(seg_off), _lib.ptr(n_seg), _lib.ptr(ws),
                                          ws.numel(), _lib.stream_ptr()), "build_segments")
    n = int(n_seg.item())
    return perm[:B], seg_row[:n], seg_off[:n + 1]

"""InvPref models with the reference's names, constructor arguments, parameter names and method
signatures (reference ``models.py:272-543``), computing on the B200 through ``libinvpref_b200.so``.

``state_dict()`` is interchangeable with the reference model's: same keys, shapes and, under the same
torch seed, the same values (layers are created and initialised in the reference's order, so the torch
RNG stream is consumed identically).
"""
from __future__ import annotations

import numpy as np
import torch
from torch import nn

from .engine import HotPath

# our short names -> attribute paths of the Parameters (reference models.py:424-432, 200)
_PARAM_PATHS = {
    "Uinv": ("embed_user_invariant", "weight"),
    "Iinv": ("embed_item_invariant", "weight"),
    "Uenv": ("embed_user_env_aware", "weight"),
    "Ienv": ("embed_item_env_aware", "weight"),
    "E": ("embed_env", "weight"),
    "W": ("env_classifier", "linear_map", "weight"),
    "b": ("env_classifier", "linear_map", "bias"),
}


class EnvClassifier(nn.Module):
    """Type name kept from the reference (models.py:53-64)."""


class LinearLogSoftMaxEnvClassifier(EnvClassifier):
    """Linear(D -> K) + LogSoftmax(dim=1), xavier-uniform weight (reference models.py:197-220).

    Inside the model the classifier is evaluated by the fused kernels; this module's own ``forward`` is
    plain torch for stand-alone use."""

    def __init__(self, factor_dim: int, env_num: int):
        super().__init__()
        self.linear_map = nn.Linear(factor_dim, env_num)
        self.classifier_func = nn.LogSoftmax(dim=1)
        nn.init.xavier_uniform_(self.linear_map.weight)
        self.elements_num = float(factor_dim * env_num)
        self.bias_num = float(env_num)

    def forward(self, invariant_preferences):
        return self.classifier_func(self.linear_map(invariant_preferences))

    def _reg(self, p: int):
        w, b = self.linear_map.weight, self.linear_map.bias
        if p == 2:
            return w.norm(2).pow(2) / self.elements_num + b.norm(2).pow(2) / self.bias_num
        return w.norm(1) / self.elements_num + b.norm(1) / self.bias_num

    def get_L1_reg(self):
        return self._reg(1)

    def get_L2_reg(self):
        return self._reg(2)


class _FusedForward(torch.autograd.Function):
    """models.py:448-467 / 307-326 as one kernel; backward = ``invpref_backward`` (deterministic
    sort-segmented reduction, gradient reversal folded in as -alpha)."""

    @staticmethod
    def forward(ctx, model, users, items, envs, alpha, *params):
        hp = model.hot_path()
        users, items, envs = users.contiguous(), items.contiguous(), envs.contiguous()
        s_inv, s_env, logp = hp.forward(users, items, envs)
        ctx.model, ctx.alpha = model, float(alpha)
        ctx.save_for_backward(users, items, envs)
        return s_inv, s_env, logp

    @staticmethod
    def backward(ctx, g_s_inv, g_s_env, g_logp):
        users, items, envs = ctx.saved_tensors
        hp = ctx.model.hot_path()
        grads = {k: torch.zeros_like(hp.params[k]) for k in hp.params}
        c = lambda g: None if g is None else g.contiguous().float()
        hp.backward(users, items, envs, ctx.alpha, c(g_s_inv), c(g_s_env), c(g_logp), grads)
        order = ("Uinv", "Iinv", "Uenv", "Ienv", "E", "W", "b")
        return (None, None, None, None, None) + tuple(grads[k] for k in order)


class _InvPref(nn.Module):
    implicit = False

    def __init__(self, user_num: int, item_num: int, env_num: int, factor_num: int, reg_only_embed: bool = False,
                 reg_env_embed: bool = True):
        super().__init__()
        self.user_num, self.item_num, self.env_num = user_num, item_num, env_num
        self.factor_num: int = factor_num
        # creation order == reference (models.py:424-432) so the RNG stream matches
        self.embed_user_invariant = nn.Embedding(user_num, factor_num)
        self.embed_item_invariant = nn.Embedding(item_num, factor_num)
        self.embed_user_env_aware = nn.Embedding(user_num, factor_num)
        self.embed_item_env_aware = nn.Embedding(item_num, factor_num)
        self.embed_env = nn.Embedding(env_num, factor_num)
        self.env_classifier: EnvClassifier = LinearLogSoftMaxEnvClassifier(factor_num, env_num)
        if self.implicit:
            self.output_func = nn.Sigmoid()
        self.reg_only_embed: bool = reg_only_embed
        self.reg_env_embed: bool = reg_env_embed
        self._init_weight()
        self._hot: HotPath | None = None

    def _init_weight(self):
        for emb in (self.embed_user_invariant, self.embed_item_invariant, self.embed_user_env_aware,
                    self.embed_item_env_aware, self.embed_env):
            nn.init.normal_(emb.weight, std=0.01)                      # models.py:441-446

    # ---- binding to the fused engine ---------------------------------------------------------
    def _param(self, key) -> nn.Parameter:
        obj = self
        for a in _PARAM_PATHS[key]:
            obj = getattr(obj, a)
        return obj

    def named_hot_params(self):
        return {k: self._param(k) for k in _PARAM_PATHS}

    def _repoint(self, tensors):
        for k, t in tensors.items():
            p = self._param(k)
            if p.data.data_ptr() != t.data_ptr():
                p.data = t

    def hot_path(self, lr: float = 1e-3, lazy: bool = None) -> HotPath:
        """The engine bound to this model's parameter storages (created on first use).  ``lazy``: see
        ``HotPath``; every read through this module (forward, predict, state_dict) flushes first."""
        cur = {k: p.data for k, p in self.named_hot_params().items()}
        if self._hot is None or any(self._hot.params[k].data_ptr() != cur[k].data_ptr() for k in cur):
            if not cur["Uinv"].is_cuda:
                raise RuntimeError("InvPref runs on CUDA only: move the model to a B200 (`.to('cuda')`); "
                                   "there is no CPU fallback")
            keep = self._hot
            self._hot = HotPath(cur, self.implicit, self.reg_only_embed, self.reg_env_embed, lr=lr,
                                on_swap=self._repoint, lazy=bool(lazy))
            if keep is not None and keep.m is not None and keep.params["Uinv"].shape == cur["Uinv"].shape:
                self._hot.m, self._hot.v, self._hot.step = keep.m, keep.v, keep.step
        elif lazy is not None:
            self._hot.set_lazy(lazy)
        return self._hot

    def state_dict(self, *a, **kw):
        if self._hot is not None:
            self._hot.flush()           # lazily updated user rows are brought up to date first
        return super().state_dict(*a, **kw)

    def _apply(self, fn, *a, **kw):
        """``.to(device)`` / ``.float()`` / ``.cuda()``: lazily updated user rows are brought up to date first; the
        engine (which holds the Adam state) is dropped only if a storage was actually re-allocated -- a no-op call
        keeps it.  A trainer built before a re-allocation refuses to step afterwards (train.py)."""
        if self._hot is not None:
            self._hot.flush()
        before = {k: p.data.data_ptr() for k, p in self.named_hot_params().items()}
        out = super()._apply(fn, *a, **kw)
        if any(p.data.data_ptr() != before[k] for k, p in self.named_hot_params().items()):
            self._hot = None
        return out

    # ---- reference API -----------------------------------------------------------------------
    def forward(self, users_id, items_id, envs_id, alpha):
        """-> (invariant_score [B], env_aware_score [B], env_outputs [B, K] log-probabilities)."""
        ps = self.named_hot_params()
        order = ("Uinv", "Iinv", "Uenv", "Ienv", "E", "W", "b")
        s_inv, s_env, logp = _FusedForward.apply(self, users_id, items_id, envs_id, alpha, *[ps[k] for k in order])
        return s_inv.reshape(-1), s_env.reshape(-1), logp.reshape(-1, self.env_num)

    def _pair_reg(self, inv: nn.Embedding, env: nn.Embedding, ids, norm: int):
        if self._hot is not None:
            self._hot.flush()
        a, b = inv(ids), env(ids)
        den = float(len(ids)) * float(self.factor_num) * 2
        if norm == 2:
            return (b.norm(2).pow(2) + a.norm(2).pow(2)) / den
        if norm == 1:
            return (b.norm(1) + a.norm(1)) / den
        raise KeyError("norm must be 1 or 2")

    def get_users_reg(self, users_id, norm: int):
        return self._pair_reg(self.embed_user_invariant, self.embed_user_env_aware, users_id, norm)

    def get_items_reg(self, items_id, norm: int):
        return self._pair_reg(self.embed_item_invariant, self.embed_item_env_aware, items_id, norm)

    def get_envs_reg(self, envs_id, norm: int):
        g = self.embed_env(envs_id)
        den = float(len(envs_id)) * float(self.factor_num)
        if norm == 2:
            return g.norm(2).pow(2) / den
        if norm == 1:
            return g.norm(1) / den
        raise KeyError("norm must be 1 or 2")

    def _reg(self, users_id, items_id, envs_id, norm: int):
        """models.py:506-532.  Plain torch (differentiable); the fused train step computes the same value
        and its gradient in-kernel and does not call this."""
        r = self.get_users_reg(users_id, norm) + self.get_items_reg(items_id, norm)
        if not self.reg_only_embed:
            r = (self.env_classifier.get_L2_reg() if norm == 2 else self.env_classifier.get_L1_reg()) + r
        if self.reg_env_embed:
            r = r + self.get_envs_reg(envs_id, norm)
        return r

    def get_L2_reg(self, users_id, items_id, envs_id):
        return self._reg(users_id, items_id, envs_id, 2)

    def get_L1_reg(self, users_id, items_id, envs_id):
        return self._reg(users_id, items_id, envs_id, 1)

    def recommend(self, users_id, k: int, exclude=None):
        """The ``k`` best items of each user over the whole catalogue -> (items int64 [b, k], scores fp32 [b, k]),
        score descending (the implicit model's sigmoid), ties to the lower item id.  ``exclude``: ``(off, items)``
        CSR over user ids (numpy arrays or tensors, e.g. ``dataloader.user_item_csr`` of the training pairs, or an
        implicit loader's ``mask_off`` / ``mask_items``), uploaded per call: those items are never returned, and a
        user with fewer than ``k`` eligible items gets item -1 / score -inf in the trailing slots.  Scores can differ
        from ``predict`` in the last bits (a different summation order)."""
        hp = self.hot_path()
        return hp.recommend(_ids_on(users_id, hp.device), k, _csr_on(exclude, hp.device))

    def similar_items(self, items_id, k: int):
        """The ``k`` items nearest to each given item by cosine of the invariant item embeddings -> (items int64
        [b, k], cosines fp32 [b, k]), descending, ties to the lower item id; an item is never its own neighbour, so
        ``k == item_num`` ends in item -1 / score -inf.  No sigmoid on either model.  Zero rows score +0 against every
        finite row; a row holding NaN or inf scores NaN (ranked first).  ``items_id``: numpy array or tensor."""
        hp = self.hot_path()
        return hp.similar_items(_ids_on(items_id, hp.device), k)

    def top_users(self, items_id, k: int, exclude=None):
        """The ``k`` users of largest score for each given item -> (users int64 [b, k], scores fp32 [b, k]), score
        descending, ties to the lower user id; the scores are ``recommend``'s for the same (user, item), bit for bit.
        ``exclude``: ``(off, users)`` CSR over item ids (numpy arrays or tensors), e.g. the users who already
        interacted with each item, ``dataloader.user_item_csr(items, users, item_num)`` of the training pairs: those
        users are never returned, and an item with fewer than ``k`` eligible users gets user -1 / score -inf in the
        trailing slots."""
        hp = self.hot_path()
        return hp.top_users(_ids_on(items_id, hp.device), k, _csr_on(exclude, hp.device))

    def fold_in_users(self, off, items, scores, l2: float, max_iter: int = 25, return_iters: bool = False):
        """Invariant rows for users who are not in the table (signed up after training) -> fp32 [b, D], with the item
        table fixed: row r minimises the model's own invariant loss over the user's history (items[off[r]:off[r+1]],
        scores[...]) plus ``l2 / 2 * |u|^2`` -- ridge regression on the explicit model, logistic regression (damped
        Newton, at most ``max_iter`` steps) on the implicit one -- in fp64 on the GPU, rounded to fp32 once.  Rank the
        catalogue for the new users with ``recommend_rows``.  ``l2`` > 0 has no default: the training L2 term is a
        per-batch mean and does not map onto a per-row ridge.  ``off`` / ``items`` / ``scores``: numpy arrays or
        tensors, e.g. ``dataloader.interaction_csr(rows, items, scores, b)``.  An empty history gives the zero row; a
        NaN / inf score or table row makes that row NaN.  ``return_iters``: also return the Newton step counts (int32
        [b]; 1 on the explicit model, 0 for an empty history, ``-max_iter`` if the stopping rule was not met).  Ids
        outside the item table raise IndexError."""
        hp = self.hot_path()
        return hp.fold_in_users(*_history_on(off, items, scores, hp.device), l2, max_iter, return_iters)

    def fold_in_items(self, off, users, scores, l2: float, max_iter: int = 25, return_iters: bool = False):
        """``fold_in_users`` for items that are not in the table (e.g. news published after training), from their
        (user, score) histories, against the user table -> fp32 item rows [b, D] for ``top_users_rows``."""
        hp = self.hot_path()
        return hp.fold_in_items(*_history_on(off, users, scores, hp.device), l2, max_iter, return_iters)

    def recommend_rows(self, rows, k: int, exclude=None):
        """``recommend`` for user rows that are not in the table (e.g. from ``fold_in_users``): ``rows`` fp32 [b, D]
        -> (items int64 [b, k], scores fp32 [b, k]); the scores are ``recommend``'s for a user with that row, bit for
        bit.  ``exclude``: ``(off, items)`` CSR over the b rows (e.g. the history that was folded in)."""
        hp = self.hot_path()
        return hp.recommend_rows(torch.as_tensor(rows, dtype=torch.float32).to(hp.device), k,
                                 _csr_on(exclude, hp.device))

    def top_users_rows(self, rows, k: int, exclude=None):
        """``top_users`` for item rows that are not in the table (e.g. from ``fold_in_items``): ``rows`` fp32 [b, D]
        -> (users int64 [b, k], scores fp32 [b, k]).  ``exclude``: ``(off, users)`` CSR over the b rows."""
        hp = self.hot_path()
        return hp.top_users_rows(torch.as_tensor(rows, dtype=torch.float32).to(hp.device), k,
                                 _csr_on(exclude, hp.device))

    def cluster_predict(self, users_id, items_id, envs_id) -> torch.Tensor:
        """models.py:541-543 / 409-411: env-aware score only (the classifier pass is skipped)."""
        hp = self.hot_path()
        _, s_env, _ = hp.forward(users_id.contiguous(), items_id.contiguous(), envs_id.contiguous(), want_logp=False)
        return s_env


def _ids_on(ids, dev) -> torch.Tensor:
    return torch.as_tensor(ids, dtype=torch.int64).reshape(-1).to(dev)


def _csr_on(csr, dev):
    """(off, ids) numpy arrays or tensors -> tensors on `dev` (uploaded per call); None stays None."""
    if csr is None:
        return None
    return tuple(torch.as_tensor(np.ascontiguousarray(x) if isinstance(x, np.ndarray) else x).to(dev) for x in csr)


def _history_on(off, ids, scores, dev):
    """A fold-in history (off, ids, scores) of numpy arrays or tensors -> int64 / int64 / fp32 tensors on `dev`."""
    off, ids = _csr_on((off, ids), dev)
    scores = torch.as_tensor(np.ascontiguousarray(scores) if isinstance(scores, np.ndarray) else scores)
    return off.to(torch.int64), ids.to(torch.int64), scores.to(dev, torch.float32)


class BasicRecommender(nn.Module):
    """Type names kept from the reference (models.py:67-148); they carry no arithmetic."""


class BasicExplicitRecommender(nn.Module):
    pass


class GeneralDebiasImplicitRecommender(BasicRecommender):
    pass


class GeneralDebiasExplicitRecommender(BasicExplicitRecommender):
    pass


class InvPrefExplicit(_InvPref, GeneralDebiasExplicitRecommender):
    """reference models.py:414-543."""
    implicit = False

    def predict(self, users_id, items_id):
        """models.py:534-539: invariant score of (user, item) pairs."""
        return self.hot_path().predict(users_id.contiguous(), items_id.contiguous()).reshape(-1)


class InvPrefImplicit(_InvPref, GeneralDebiasImplicitRecommender):
    """reference models.py:272-411."""
    implicit = True

    def predict(self, users_id):
        """models.py:393-407: sigmoid(<u_inv, i_inv>) for every item -> [b, item_num].  The reference
        materialises a [b*I, D] repeat; this is the same contraction as one GEMM (evaluation is off the
        hot path, SURVEY.md §8f rank 1)."""
        if self._hot is not None:
            self._hot.flush()
        u = self.embed_user_invariant(users_id)
        return torch.sigmoid(u @ self.embed_item_invariant.weight.t())

"""Data loaders with the attribute surface the drivers / evaluators use (reference ``dataloader.py:118-243``
``YahooImplicitBCELossDataLoader`` and ``:388-483`` ``ExplicitDataLoader``): CSV ``user_id,item_id,score`` with a
header line -> ``int64 [N, 3]``; table sizes = max id + 1.  Host-side ingest, vectorised with numpy (the
reference parses line by line in Python); off the hot path (SURVEY.md §8f rank 3).
"""
from __future__ import annotations

import os

import numpy as np
import torch


# ---- binary columnar cache of an interaction file (SURVEY.md 8f rank 3) -------------------------------------------
# The reference re-parses ``user_id,item_id,score`` text line by line in Python on every run (utils.py:208-252):
# minutes at 10^9 rows.  The first read of a CSV here writes ``<file>.invpref.bin`` next to it -- a 64-byte header and
# three columns, ids compressed to the narrowest of int16 / int32 that holds them, scores to int8 when they are small
# integers (ratings 1..5, clicks 0/1) and fp32 otherwise -- and later reads memory-map it: 9 (or 5) bytes per
# interaction instead of ~12 bytes of text to tokenise.  The cache is keyed on the CSV's size and mtime; the API keeps
# handing out int64 [N, 3] arrays, as the reference does.
_MAGIC = b"INVPREF1"
_CODES = {1: np.int8, 2: np.int16, 4: np.int32, 14: np.float32}


def _narrow_ids(col: np.ndarray):
    mx, mn = (int(col.max()), int(col.min())) if col.size else (0, 0)
    if mn >= 0 and mx < (1 << 15):
        return 2, col.astype(np.int16)
    if mn >= -(1 << 31) and mx < (1 << 31):
        return 4, col.astype(np.int32)
    raise ValueError("ids beyond int32 are not supported (tables are limited to 2^31 rows)")


def _narrow_col(col: np.ndarray, is_id: bool):
    if is_id:
        return _narrow_ids(col)
    if np.all(col == np.round(col)) and (col.size == 0 or (col.min() >= -128 and col.max() <= 127)):
        return 1, col.astype(np.int8)
    return 14, col.astype(np.float32)


def write_interaction_cache(path: str, data: np.ndarray, src_size: int = 0, src_mtime_ns: int = 0) -> None:
    """``data``: [N, C], C = 2 (user, item: test / item-pool files) or 3 (user, item, score).  Atomic (written to a
    temporary file, then renamed)."""
    data = np.asarray(data)
    n, c = int(data.shape[0]), int(data.shape[1])
    if not 2 <= c <= 3:
        raise ValueError("interaction files have 2 or 3 columns")
    cols = [_narrow_col(data[:, j], j < 2) for j in range(c)]
    header = np.zeros(8, dtype=np.int64)
    header[0] = int.from_bytes(_MAGIC, "little")
    header[1:4] = (n, int(src_size), int(src_mtime_ns))
    header[4] = c
    for j, (code, _) in enumerate(cols):
        header[5 + j] = code
    tmp = path + f".tmp{os.getpid()}"
    with open(tmp, "wb") as f:
        f.write(header.tobytes())
        for _, col in cols:
            f.write(np.ascontiguousarray(col).tobytes())
            f.write(b"\0" * ((-col.nbytes) % 8))                     # columns start 8-byte aligned
    os.replace(tmp, path)


def read_interaction_cache(path: str, src_size: int = None, src_mtime_ns: int = None):
    """int64 [N, C], or None if the file is missing, foreign, or stale against (src_size, src_mtime_ns)."""
    try:
        header = np.fromfile(path, dtype=np.int64, count=8)
    except (FileNotFoundError, OSError):
        return None
    if header.size < 8 or int(header[0]) != int.from_bytes(_MAGIC, "little"):
        return None
    n, size, mtime, c = (int(x) for x in header[1:5])
    codes = [int(x) for x in header[5:5 + max(0, min(c, 3))]]
    if src_size is not None and (size, mtime) != (int(src_size), int(src_mtime_ns)):
        return None
    if not 2 <= c <= 3 or any(code not in _CODES for code in codes):
        return None
    out = np.empty((n, c), dtype=np.int64)
    off = 64
    for j, code in enumerate(codes):
        dt = np.dtype(_CODES[code])
        col = np.memmap(path, dtype=dt, mode="r", offset=off, shape=(n,)) if n else np.zeros(0, dt)
        out[:, j] = col                                              # widening copy, column by column
        off += n * dt.itemsize + ((-n * dt.itemsize) % 8)
    return out


def _read_csv(path: str, cache: bool = True) -> np.ndarray:
    """``user_id,item_id,score`` with a header line -> int64 [N, 3]; through the binary cache when possible."""
    st = os.stat(path)
    bin_path = path + ".invpref.bin"
    if cache:
        got = read_interaction_cache(bin_path, st.st_size, st.st_mtime_ns)
        if got is not None:
            return got
    import pandas as pd
    data = pd.read_csv(path).values.astype(np.int64)
    if cache:
        try:
            write_interaction_cache(bin_path, data, st.st_size, st.st_mtime_ns)
        except (OSError, ValueError):
            pass                                                     # read-only dataset directory: parse every time
    return data


def user_item_csr(users: np.ndarray, items: np.ndarray, n_users: int):
    """Per-user sorted unique item lists as (offsets [n_users+1], items [nnz]): the list format of the evaluator and
    of ``recommend(..., exclude=...)`` (e.g. the training pairs, to leave out items a user has already seen).  With
    the roles swapped, ``user_item_csr(items, users, n_items)`` gives the users of each item: the ``exclude`` lists
    of ``top_users`` (users who already interacted with an item)."""
    users, items = np.asarray(users), np.asarray(items)
    width = int(items.max()) + 1 if items.size else 1
    key = np.unique(users.astype(np.int64) * width + items)
    off = np.zeros(n_users + 1, dtype=np.int64)
    np.add.at(off, key // width + 1, 1)
    return np.cumsum(off), key % width


def interaction_csr(rows: np.ndarray, cols: np.ndarray, scores: np.ndarray, n_rows: int):
    """Interaction triples grouped by row as (offsets int64 [n_rows + 1], cols int64 [n], scores fp32 [n]): the
    history format of ``fold_in_users`` (rows = new users, cols = items) and ``fold_in_items`` (rows = new items,
    cols = users).  Stable: a row's entries keep their input order; duplicates are kept (each is an observation)."""
    rows = np.asarray(rows, dtype=np.int64).reshape(-1)
    cols = np.asarray(cols, dtype=np.int64).reshape(-1)
    scores = np.asarray(scores, dtype=np.float32).reshape(-1)
    if not (rows.size == cols.size == scores.size):
        raise ValueError(f"rows, cols and scores differ in length: {rows.size}, {cols.size}, {scores.size}")
    if rows.size and (rows.min() < 0 or rows.max() >= n_rows):
        raise IndexError(f"row id outside [0, {n_rows})")
    order = np.argsort(rows, kind="stable")
    off = np.zeros(n_rows + 1, dtype=np.int64)
    np.cumsum(np.bincount(rows, minlength=n_rows), out=off[1:])
    return off, cols[order], scores[order]


_csr = user_item_csr        # tests/test_gpu_drivers.py imports the earlier private name


class ExplicitDataLoader:
    """reference dataloader.py:388-483."""

    def __init__(self, dataset_path: str, device: torch.device, train: np.ndarray = None, test: np.ndarray = None,
                 cache: bool = True):
        """``cache``: keep / use the binary columnar cache ``<file>.invpref.bin`` next to each CSV."""
        self.dataset_path, self.device = dataset_path, device
        self._train_data = train if train is not None else _read_csv(os.path.join(dataset_path, "train.csv"), cache)
        self._test_data = test if test is not None else _read_csv(os.path.join(dataset_path, "test.csv"), cache)
        self._user_num = int(self._train_data[:, 0].max()) + 1          # dataloader.py:406-407
        self._item_num = int(self._train_data[:, 1].max()) + 1
        self._test_pairs_tensor = torch.LongTensor(self._test_data[:, 0:2]).to(device)
        self._test_scores_tensor = torch.Tensor(self._test_data[:, 2].astype(np.float64)).to(device)

    user_num = property(lambda self: self._user_num)
    item_num = property(lambda self: self._item_num)
    train_data_np = property(lambda self: self._train_data)
    test_data_np = property(lambda self: self._test_data)
    train_data_len = property(lambda self: self._train_data.shape[0])
    test_data_len = property(lambda self: self._test_data.shape[0])
    all_test_pairs_tensor = property(lambda self: self._test_pairs_tensor)
    all_test_scores_tensor = property(lambda self: self._test_scores_tensor)


class YahooImplicitBCELossDataLoader:
    """reference dataloader.py:118-243: train triples with 0/1 scores, test positives per user, the set of
    train positives per user (masked at evaluation), optional test item pool."""

    def __init__(self, dataset_path: str, device: torch.device, has_item_pool_file: bool = False,
                 train: np.ndarray = None, test: np.ndarray = None, cache: bool = True):
        self.dataset_path, self.device = dataset_path, device
        self._train_data = train if train is not None else _read_csv(os.path.join(dataset_path, "train.csv"), cache)
        self._test_data = test if test is not None else _read_csv(os.path.join(dataset_path, "test.csv"), cache)
        self.has_item_pool = has_item_pool_file
        tr, te = self._train_data, self._test_data
        self._user_num = int(max(tr[:, 0].max(), te[:, 0].max())) + 1     # dataloader.py:179-180
        self._item_num = int(max(tr[:, 1].max(), te[:, 1].max())) + 1
        pos = tr[tr[:, 2] > 0]
        self.mask_off, self.mask_items = user_item_csr(pos[:, 0], pos[:, 1], self._user_num)
        self.gt_off, self.gt_items = user_item_csr(te[:, 0], te[:, 1], self._user_num)
        # test users ascending (utils.py:228-233 sorts the user list)
        self.test_user_list = np.unique(te[:, 0]).tolist()
        self.test_users_tensor = torch.LongTensor(self.test_user_list).to(device)
        if has_item_pool_file and train is None:
            self.set_item_pool(_read_csv(os.path.join(dataset_path, "test_item_pool.csv"), cache))

    def set_item_pool(self, pool: np.ndarray):
        """pool: int [n, >=2] (user_id, item_id) rows of test_item_pool.csv (dataloader.py:168-176)."""
        self.has_item_pool = True
        self.pool_off, self.pool_items = user_item_csr(pool[:, 0], pool[:, 1], self._user_num)

    def _row(self, off, items, user_id):
        return set(items[off[user_id]:off[user_id + 1]].tolist())

    def user_mask_items(self, user_id: int) -> set:
        return self._row(self.mask_off, self.mask_items, user_id)

    def user_highlight_items(self, user_id: int) -> set:
        if not self.has_item_pool:
            raise NotImplementedError('Not has item pool!')
        return self._row(self.pool_off, self.pool_items, user_id)

    def get_user_ground_truth(self, user_id: int) -> set:
        return self._row(self.gt_off, self.gt_items, user_id)

    user_num = property(lambda self: self._user_num)
    item_num = property(lambda self: self._item_num)
    train_data_np = property(lambda self: self._train_data)
    test_data_np = property(lambda self: self._test_data)
    train_data_len = property(lambda self: self._train_data.shape[0])
    test_data_len = property(lambda self: self._test_data.shape[0])
    all_test_users_by_sorted_tensor = property(lambda self: self.test_users_tensor)
    all_test_users_by_sorted_list = property(lambda self: self.test_user_list)

    @property
    def get_sorted_all_test_users_ground_truth(self) -> list:
        return [self.get_user_ground_truth(u) for u in self.test_user_list]


def synthetic_item_pool(test: np.ndarray, n_users: int, n_items: int, extra: int = 50, seed: int = 11) -> np.ndarray:
    """A stand-in for test_item_pool.csv on synthetic data: per test user its test items plus `extra` random ones."""
    rng = np.random.default_rng(seed)
    users = np.unique(test[:, 0])
    rnd = np.stack([np.repeat(users, extra), rng.integers(0, n_items, users.size * extra)], axis=1)
    return np.concatenate([test[:, :2], rnd]).astype(np.int64)


def synthetic_interactions(n_users, n_items, n, implicit, seed=20220814):
    """SURVEY.md §8d generators, for the configs whose train.csv is not in the reference checkout
    (MovieLens, MIND: .MISSING_LARGE_BLOBS)."""
    rng = np.random.default_rng(seed)
    u = np.floor(n_users * rng.random(n) ** 1.5).astype(np.int64)
    i = np.floor(n_items * rng.random(n) ** 3).astype(np.int64)
    u[0], i[0] = n_users - 1, n_items - 1
    y = rng.integers(0, 2, n) if implicit else rng.integers(1, 6, n)
    return np.stack([u, i, y], axis=1).astype(np.int64)

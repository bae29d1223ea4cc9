"""ctypes binding of ``libinvpref_b200.so`` (C ABI in ``include/invpref_b200.h``).

PyTorch is used only for device memory and streams: tensors are passed as raw device
pointers.  There is no CPU fallback -- a missing library or a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# INVPREF_LIB: load another build of the same library instead of the in-tree one
LIB_PATH = os.environ.get("INVPREF_LIB") or os.path.join(_HERE, "libinvpref_b200.so")

MAX_ENVS = 8
MAX_DIM = 256
LOSS_KEYS = ("invariant_loss", "env_aware_loss", "envs_loss", "L2_reg", "L1_reg", "loss")  # train.py:836-843
PARAM_FIELDS = ("Uinv", "Iinv", "Uenv", "Ienv", "E", "W", "b")

EXPORTS = (
    "invpref_strerror", "invpref_abi_version", "invpref_workspace_bytes", "invpref_plan_bytes",
    "invpref_build_plan", "invpref_build_segments", "invpref_forward", "invpref_predict",
    "invpref_backward", "invpref_train_step", "invpref_cluster", "invpref_stat_envs",
    "invpref_env_hist", "invpref_launch_count", "invpref_profile_enable", "invpref_profile_steps",
    "invpref_profile_read", "invpref_adam_dense", "invpref_gather_rows", "invpref_scatter_add_rows",
    "invpref_user_sweep", "invpref_flush_users", "invpref_fetch_rows_p2p",
    "invpref_mask_scores", "invpref_hits_from_csr", "invpref_upass_supported", "invpref_plan_status",
    "invpref_check_ids", "invpref_dyn_fill", "invpref_graph_begin", "invpref_graph_end", "invpref_graph_launch",
    "invpref_graph_destroy", "invpref_graph_launches", "invpref_owner_adam_push", "invpref_eval_topk",
    "invpref_cluster_sorted", "invpref_peer_allreduce", "invpref_mt_jump_bytes", "invpref_mt_build_jumps",
    "invpref_mt_randint", "invpref_recommend", "invpref_similar_items", "invpref_top_users",
    "invpref_fold_in_users", "invpref_fold_in_items", "invpref_recommend_rows", "invpref_top_users_rows",
)
# execution order; on the fused path "forward" is empty and chunks_users / rows_users are the fused user pass
PHASES = ("plan", "forward", "chunks_users", "rows_users", "chunks_items", "rows_items", "sweep_items",
          "sweep_users", "tail")


class Desc(C.Structure):
    _fields_ = [("n_users", C.c_int64), ("n_items", C.c_int64), ("n_envs", C.c_int32), ("dim", C.c_int32),
                ("implicit", C.c_int32), ("reg_only_embed", C.c_int32), ("reg_env_embed", C.c_int32),
                ("_pad", C.c_int32)]


class Params(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in PARAM_FIELDS]


class Adam(C.Structure):
    _fields_ = [("m", Params), ("v", Params), ("user_last_step", C.c_void_p), ("sched", C.c_void_p),
                ("sched_cap", C.c_int64)]


class Batch(C.Structure):
    _fields_ = [("users", C.c_void_p), ("items", C.c_void_p), ("envs", C.c_void_p), ("scores", C.c_void_p),
                ("weights", C.c_void_p), ("B", C.c_int64)]


class Hyper(C.Structure):
    _fields_ = [("c_inv", C.c_double), ("c_ea", C.c_double), ("c_env", C.c_double), ("c_L2", C.c_double),
                ("c_L1", C.c_double), ("alpha", C.c_double), ("lr", C.c_double), ("beta1", C.c_double),
                ("beta2", C.c_double), ("eps", C.c_double), ("step", C.c_int64), ("use_class_rw", C.c_int32),
                ("use_rec_rw", C.c_int32), ("global_batch", C.c_int64), ("flags", C.c_int32), ("_pad", C.c_int32),
                ("dyn", C.c_void_p), ("push", C.c_void_p)]


class Push(C.Structure):
    """invpref_push: where the item pass stores its exported partial gradients in peer memory."""
    _fields_ = [("base", C.c_void_p), ("owner", C.c_void_p), ("index", C.c_void_p), ("world", C.c_int32),
                ("_pad", C.c_int32)]


class Dyn(C.Structure):
    """invpref_dyn: the step-dependent scalars of one train step (device record for CUDA-graph replay)."""
    _fields_ = [("step_size", C.c_float), ("inv_bc2_sqrt", C.c_float), ("neg_alpha", C.c_float), ("step", C.c_int32)]


EXPORT_USER_GRADS, EXPORT_ITEM_GRADS, EXPORT_SMALL_GRADS, SKIP_PARAM_REG, DEFER_USER_SWEEP = 1, 2, 4, 8, 16


_lib = None


def load() -> C.CDLL:
    """Loads the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C invpref_kdd_2022_b200/csrc -j`.  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i64, sz = C.c_void_p, C.c_int64, C.c_size_t
    lib.invpref_strerror.restype = C.c_char_p
    lib.invpref_strerror.argtypes = [C.c_int]
    lib.invpref_abi_version.restype = C.c_int
    lib.invpref_launch_count.restype = C.c_int64
    lib.invpref_workspace_bytes.argtypes = [C.POINTER(Desc), i64, C.POINTER(sz)]
    lib.invpref_plan_bytes.argtypes = [C.POINTER(Desc), i64, C.POINTER(sz)]
    lib.invpref_build_plan.argtypes = [C.POINTER(Desc), vp, vp, i64, vp, sz, vp, sz, vp]
    lib.invpref_upass_supported.argtypes = [C.POINTER(Desc)]
    lib.invpref_plan_status.argtypes = [C.POINTER(Desc), vp, i64, vp]
    lib.invpref_check_ids.argtypes = [C.POINTER(Desc), vp, vp, vp, i64, vp, vp]
    lib.invpref_dyn_fill.argtypes = [C.POINTER(Hyper), C.POINTER(Dyn)]
    lib.invpref_graph_begin.argtypes = [vp]
    lib.invpref_graph_end.argtypes = [vp, C.POINTER(vp)]
    lib.invpref_graph_launch.argtypes = [vp, vp]
    lib.invpref_graph_destroy.argtypes = [vp]
    lib.invpref_graph_launches.argtypes = [vp]
    lib.invpref_graph_launches.restype = C.c_int64
    lib.invpref_build_segments.argtypes = [vp, i64, i64, vp, vp, vp, vp, vp, sz, vp]
    lib.invpref_forward.argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, vp, vp, i64, vp, vp, vp, vp]
    lib.invpref_predict.argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, vp, i64, vp, vp]
    lib.invpref_backward.argtypes = [C.POINTER(Desc), C.POINTER(Params), C.POINTER(Batch), C.c_double, vp, vp, vp, vp,
                                     C.POINTER(Params), vp, sz, vp]
    lib.invpref_train_step.argtypes = [C.POINTER(Desc), C.POINTER(Params), C.POINTER(Params), C.POINTER(Adam),
                                       C.POINTER(Batch), C.POINTER(Hyper), vp, vp, C.POINTER(Params), vp, sz, vp]
    lib.invpref_cluster.argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp]
    lib.invpref_cluster_sorted.argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, vp, vp, vp, vp, vp, vp, i64, vp, vp,
                                           vp, vp]
    lib.invpref_stat_envs.argtypes = [vp, i64, C.c_int32, vp, vp, vp, vp]
    lib.invpref_env_hist.argtypes = [vp, i64, C.c_int32, vp, vp]
    lib.invpref_adam_dense.argtypes = [vp, vp, vp, vp, i64, C.POINTER(Hyper), vp]
    lib.invpref_flush_users.argtypes = [C.POINTER(Desc), C.POINTER(Params), C.POINTER(Adam), C.POINTER(Hyper), vp]
    lib.invpref_user_sweep.argtypes = [C.POINTER(Desc), C.POINTER(Params), C.POINTER(Params), C.POINTER(Adam),
                                       C.POINTER(Hyper), vp, i64, vp]
    lib.invpref_gather_rows.argtypes = [vp, vp, i64, C.c_int32, vp, vp]
    lib.invpref_scatter_add_rows.argtypes = [vp, vp, i64, C.c_int32, vp, vp]
    lib.invpref_fetch_rows_p2p.argtypes = [C.POINTER(vp), C.c_int32, vp, vp, i64, C.c_int32, vp, vp, vp]
    lib.invpref_owner_adam_push.argtypes = [vp, vp, vp, vp, vp, vp, i64, C.c_int32, C.c_int32, vp, vp, vp,
                                            C.POINTER(vp), vp, C.POINTER(Hyper), vp]
    lib.invpref_peer_allreduce.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(vp), C.POINTER(vp),
                                           vp, vp, vp]
    lib.invpref_eval_topk.argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, i64, vp, vp, vp, vp, vp, vp, C.c_int32,
                                      vp, vp, vp, vp, vp]
    lib.invpref_recommend.argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, i64, vp, vp, C.c_int32, vp, vp, vp]
    lib.invpref_similar_items.argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, i64, C.c_int32, vp, vp, vp, vp]
    lib.invpref_top_users.argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, i64, vp, vp, C.c_int32, vp, vp, vp]
    for name in ("invpref_fold_in_users", "invpref_fold_in_items"):
        getattr(lib, name).argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, vp, vp, i64, C.c_double, C.c_int32, vp,
                                       vp, vp]
    for name in ("invpref_recommend_rows", "invpref_top_users_rows"):
        getattr(lib, name).argtypes = [C.POINTER(Desc), C.POINTER(Params), vp, vp, i64, vp, vp, C.c_int32, vp, vp, vp]
    lib.invpref_mask_scores.argtypes = [vp, i64, i64, vp, vp, vp, C.c_float, C.c_int32, vp]
    lib.invpref_hits_from_csr.argtypes = [vp, i64, C.c_int32, vp, vp, vp, vp, vp, vp]
    lib.invpref_mt_jump_bytes.argtypes = [C.POINTER(sz), C.POINTER(sz)]
    lib.invpref_mt_build_jumps.argtypes = [vp, sz, vp]
    lib.invpref_mt_randint.argtypes = [vp, C.c_int32, i64, i64, vp, vp, vp, vp, vp, sz, vp]
    lib.invpref_profile_enable.argtypes = [C.c_int]
    lib.invpref_profile_read.argtypes = [C.c_int, C.POINTER(C.c_float)]
    for name in EXPORTS:
        if os.environ.get("INVPREF_LIB") and not hasattr(lib, name):
            continue                     # an older variant build: entry points added since are simply absent
        fn = getattr(lib, name)
        if name not in ("invpref_strerror", "invpref_abi_version", "invpref_launch_count", "invpref_graph_launches"):
            fn.restype = C.c_int
    _lib = lib
    return lib


ABI_VERSION = 6
FOLD_IN_MAX_DIM = 128
ERR_ID_RANGE = -7


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().invpref_strerror(rc).decode()
        if rc == ERR_ID_RANGE:          # what the reference's nn.Embedding raises on CPU (models.py:449-455)
            raise IndexError(f"libinvpref_b200 {what}: {msg} (status {rc})")
        raise RuntimeError(f"libinvpref_b200 {what}: {msg} (status {rc})")


def ptr(t, dtype=None):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("libinvpref_b200 takes CUDA tensors only (no CPU fallback)")
    if not t.is_contiguous():
        raise RuntimeError("libinvpref_b200 takes contiguous tensors")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"expected {dtype}, got {t.dtype}")
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def make_desc(n_users, n_items, n_envs, dim, implicit, reg_only_embed, reg_env_embed) -> Desc:
    return Desc(int(n_users), int(n_items), int(n_envs), int(dim), int(bool(implicit)), int(bool(reg_only_embed)),
                int(bool(reg_env_embed)), 0)


def make_params(tensors) -> Params:
    """tensors: mapping or sequence in PARAM_FIELDS order of fp32 CUDA tensors."""
    if isinstance(tensors, dict):
        tensors = [tensors[k] for k in PARAM_FIELDS]
    p = Params()
    for k, t in zip(PARAM_FIELDS, tensors):
        setattr(p, k, ptr(t, torch.float32))
    return p


def workspace_bytes(desc: Desc, max_batch: int) -> int:
    out = C.c_size_t(0)
    check(load().invpref_workspace_bytes(C.byref(desc), int(max_batch), C.byref(out)), "workspace_bytes")
    return out.value


def plan_bytes(desc: Desc, max_batch: int) -> int:
    out = C.c_size_t(0)
    check(load().invpref_plan_bytes(C.byref(desc), int(max_batch), C.byref(out)), "plan_bytes")
    return out.value


def launch_count() -> int:
    return int(load().invpref_launch_count())


def profile_enable(max_steps: int) -> None:
    check(load().invpref_profile_enable(int(max_steps)), "profile_enable")


def profile_read_all():
    """[steps][phase] milliseconds of the recorded train steps (call after torch.cuda.synchronize())."""
    lib = load()
    out = []
    buf = (C.c_float * len(PHASES))()
    for s in range(lib.invpref_profile_steps()):
        check(lib.invpref_profile_read(s, buf), "profile_read")
        out.append([float(x) for x in buf])
    return out

"""GPU, every kernel instantiation and every segment-length regime of the train step against an fp64 reference.

How the library runs depends on two things: the table shape picks a template instantiation (``make_geometry`` maps D
to (VEC, NV) and K to the env capacity KT; the dispatch chains of upass.cu / bwd.cu / cluster.cu pick exact (D, K)
kernels, generic ones, the staged / ring kernels for NV * VEC <= 4 or the register kernels, and the unfused user side
when the per-CTA dE / dW slices do not fit), and the batch size picks the chunk size (``chunk_for``) that decides
which segments are pre-reduced in chunks and which go to the hot list.  This module runs each of those paths and
proves, with ``torch.profiler``, that the kernel a case names is the one that ran:

  1. geometry sweep: every (VEC, NV, KT) and every exact specialisation; train step (dense and lazy), the generic
     backward, forward / predict, and the re-assignment (plain and over the user-sorted view);
  2. segment regimes: every chunk_for band and its switch points, with segments of 1, 2, 2c, 2c + 1, 16c, 16c + 1,
     31c + 1 and 40c + 3 interactions on both sides (deferred / chunked, non-hot / hot), one-row and all-unique batches, B = 1, 2;
  3. saturated implicit inputs: |sigmoid argument| >= 25 and classifier logits that underflow exp for all but one
     class.

The reference is ``oracle.invpref_torch_cpu``'s op sequence run on CUDA tensors, in fp32 and in fp64.  Gates, per
tensor and norm-wise: err(ours, fp64) <= max(1e-5, 2 err(ref fp32, fp64)); losses within 1e-5 of the fp32 op sequence;
the Adam update where |g| > 1e-7; re-assignment bit-exact outside fp32 near-ties, histogram and diff count exact.
"""
import re
from collections import Counter

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from invpref_kdd_2022_b200 import _lib
from oracle import invpref_numpy as on
from oracle import invpref_torch_cpu as ot

pytestmark = pytest.mark.gpu

TOL = 1e-5
LR = 1e-2
COEF = dict(c_inv=0.8, c_ea=1.7, c_env=1.1, c_L2=0.6, c_L1=0.03)
HOT_CHUNKS = 16                     # common.cuh: segments with more chunks are reduced by a whole CTA


def _dev():
    return torch.device("cuda:0")


def _nerr(a, b):
    den = float(b.abs().max())
    return float((a - b).abs().max()) / (den if den > 0 else 1.0)


def chunk_for(B):
    """common.cuh chunk_for: the chunk size of a batch of B interactions."""
    if B >= 1 << 22:
        return 256
    c = 8
    while c < 128 and c * 32768 < B:
        c *= 2
    return c


def geometry(D, K):
    """common.cuh make_geometry: (VEC, NV, KT)."""
    if D % 4 == 0:
        vec, nv = 4, (1 if D <= 64 else (2 if D <= 128 else 4))
    elif D % 2 == 0:
        vec, nv = 2, (1 if D <= 32 else 2)
    else:
        vec, nv = 1, 4
    kt = 2 if K <= 2 else (4 if K <= 4 else (6 if K <= 6 else 8))
    return vec, nv, kt


def _launched(fn):
    """Runs fn() under torch.profiler; returns its result and a Counter of the CUDA kernels it launched (name ->
    number of launches), with bool template arguments written 0 / 1."""
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    norm = lambda n: re.sub(r"\btrue\b", "1", re.sub(r"\bfalse\b", "0", n))
    return out, Counter(norm(e.name()) for e in prof.profiler.kineto_results.events()
                        if e.device_type() == torch.autograd.DeviceType.CUDA)


def _assert_ran(names, expected, tag):
    """expected: kernel-name substrings, or (substring, n) for a kernel that must be launched exactly n times."""
    ours = sorted(n for n in names if "invpref::" in n)
    for want in expected:
        want, n = want if isinstance(want, tuple) else (want, None)
        got = sum(c for name, c in names.items() if want in name)
        assert got >= 1 if n is None else got == n, (tag, want, n, got, ours)


def _tables(U, I, K, D, seed):
    rng = np.random.default_rng(seed)
    p = {"Uinv": rng.normal(0, 0.1, (U, D)), "Iinv": rng.normal(0, 0.1, (I, D)), "Uenv": rng.normal(0, 0.3, (U, D)),
         "Ienv": rng.normal(0, 0.3, (I, D)), "E": rng.normal(0, 0.5, (K, D)), "W": rng.normal(0, 0.3, (K, D)),
         "b": rng.normal(0, 0.1, (K,))}
    return {k: torch.tensor(v.astype(np.float32), device=_dev()) for k, v in p.items()}


def _hot(init, implicit, lazy=False):
    from invpref_kdd_2022_b200.engine import HotPath
    return HotPath({k: v.clone() for k, v in init.items()}, implicit, False, True, lr=LR, lazy=lazy)


def _step(hp, batch, alpha, **kw):
    u, i, y, e, w = batch
    return hp.train_step(u, i, y, e, w, alpha=alpha, use_class_rw=True, use_rec_rw=True, **COEF, **kw)


def _check_step(tag, init, hp, grads, loss, batch, implicit, alpha, grad_vs_fp32=False):
    """One dense step from `init` against the reference op sequence in fp32 and fp64 (tolerance rule in the module
    docstring).  grad_vs_fp32: gradients also within 1e-5 of the fp32 run (where fp64 differs in semantics, e.g. a
    BCE argument that rounds to 1 in fp32)."""
    u, i, y, e, w = batch
    flags = on.Flags(implicit, False, True)
    hyp = on.Hyper(alpha=alpha, lr=LR, use_class_rw=True, use_rec_rw=True, **COEF)
    P = {k: v.clone().requires_grad_(True) for k, v in init.items()}
    ref = ot.CpuTrainer(P, flags, hyp).train_a_batch(u, i, y, e, w, alpha)
    loss = loss.double().cpu().numpy()
    assert np.isfinite(loss).all(), (tag, loss)
    for j, k in enumerate(on.LOSS_KEYS):
        assert abs(loss[j] - ref[k]) <= TOL * abs(ref[k]), (tag, k, loss[j], ref[k])
    P64 = {k: v.double().requires_grad_(True) for k, v in init.items()}
    tr64 = ot.CpuTrainer(P64, flags, hyp)
    tr64.opt.step = lambda *a, **k_: None
    tr64.train_a_batch(u, i, y.double(), e, w.double(), alpha)
    for k in on.PARAM_ORDER:
        assert bool(torch.isfinite(grads[k]).all()) and bool(torch.isfinite(hp.params[k]).all()), (tag, k)
        g64 = P64[k].grad
        err_ours, err_ref = _nerr(grads[k].double(), g64), _nerr(P[k].grad.double(), g64)
        assert err_ours <= max(TOL, 2 * err_ref), (tag, k, err_ours, err_ref)
        if grad_vs_fp32:
            assert _nerr(grads[k], P[k].grad) <= TOL, (tag, k, _nerr(grads[k], P[k].grad))
        ok = P[k].grad.abs() > 1e-7                       # Adam's first step is -lr g / (|g| + eps)
        if bool(ok.any()):
            d_ours, d_ref = (hp.params[k] - init[k])[ok], (P[k].detach() - init[k])[ok]
            assert float((d_ours - d_ref).abs().max()) <= 1e-3 * LR, (tag, k)


def _check_backward(tag, hp, init, batch, implicit, alpha, expected):
    """invpref_backward (forward kernel + EPI_ACCUM rows kernels): gradients of
    sum(ga s_inv) + sum(gb s_env) + sum(gc logp) against autograd of the reference forward."""
    u, i, _, e, _ = batch
    B, K = u.numel(), init["E"].shape[0]
    g = torch.Generator(device=_dev()).manual_seed(B + K)
    ga, gb = torch.randn(B, device=_dev(), generator=g), torch.randn(B, device=_dev(), generator=g)
    gc = torch.randn((B, K), device=_dev(), generator=g)
    grads = {k: torch.zeros_like(v) for k, v in init.items()}
    _, names = _launched(lambda: hp.backward(u, i, e, alpha, ga, gb, gc, grads))
    _assert_ran(names, expected, tag + "/backward")
    ref = {}
    for dt in (torch.float32, torch.float64):
        P = {k: v.to(dt, copy=True).requires_grad_(True) for k, v in init.items()}
        s_inv, s_env, logp = ot.forward(P, u, i, e, alpha, implicit)
        ((s_inv * ga.to(dt)).sum() + (s_env * gb.to(dt)).sum() + (logp * gc.to(dt)).sum()).backward()
        ref[dt] = {k: P[k].grad for k in on.PARAM_ORDER}
    for k in on.PARAM_ORDER:
        g64 = ref[torch.float64][k]
        err_ours, err_ref = _nerr(grads[k].double(), g64), _nerr(ref[torch.float32][k].double(), g64)
        assert err_ours <= max(TOL, 2 * err_ref), (tag, "backward", k, err_ours, err_ref)


# ------------------------------------------------------------------------------------------------------------------
# 1. geometry sweep
#
# Each case names the kernels its shape must launch.  {L} is the lazy flag of the user pass (LAZY) and of the item
# pass (STASH: it reads the caught-up user rows from the stash); it is 0 on the unfused shapes, where lazy Adam is not
# available and the lazy run is the dense one.  Columns: D, K, implicit, user-pass rows kernel (None: unfused, the
# forward kernel and the generic user-side rows kernel run instead), item-pass rows kernel, item-pass chunks kernel,
# re-assignment kernel.  (VEC, NV, KT) of the generic dispatch (forward, chunks of the user pass) follow geometry().
GEOMETRY_CASES = [
    # VEC 1, NV 4 (odd D): 1 of 4 vectors (D = 1), 2 of 4 + one lane (33), 3 of 4 but the last lane (63)
    (1, 2, True, "upass_rows_staged_kernel<1, 4, 2, 0, {L}, 0>", "bwd_rows_ring_kernel<1, 4, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<1, 4, {L}, 0, 64>", "cluster_kernel<1, 4, 2, 0>"),
    (33, 3, False, "upass_rows_staged_kernel<1, 4, 4, 0, {L}, 0>", "bwd_rows_ring_kernel<1, 4, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<1, 4, {L}, 0, 64>", "cluster_kernel<1, 4, 4, 0>"),
    (63, 5, True, "upass_rows_staged_kernel<1, 4, 6, 0, {L}, 0>", "bwd_rows_ring_kernel<1, 4, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<1, 4, {L}, 0, 64>", "cluster_kernel<1, 4, 6, 0>"),
    (63, 6, False, "upass_rows_staged_kernel<1, 4, 6, 0, {L}, 0>", "bwd_rows_ring_kernel<1, 4, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<1, 4, {L}, 0, 64>", "cluster_kernel<1, 4, 6, 0>"),
    (33, 8, True, "upass_rows_staged_kernel<1, 4, 8, 0, {L}, 0>", "bwd_rows_ring_kernel<1, 4, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<1, 4, {L}, 0, 64>", "cluster_kernel<1, 4, 8, 0>"),
    # VEC 2, NV 1 (even D <= 32, not a multiple of 4)
    (30, 2, True, "upass_rows_staged_kernel<2, 1, 2, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 1, 0, {L}, 0, 32>",
     "bwd_chunks_ring_kernel<2, 1, {L}, 0, 32>", "cluster_kernel<2, 1, 2, 0>"),
    (14, 4, False, "upass_rows_staged_kernel<2, 1, 4, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 1, 0, {L}, 0, 32>",
     "bwd_chunks_ring_kernel<2, 1, {L}, 0, 32>", "cluster_kernel<2, 1, 4, 0>"),
    (2, 6, False, "upass_rows_staged_kernel<2, 1, 6, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 1, 0, {L}, 0, 32>",
     "bwd_chunks_ring_kernel<2, 1, {L}, 0, 32>", "cluster_kernel<2, 1, 6, 0>"),
    (6, 8, True, "upass_rows_staged_kernel<2, 1, 8, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 1, 0, {L}, 0, 32>",
     "bwd_chunks_ring_kernel<2, 1, {L}, 0, 32>", "cluster_kernel<2, 1, 8, 0>"),
    # VEC 2, NV 2 (even D 34..62, not a multiple of 4): the second vector partly filled
    (34, 2, False, "upass_rows_staged_kernel<2, 2, 2, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 2, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<2, 2, {L}, 0, 64>", "cluster_kernel<2, 2, 2, 0>"),
    (50, 3, True, "upass_rows_staged_kernel<2, 2, 4, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 2, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<2, 2, {L}, 0, 64>", "cluster_kernel<2, 2, 4, 0>"),
    (62, 6, False, "upass_rows_staged_kernel<2, 2, 6, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 2, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<2, 2, {L}, 0, 64>", "cluster_kernel<2, 2, 6, 0>"),
    (46, 8, True, "upass_rows_staged_kernel<2, 2, 8, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 2, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<2, 2, {L}, 0, 64>", "cluster_kernel<2, 2, 8, 0>"),
    # VEC 4, NV 1, generic: D not 40 / 64, or 40 / 64 with a K that misses the exact kernels
    (44, 3, False, "upass_rows_staged_kernel<4, 1, 4, 0, {L}, 0>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 0, 64>", "cluster_kernel<4, 1, 4, 0>"),
    (60, 7, True, "upass_rows_staged_kernel<4, 1, 8, 0, {L}, 0>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 0, 64>", "cluster_kernel<4, 1, 8, 0>"),
    (40, 3, True, "upass_rows_staged_kernel<4, 1, 4, 0, {L}, 0>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 0, 64>", "cluster_kernel<4, 1, 4, 0>"),
    (64, 7, False, "upass_rows_staged_kernel<4, 1, 8, 0, {L}, 0>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 0, 64>", "cluster_kernel<4, 1, 8, 0>"),
    # exact D = 64 (K = KT): user pass and re-assignment for K = 2, 4, 6, 8, item pass for K = 2, 4, 6
    (64, 2, True, "upass_rows_staged_kernel<4, 1, 2, 0, {L}, 64>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 2, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 2, 64>", "cluster_kernel<4, 1, 2, 64>"),
    (64, 4, False, "upass_rows_staged_kernel<4, 1, 4, 0, {L}, 64>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 4, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 4, 64>", "cluster_kernel<4, 1, 4, 64>"),
    (64, 6, True, "upass_rows_staged_kernel<4, 1, 6, 0, {L}, 64>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 6, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 6, 64>", "cluster_kernel<4, 1, 6, 64>"),
    (64, 8, False, "upass_rows_staged_kernel<4, 1, 8, 0, {L}, 64>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 0, 64>", "cluster_kernel<4, 1, 8, 64>"),
    # exact D = 40: user pass and re-assignment for K = 2, 4, 5, 6, 8, item pass for K = 2, 5, 6 (K = 5 next to the
    # g-pack width switch at K = 6)
    (40, 2, False, "upass_rows_staged_kernel<4, 1, 2, 0, {L}, 40>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 2, 40>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 2, 40>", "cluster_kernel<4, 1, 2, 40>"),
    (40, 4, True, "upass_rows_staged_kernel<4, 1, 4, 0, {L}, 40>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 0, 64>", "cluster_kernel<4, 1, 4, 40>"),
    (40, 5, False, "upass_rows_staged_kernel<4, 1, 5, 0, {L}, 40>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 5, 40>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 5, 40>", "cluster_kernel<4, 1, 5, 40>"),
    (40, 6, True, "upass_rows_staged_kernel<4, 1, 6, 0, {L}, 40>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 6, 40>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 6, 40>", "cluster_kernel<4, 1, 6, 40>"),
    (40, 8, False, "upass_rows_staged_kernel<4, 1, 8, 0, {L}, 40>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 0, 64>",
     "bwd_chunks_ring_kernel<4, 1, {L}, 0, 64>", "cluster_kernel<4, 1, 8, 40>"),
    # VEC 4, NV 2 (D 68..128): register kernels, the last vector partly filled except at D = 128
    (68, 2, True, "upass_rows_kernel<4, 2, 2, 0, {L}>", "bwd_rows_kernel<4, 2, 0, {L}>", "bwd_chunks_kernel<4, 2, {L}>",
     "cluster_kernel<4, 2, 2, 0>"),
    (96, 4, False, "upass_rows_kernel<4, 2, 4, 0, {L}>", "bwd_rows_kernel<4, 2, 0, {L}>", "bwd_chunks_kernel<4, 2, {L}>",
     "cluster_kernel<4, 2, 4, 0>"),
    (124, 5, True, "upass_rows_kernel<4, 2, 6, 0, {L}>", "bwd_rows_kernel<4, 2, 0, {L}>", "bwd_chunks_kernel<4, 2, {L}>",
     "cluster_kernel<4, 2, 6, 0>"),
    (68, 7, True, "upass_rows_kernel<4, 2, 8, 0, {L}>", "bwd_rows_kernel<4, 2, 0, {L}>", "bwd_chunks_kernel<4, 2, {L}>",
     "cluster_kernel<4, 2, 8, 0>"),
    (100, 8, False, None, "bwd_rows_kernel<4, 2, 0, {L}>", "bwd_chunks_kernel<4, 2, {L}>", "cluster_kernel<4, 2, 8, 0>"),
    # VEC 4, NV 4 (D 132..256)
    (132, 2, False, "upass_rows_kernel<4, 4, 2, 0, {L}>", "bwd_rows_kernel<4, 4, 0, {L}>",
     "bwd_chunks_kernel<4, 4, {L}>", "cluster_kernel<4, 4, 2, 0>"),
    (200, 3, True, "upass_rows_kernel<4, 4, 4, 0, {L}>", "bwd_rows_kernel<4, 4, 0, {L}>",
     "bwd_chunks_kernel<4, 4, {L}>", "cluster_kernel<4, 4, 4, 0>"),
    (132, 5, True, "upass_rows_kernel<4, 4, 6, 0, {L}>", "bwd_rows_kernel<4, 4, 0, {L}>",
     "bwd_chunks_kernel<4, 4, {L}>", "cluster_kernel<4, 4, 6, 0>"),
    (252, 6, False, None, "bwd_rows_kernel<4, 4, 0, {L}>", "bwd_chunks_kernel<4, 4, {L}>", "cluster_kernel<4, 4, 6, 0>"),
    (136, 8, True, None, "bwd_rows_kernel<4, 4, 0, {L}>", "bwd_chunks_kernel<4, 4, {L}>", "cluster_kernel<4, 4, 8, 0>"),
]


def _power_law_batch(U, I, N, K, implicit, seed):
    """Ids as in the synthetic workloads: user 0 has a chunked segment, item 0 a hot one (chunk 8 at these sizes)."""
    rng = np.random.default_rng(seed)
    u = np.floor(U * rng.random(N) ** 1.5).astype(np.int64)
    i = np.floor(I * rng.random(N) ** 3).astype(np.int64)
    y = (rng.integers(0, 2, N) if implicit else rng.integers(1, 6, N)).astype(np.float32)
    e = rng.integers(0, K, N).astype(np.int64)
    w = (0.25 + rng.random(N)).astype(np.float32)
    return tuple(torch.tensor(a, device=_dev()) for a in (u, i, y, e, w))


@pytest.mark.parametrize("case", GEOMETRY_CASES, ids=lambda c: f"D{c[0]}-K{c[1]}-{'imp' if c[2] else 'exp'}")
def test_geometry_dispatch_matches_fp64(case):
    D, K, implicit, up_k, it_k, ch_k, cl_k = case
    V, NV, KT = geometry(D, K)
    U, I, N = 300, 200, 24011
    tag = f"D{D}K{K}"
    init = _tables(U, I, K, D, 7 * D + K)
    batch = _power_law_batch(U, I, N, K, implicit, D + 13 * K)
    alpha = 1.3

    # dense step, gradients exported
    hp = _hot(init, implicit)
    assert (hp.lazy_supported) == (up_k is not None), tag
    grads = {k: torch.zeros_like(v) for k, v in init.items()}
    loss, names = _launched(lambda: _step(hp, batch, alpha, grads_out=grads).clone())
    # unfused: the user side launches the same generic rows / chunks kernels as the item pass, so each runs twice
    user = ([up_k, f"upass_chunks_kernel<{V}, {NV}, {KT}, {{L}}>"] if up_k is not None else
            [f"fwd_train_kernel<{V}, {NV}, {KT}>", (it_k, 2), (ch_k, 2)])
    fmt = lambda s, L: (s[0].format(L=L), s[1]) if isinstance(s, tuple) else s.format(L=L)
    _assert_ran(names, [fmt(s, 0) for s in user + [it_k, ch_k]] + [f"sweep_kernel<{V}, {NV}>"], tag + "/dense")
    _check_step(tag, init, hp, grads, loss, batch, implicit, alpha)

    # lazy == dense bit for bit (the multi-step replay is test_lazy_steps_are_bitwise_dense)
    hz = _hot(init, implicit, lazy=True)
    lz = int(hz.lazy)
    l0, names = _launched(lambda: _step(hz, batch, alpha).clone())
    _assert_ran(names, [fmt(s, lz) for s in user + [it_k, ch_k]], tag + "/lazy")
    _, names = _launched(hz.flush)
    if lz:
        _assert_ran(names, [f"flush_kernel<{V}, {NV}>"], tag + "/flush")
    assert torch.equal(loss, l0), tag
    for k in on.PARAM_ORDER:
        assert torch.equal(hp.params[k], hz.params[k]), (tag, k)
        assert torch.equal(hp.m[k], hz.m[k]) and torch.equal(hp.v[k], hz.v[k]), (tag, k)

    # generic backward (forward kernel + EPI_ACCUM rows kernels on both sides)
    hb = _hot(init, implicit)
    _check_backward(tag, hb, init, batch, implicit, alpha,
                    [f"fwd_train_kernel<{V}, {NV}, {KT}>", f"bwd_rows_kernel<{V}, {NV}, 1, 0>", ch_k.format(L=0)])

    # forward and predict
    u, i, y, e, _ = batch
    (s_inv, s_env, logp), names = _launched(lambda: hb.forward(u, i, e))
    _assert_ran(names, [f"fwd_only_kernel<{V}, {NV}, {KT}>"], tag + "/forward")
    pred, names = _launched(lambda: hb.predict(u, i))
    _assert_ran(names, [f"predict_kernel<{V}, {NV}>"], tag + "/predict")
    with torch.no_grad():
        ref = {dt: ot.forward({k: v.to(dt) for k, v in init.items()}, u, i, e, 0.0, implicit)
               for dt in (torch.float32, torch.float64)}
        z = {dt: (init["Uinv"].to(dt)[u] * init["Iinv"].to(dt)[i]).sum(1) for dt in (torch.float32, torch.float64)}
    for j, ours in enumerate((s_inv, s_env, logp)):
        r64, r32 = ref[torch.float64][j], ref[torch.float32][j]
        assert _nerr(ours.double(), r64) <= max(TOL, 2 * _nerr(r32.double(), r64)), (tag, "forward", j)
    assert _nerr(pred.double(), z[torch.float64]) <= max(TOL, 2 * _nerr(z[torch.float32].double(), z[torch.float64]))

    # re-assignment with the tie-break table, plain and over the user-sorted view.  The env-aware tables are scaled so
    # that the env-aware score has a spread of about 1: the K distances are apart, few samples are fp32 near-ties.
    f = (1.0 / (0.045 * D ** 0.5)) ** (1.0 / 3.0)
    sep = {k: v * f if k in ("Uenv", "Ienv", "E") else v for k, v in init.items()}
    hc = _hot(sep, implicit)
    eps = torch.tensor(on.init_eps(K), device=_dev())
    pidx = torch.tensor(np.random.default_rng(K + D).integers(0, eps.shape[0], N), device=_dev())
    (new, hist, diff), names = _launched(lambda: hc.cluster(u, i, y, pidx, eps, e))
    _assert_ran(names, [cl_k], tag + "/cluster")
    view = hc.sorted_view(u, i, y)
    (new_s, hist_s, diff_s), names = _launched(lambda: hc.cluster_sorted(view, pidx, eps, e))
    _assert_ran(names, [cl_k.replace("cluster_kernel", "cluster_sorted_kernel")], tag + "/cluster_sorted")
    assert torch.equal(new, new_s) and torch.equal(hist, hist_s) and torch.equal(diff, diff_s), tag
    with torch.no_grad():
        cols = []
        for k in range(K):
            _, s_k, _ = ot.forward(sep, u, i, torch.full_like(e, k), 0.0, implicit)
            cols.append(torch.nn.functional.binary_cross_entropy(s_k, y, reduction="none") if implicit
                        else (s_k - y) ** 2)
        dist = torch.stack(cols, 1) + eps[pidx]
    ties = on.near_tie_mask(dist.cpu().numpy())
    mism = (new != torch.argmin(dist, 1)).cpu().numpy()
    assert not (mism & ~ties).any(), (tag, int((mism & ~ties).sum()))
    assert ties.mean() < 0.05, (tag, float(ties.mean()))
    assert torch.equal(hist, torch.bincount(new, minlength=K)) and int(diff) == int((new != e).sum()), tag


# (D, K) where the "thirds" sequence below finds lazy != dense: the lazy and the dense instantiations of the fused user
# pass are the same source, but the compiler contracts mul + add into FMAs differently in the two, and a few
# interactions' gradients differ by one ulp (the user and the item row of each).  Built with -fmad=false for upass*.cu
# the two agree on every case here, at 3 % of the C5 step; the fix has to pin only the expressions that differ.
LAZY_FMA_CONTRACTION_DIFFERS = {(64, 8), (68, 2)}


@pytest.mark.parametrize("seq", ["halves", "thirds"])
@pytest.mark.parametrize("case", GEOMETRY_CASES, ids=lambda c: f"D{c[0]}-K{c[1]}-{'imp' if c[2] else 'exp'}")
def test_lazy_steps_are_bitwise_dense(case, seq, request):
    """Three steps, lazy against dense Adam; losses, tables and moments must be identical bit for bit.
    halves: the second batch has only the users below U / 2 (the others are replayed in the user pass of the third
    step), the third only those from U / 4 on (the first quarter is replayed by flush()).
    thirds: full batch, its first third, full batch (every user in every step: the lazy kernels replay nothing, so
    they must round every interaction exactly as the dense ones do)."""
    D, K, implicit = case[:3]
    if seq == "thirds" and (D, K) in LAZY_FMA_CONTRACTION_DIFFERS:
        request.applymarker(pytest.mark.xfail(strict=True, reason="lazy / dense user pass: different FMA contraction"))
    U, I, N = 300, 200, 24011
    init = _tables(U, I, K, D, 7 * D + K)
    batch = _power_law_batch(U, I, N, K, implicit, D + 13 * K)
    if seq == "halves":
        steps = ((batch, 1.3), (tuple(t[batch[0] < U // 2] for t in batch), 0.9),
                 (tuple(t[batch[0] >= U // 4] for t in batch), 0.4))
    else:
        steps = ((batch, 1.3), (tuple(t[: N // 3] for t in batch), 0.9), (batch, 0.4))
    res = {}
    for lazy in (False, True):
        h = _hot(init, implicit, lazy=lazy)
        losses = [_step(h, b, a).clone() for b, a in steps]
        h.flush()
        res[lazy] = (torch.stack(losses), h)
    assert torch.equal(res[False][0], res[True][0]), case[:3]
    hd, hz = res[False][1], res[True][1]
    for k in on.PARAM_ORDER:
        assert torch.equal(hd.params[k], hz.params[k]), (case[:3], k)
        assert torch.equal(hd.m[k], hz.m[k]) and torch.equal(hd.v[k], hz.v[k]), (case[:3], k)


# ------------------------------------------------------------------------------------------------------------------
# 2. segment regimes
#
# chunk_for bands: 8 up to 2^18, then 16, 32, 64, 128 up to 2^22, 256 from 2^22 on; both sides of each switch.
BATCHES = (262144, 262145, 300000, 600000, 1200000, 2500000, 4194303, 4194304)
# (D, K, user-pass rows kernel, item-pass rows kernel, item-pass chunks kernel, user-pass chunks kernel): the exact
# C5 kernels, and one generic geometry of part 1 (staged / ring, two vectors per lane)
REGIME_GEOMS = {
    "d64k4": (64, 4, "upass_rows_staged_kernel<4, 1, 4, 0, {L}, 64>", "bwd_rows_ring_kernel<4, 1, 0, {L}, 4, 64>",
              "bwd_chunks_ring_kernel<4, 1, {L}, 4, 64>", "upass_chunks_kernel<4, 1, 4, {L}>"),
    "d50k3": (50, 3, "upass_rows_staged_kernel<2, 2, 4, 0, {L}, 0>", "bwd_rows_ring_kernel<2, 2, 0, {L}, 0, 64>",
              "bwd_chunks_ring_kernel<2, 2, {L}, 0, 64>", "upass_chunks_kernel<2, 2, 4, {L}>"),
}


def _engineered_column(B, lengths, n_bg, rng):
    """Rows 0..len(lengths)-1 get exactly lengths[r] interactions; the rest of the batch goes to background rows
    drawn from the reserved range [len(lengths), len(lengths) + n_bg), shuffled."""
    eng = np.repeat(np.arange(len(lengths), dtype=np.int64), lengths)
    rest = B - len(eng)
    assert rest >= 0
    col = np.concatenate([eng, len(lengths) + rng.integers(0, n_bg, rest)])
    rng.shuffle(col)
    return col


def _regime_batch(kind, B, K, seed):
    rng = np.random.default_rng(seed)
    c = chunk_for(B)
    if kind == "bands":
        lengths = [1, 2, 2 * c, 2 * c + 1, 16 * c, 16 * c + 1, 31 * c + 1, 40 * c + 3]
        U, I = len(lengths) + 65536, len(lengths) + 16384
        u = _engineered_column(B, lengths, U - len(lengths), rng)
        i = _engineered_column(B, lengths, I - len(lengths), rng)
    elif kind == "one_row":               # every interaction on user 3 and item 5: one segment per side
        U, I = 8, 8
        u, i = np.full(B, 3, np.int64), np.full(B, 5, np.int64)
    elif kind == "unique":                # every id once
        U, I = B, B
        u, i = rng.permutation(B).astype(np.int64), rng.permutation(B).astype(np.int64)
    else:                                 # B = 1, 2: one user, one item each
        U, I = 8, 8
        u, i = np.full(B, 3, np.int64), 5 + np.arange(B, dtype=np.int64)
    y = rng.integers(1, 6, B).astype(np.float32)
    e = rng.integers(0, K, B).astype(np.int64)
    w = (0.25 + rng.random(B)).astype(np.float32)
    return U, I, u, i, tuple(torch.tensor(a, device=_dev()) for a in (u, i, y, e, w))


def _plan_counters(hp, plan, U, I, B):
    """counters[0..4] (n_seg, n_chunks, -, n_ranges, n_hot) of the user and the item side of a plan."""
    user_side = _lib.plan_bytes(_lib.make_desc(U, U, hp.n_envs, hp.dim, 0, 0, 0), B) // 2
    return (plan[:64].view(torch.int32).cpu().numpy()[:5],
            plan[user_side:user_side + 64].view(torch.int32).cpu().numpy()[:5])


def _expected_counters(ids, c):
    cnt = np.bincount(ids)
    cnt = cnt[cnt > 0]
    long = cnt > 2 * c
    chunks = -(-cnt // c) * long
    return len(cnt), int(chunks.sum()), int((chunks > HOT_CHUNKS).sum())


def _run_regime(kind, B, geo):
    D, K, up_k, it_k, ch_k, uch_k = REGIME_GEOMS[geo]
    V, NV, KT = geometry(D, K)
    implicit = False
    U, I, u_np, i_np, batch = _regime_batch(kind, B, K, B + D)
    c = chunk_for(B)
    tag = f"{kind}/B{B}/{geo}"
    init = _tables(U, I, K, D, B % 9973 + D)
    alpha = 1.1
    hp = _hot(init, implicit)
    u, i = batch[0], batch[1]
    plan = hp.new_plan(u, i)
    cu, ci = _plan_counters(hp, plan, U, I, B)
    for side, ids, got in (("user", u_np, cu), ("item", i_np, ci)):
        n_seg, n_chunks, n_hot = _expected_counters(ids, c)
        assert (got[0], got[1], got[4]) == (n_seg, n_chunks, n_hot), (tag, side, got, (n_seg, n_chunks, n_hot))
    grads = {k: torch.zeros_like(v) for k, v in init.items()}
    loss, names = _launched(lambda: _step(hp, batch, alpha, plan=plan, grads_out=grads).clone())
    _assert_ran(names, [s.format(L=0) for s in (up_k, it_k, ch_k, uch_k)], tag)
    _check_step(tag, init, hp, grads, loss, batch, implicit, alpha)

    hz = _hot(init, implicit, lazy=True)
    assert hz.lazy
    lz, names = _launched(lambda: _step(hz, batch, alpha, plan=plan).clone())
    _assert_ran(names, [s.format(L=1) for s in (up_k, it_k, ch_k, uch_k)], tag + "/lazy")
    hz.flush()
    assert torch.equal(loss, lz), tag
    for k in on.PARAM_ORDER:
        assert torch.equal(hp.params[k], hz.params[k]), (tag, k)
        assert torch.equal(hp.m[k], hz.m[k]) and torch.equal(hp.v[k], hz.v[k]), (tag, k)
    del hp, hz, grads

    _check_backward(tag, _hot(init, implicit), init, batch, implicit, alpha,
                    [f"fwd_train_kernel<{V}, {NV}, {KT}>", f"bwd_rows_kernel<{V}, {NV}, 1, 0>", ch_k.format(L=0)])
    torch.cuda.empty_cache()


@pytest.mark.parametrize("geo", sorted(REGIME_GEOMS))
@pytest.mark.parametrize("B", BATCHES)
def test_segment_regimes_match_fp64(B, geo):
    """Per side: segments of 1 and 2 interactions, the longest deferred segment (2c) and the shortest chunked one
    (2c + 1), the last non-hot segment (16c: 16 chunks) and the first hot one (16c + 1: 17 chunks, so a CTA's groups
    9-15 get no slice), a hot segment of 32 chunks (31c + 1: every group of the CTA sums two, group 15's second one is
    the one-interaction tail), one of 41 chunks (not a multiple of 16), and background rows; the plan's segment,
    chunk and hot-list counts are checked against the batch."""
    _run_regime("bands", B, geo)


@pytest.mark.parametrize("geo", sorted(REGIME_GEOMS))
@pytest.mark.parametrize("kind,B", [("one_row", 262145), ("unique", 300000), ("tiny", 1), ("tiny", 2)])
def test_degenerate_batches_match_fp64(kind, B, geo):
    """One user and one item for the whole batch (one segment spans every cost range of the ring kernel; 16 385
    chunks: more than the user-pass chunks kernel's 148 CTAs x 16 groups), every id unique (no chunk anywhere), and
    batches of one and two interactions."""
    _run_regime(kind, B, geo)


# ------------------------------------------------------------------------------------------------------------------
# 3. saturated implicit inputs and env classifier
def _saturated_tables(U, I, K, D, seed):
    """Rank-one tables along q = 1 / sqrt(D): z1 = a_u c_i, z2 = b_u d_i f_k with |z1|, |z2| in [27, 49] (sigmoid
    rounds to 0 or 1 in fp32, away from the 14-19 band where one ulp decides), classifier logits a_u c_i w_k + b_k
    with adjacent w_k 4 apart: logits more than 100 apart, exp underflows for every class but the largest."""
    rng = np.random.default_rng(seed)
    q = np.full(D, 1.0 / np.sqrt(D))
    sgn = lambda n: rng.choice([-1.0, 1.0], n)
    a, c = rng.uniform(5.2, 7.0, U) * sgn(U), rng.uniform(5.2, 7.0, I) * sgn(I)
    bu, di, fk = rng.uniform(3.0, 3.6, U) * sgn(U), rng.uniform(3.0, 3.6, I) * sgn(I), rng.uniform(3.0, 3.6, K) * sgn(K)
    wk = 4.0 * (np.arange(K) - (K - 1) / 2.0)
    p = {"Uinv": a[:, None] * q, "Iinv": c[:, None] * q, "Uenv": bu[:, None] * q, "Ienv": di[:, None] * q,
         "E": np.repeat(fk[:, None], D, 1), "W": np.repeat(wk[:, None], D, 1), "b": rng.normal(0, 0.2, K)}
    p = {k: v + rng.normal(0, 1e-4, v.shape) for k, v in p.items()}
    return {k: torch.tensor(v.astype(np.float32), device=_dev()) for k, v in p.items()}


@pytest.mark.parametrize("D,K,alpha", [(64, 4, 10.0), (40, 6, 3.0), (33, 8, 10.0), (96, 5, 10.0)])
def test_saturated_implicit_step_matches_fp32_semantics(D, K, alpha):
    """BCE at |z| >= 25 (log clamped at -100, x(1 - x) clamped at 1e-12, as nn.BCELoss does in fp32) and a softmax
    whose exponentials underflow: losses equal the reference's fp32 op sequence, gradients follow both gates, every
    output is finite."""
    U, I, N = 300, 200, 24011
    tag = f"sat/D{D}K{K}"
    init = _saturated_tables(U, I, K, D, D * K)
    batch = _power_law_batch(U, I, N, K, True, D + K)
    u, i, _, e, _ = batch
    with torch.no_grad():
        P = {k: v.double() for k, v in init.items()}
        pref = P["Uinv"][u] * P["Iinv"][i]
        z1, z2 = pref.sum(1), (P["Uenv"][u] * P["Ienv"][i] * P["E"][e]).sum(1)
        lg = torch.sort(pref @ P["W"].T + P["b"], 1).values
    assert bool((z1.abs() >= 25).all()) and bool((z2.abs() >= 25).all()), tag
    assert bool((lg[:, -1] - lg[:, 0] > 100).all()) and bool((lg[:, -1] - lg[:, -2] > 104).all()), tag
    hp = _hot(init, True)
    grads = {k: torch.zeros_like(v) for k, v in init.items()}
    loss = _step(hp, batch, alpha, grads_out=grads).clone()
    _check_step(tag, init, hp, grads, loss, batch, True, alpha, grad_vs_fp32=True)
    for k in on.PARAM_ORDER:
        assert bool(torch.isfinite(hp.m[k]).all()) and bool(torch.isfinite(hp.v[k]).all()), (tag, k)
    s_inv, s_env, logp = hp.forward(u, i, e)
    assert bool(torch.isfinite(s_inv).all() and torch.isfinite(s_env).all() and torch.isfinite(logp).all()), tag

#!/usr/bin/env python
"""CUDA-event timing of the streaming top-k kernel (eval.cu) behind ``invpref_eval_topk``, ``invpref_recommend``,
``invpref_similar_items`` and ``invpref_top_users``.  GPU only.

    python tools/time_topk.py [--baseline-lib OTHER.so] [--repeats R] [--out FILE]

Shapes: the evaluator's calls as the drivers make them (Yahoo-implicit, MovieLens, MIND with its item pool), the C5
catalogue (1 M items, D 64) at b in {1, 256, 4096, 65536} and k in {50, 256}, and an adversarial stream whose scores
ascend with the item id (every item tile raises the threshold).  Then the item-to-item and item-to-user calls: the
MIND item graph (similar_items of all 51 283 items, k 50, D 40), the C5 item graph (all 1 M items), single C5 item
queries (b 1 and 256), top_users of 1 024 items over 10 M users (k 100, D 64), and the row-norm kernel alone on the C5
item table.  Per shape: microseconds per call, queries per second and the fraction of the fp32 FMA issue bound
(b * n * D FMAs over SMs x 128 lanes x the maximum SM clock); the norm kernel reports its read bandwidth instead.
``--baseline-lib``: also times another build of the library (e.g. the parent commit's) on the evaluator and
recommend shapes, on the same inputs, alternating the two builds ``--repeats`` times (medians and every repeat are
stored).  Where the [b, I] matrix fits in 16 GiB the step-by-step device path (``predict`` GEMM,
``invpref_mask_scores`` for the evaluator's lists, ``torch.topk``) is timed as well.  ``--commit``: a label of the
source tree measured, stored in the output.  The tables are fresh random normals per shape; the C5 tables (256 MB,
2.5 GB) are larger than L2, the dataset ones fit in it.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from invpref_kdd_2022_b200 import _lib  # noqa: E402
from invpref_kdd_2022_b200.dataloader import user_item_csr  # noqa: E402
from invpref_kdd_2022_b200.engine import HotPath  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_clock_max_mhz": float(out[2]),
            "sm_clock_mhz_at_query": float(out[3])}


def timed(fn, budget_s=0.3, warmup=2):
    """Mean microseconds per call after `warmup` calls, over enough calls to fill about `budget_s` (at least 1)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    once = e0.elapsed_time(e1) / 1e3
    reps = max(1, min(200, int(budget_s / max(once, 1e-6))))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def kernel_us(fn, kernel, n=20):
    """Mean device time in microseconds of the kernels whose name contains `kernel`, over `n` calls of fn (after 2
    warm-up calls), from torch.profiler's CUDA activity records."""
    from torch.profiler import ProfilerActivity, profile
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if kernel in e.name and e.device_type == torch.autograd.DeviceType.CUDA]
    if len(ev) != n:
        raise RuntimeError(f"expected {n} launches of {kernel}, the profiler saw {len(ev)}")
    return sum(e.time_range.elapsed_us() for e in ev) / n


def lists(rng, n_users, n_items, mean, dev):
    """Ascending unique item lists of about `mean` entries per user, as int64 CSR on the device."""
    u = np.repeat(np.arange(n_users), rng.poisson(mean, n_users))
    off, items = user_item_csr(u, rng.integers(0, n_items, u.size), n_users)
    return torch.from_numpy(off).to(dev), torch.from_numpy(items if items.size else np.zeros(1, np.int64)).to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None)
    ap.add_argument("--repeats", type=int, default=1)
    ap.add_argument("--out", default=None)
    ap.add_argument("--commit", default=None)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    info = gpu_info()
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    fma_per_s = n_sm * 128 * info["sm_clock_max_mhz"] * 1e6
    base = None
    if args.baseline_lib:
        base = C.CDLL(args.baseline_lib)
        for fn in ("invpref_eval_topk", "invpref_recommend"):
            getattr(base, fn).argtypes = getattr(_lib.load(), fn).argtypes
            getattr(base, fn).restype = C.c_int
    rng = np.random.default_rng(0)
    # kind, name, catalogue rows, D, b, k, implicit, mask mean, pool mean, scores ascending with the catalogue id
    shapes = [("eval", "yahoo_implicit_eval", 1000, 40, 1024, 7, True, 20, 0, False),
              ("eval", "movielens_eval", 3706, 40, 2048, 30, True, 100, 0, False),
              ("eval", "mind_eval", 51283, 40, 256, 40, True, 10, 100, False)]
    shapes += [("recommend", f"c5_b{b}_k{k}", 1_000_000, 64, b, k, False, 0, 0, False) for b in (1, 256, 4096, 65536)
               for k in (50, 256)]
    shapes += [("recommend", "c5_ascending_b4096_k256", 1_000_000, 64, 4096, 256, False, 0, 0, True)]
    shapes += [("similar", "mind_similar_all_k50", 51283, 40, 51283, 50, False, 0, 0, False),
               ("similar", "c5_similar_b1_k50", 1_000_000, 64, 1, 50, False, 0, 0, False),
               ("similar", "c5_similar_b256_k50", 1_000_000, 64, 256, 50, False, 0, 0, False),
               ("similar", "c5_similar_all_k50", 1_000_000, 64, 1_000_000, 50, False, 0, 0, False),
               ("top_users", "c5_top_users_b1024_k100", 10_000_000, 64, 1024, 100, False, 0, 0, False),
               ("norm", "c5_item_inv_norm", 1_000_000, 64, 0, 0, False, 0, 0, False)]
    out = []
    for kind, name, I, D, b, k, implicit, m_mean, p_mean, asc in shapes:
        # the catalogue table has I rows; the query table has max(b, 2) rows (the item table itself for similar)
        n_q = max(b, 2)
        Cat = torch.randn((I, D), device=dev)
        Qt = Cat if kind in ("similar", "norm") else torch.randn((n_q, D), device=dev)
        if asc:                                  # z = <e_0, item row> = i / I: ascending scores
            Qt.zero_()
            Qt[:, 0] = 1.0
            Cat.zero_()
            Cat[:, 0] = torch.arange(I, device=dev, dtype=torch.float32) / I
        E = torch.zeros((1, D), device=dev)
        if kind == "top_users":                  # catalogue = users, queries = items
            tabs = {"Uinv": Cat, "Iinv": Qt}
        elif kind in ("similar", "norm"):
            tabs = {"Uinv": torch.zeros((2, D), device=dev), "Iinv": Cat}
        else:
            tabs = {"Uinv": Qt, "Iinv": Cat}
        hp = HotPath({**tabs, "Uenv": tabs["Uinv"], "Ienv": tabs["Iinv"], "E": E, "W": E,
                      "b": torch.zeros(1, device=dev)}, implicit, False, False)
        n_query_rows = I if kind == "similar" else n_q
        ids = torch.from_numpy(rng.permutation(n_query_rows)[:max(b, 1)].astype(np.int64)).to(dev)
        m_off, m_it = lists(rng, n_q, I, m_mean, dev) if m_mean else (None, None)
        p_off, p_it = lists(rng, n_q, I, p_mean, dev) if p_mean else (None, None)
        g_off, g_it = lists(rng, n_q, I, 5, dev) if kind == "eval" else (None, None)
        top = torch.empty((max(b, 1), max(k, 1)), dtype=torch.int64, device=dev)
        sc = torch.empty((max(b, 1), max(k, 1)), dtype=torch.float32, device=dev)
        hits = torch.empty((max(b, 1), max(k, 1)), dtype=torch.uint8, device=dev)
        ngt = torch.empty(max(b, 1), dtype=torch.int64, device=dev)
        inv_norm = torch.empty(I, dtype=torch.float32, device=dev)
        p = _lib.make_params(hp.params)
        P = _lib.ptr
        st = _lib.stream_ptr()

        def call(lib):
            if kind == "eval":
                rc = lib.invpref_eval_topk(C.byref(hp.desc), C.byref(p), P(ids), b, P(m_off), P(m_it), P(p_off),
                                           P(p_it), P(g_off), P(g_it), k, P(top), None, P(hits), P(ngt), st)
            elif kind == "recommend":
                rc = lib.invpref_recommend(C.byref(hp.desc), C.byref(p), P(ids), b, None, None, k, P(top), P(sc), st)
            elif kind == "similar":
                rc = lib.invpref_similar_items(C.byref(hp.desc), C.byref(p), P(ids), b, k, P(inv_norm), P(top),
                                               P(sc), st)
            elif kind == "top_users":
                rc = lib.invpref_top_users(C.byref(hp.desc), C.byref(p), P(ids), b, None, None, k, P(top), P(sc), st)
            else:                                # similar_items of one item: the row-norm kernel is timed out of it
                rc = lib.invpref_similar_items(C.byref(hp.desc), C.byref(p), P(ids), 1, 1, P(inv_norm), P(top),
                                               P(sc), st)
            _lib.check(rc, name)

        r = {"shape": name, "call": kind, "rows": I, "D": D, "b": b, "k": k}
        big = b * I * D > 1e13                   # seconds per call: one warm-up, one timed call
        mine_t, base_t, same = [], [], True
        if kind == "norm":
            mine_t.append(kernel_us(lambda: call(hp.lib), "row_inv_norm_kernel"))
        for rep in range(0 if kind == "norm" else
                         max(1, args.repeats) if base is not None and kind in ("eval", "recommend") else 1):
            mine_t.append(timed(lambda: call(hp.lib), warmup=1 if big else 2))
            if base is not None and kind in ("eval", "recommend") and (b <= 4096 or kind == "eval"):
                mine = top.clone()
                base_t.append(timed(lambda: call(base), budget_s=0.1))
                same = same and bool(torch.equal(mine, top))
        t = float(np.median(mine_t))
        r["us"] = round(t, 2)
        if len(mine_t) > 1:
            r["us_repeats"] = [round(x, 2) for x in mine_t]
        if kind == "norm":
            r["read_gb_per_s"] = round(I * D * 4 / (t * 1e-6) / 1e9, 1)
        else:
            r["queries_per_s"] = round(b / (t * 1e-6), 1)
            r["fma_bound_fraction"] = round(b * I * D / fma_per_s / (t * 1e-6), 4)
        if base_t:
            tb = float(np.median(base_t))
            r["baseline_us"] = round(tb, 2)
            if len(base_t) > 1:
                r["baseline_us_repeats"] = [round(x, 2) for x in base_t]
            r["speedup_vs_baseline"] = round(tb / t, 3)
            r["same_items_as_baseline"] = same
        if kind in ("eval", "recommend") and b * I * 4 <= (16 << 30):
            users = ids

            def step_by_step():
                rating = torch.sigmoid(Qt[users] @ Cat.t()) if implicit else Qt[users] @ Cat.t()
                for off, it, value, add in ((m_off, m_it, -1024.0, 0), (p_off, p_it, 1024.0, 1)):
                    if off is not None:
                        _lib.check(hp.lib.invpref_mask_scores(P(rating), b, I, P(users), P(off), P(it),
                                                              C.c_float(value), add, st), "mask")
                torch.topk(rating, k, dim=1)
            r["step_by_step_us"] = round(timed(step_by_step), 2)
        print(json.dumps(r), flush=True)
        out.append(r)
        del Qt, Cat, hp, tabs
        torch.cuda.empty_cache()
    res = {"topk_stream": out, **info, "sms": n_sm, "commit": args.commit, "baseline_lib": args.baseline_lib,
           "repeats": args.repeats}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

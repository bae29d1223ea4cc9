#!/usr/bin/env python
"""CUDA-event timing of the streaming top-k kernel (eval.cu) behind ``invpref_eval_topk`` and ``invpref_recommend``.
GPU only.

    python tools/time_topk.py [--baseline-lib OTHER.so] [--out FILE]

Shapes: the evaluator's calls as the drivers make them (Yahoo-implicit, MovieLens, MIND with its item pool), the C5
catalogue (1 M items, D 64) at b in {1, 256, 4096, 65536} and k in {50, 256}, and an adversarial stream whose scores
ascend with the item id (every item tile raises the threshold).  Per shape: microseconds per call, users per second
and the fraction of the fp32 FMA issue bound (b * I * D FMAs over SMs x 128 lanes x the maximum SM clock).
``--baseline-lib``: also times ``invpref_eval_topk`` of another build of the library (e.g. the parent commit's, whose
evaluator ran one CTA per user) on the same inputs.  Where the [b, I] matrix fits in 16 GiB the step-by-step device
path (``predict`` GEMM, ``invpref_mask_scores`` for the evaluator's lists, ``torch.topk``) is timed as well.
``--commit``: a label of the source tree measured, stored in the output.  The item tables are fresh random
normals per shape; the C5 table (256 MB) is larger than L2, the dataset ones fit in it.
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


def timed(fn, budget_s=0.3):
    """Mean microseconds per call after 2 warm-up calls, over enough calls to fill about `budget_s` (at least 1)."""
    for _ in range(2):
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


def lists(rng, n_users, n_items, mean, dev):
    """Ascending unique item lists of about `mean` entries per user, as int64 CSR on the device."""
    u = np.repeat(np.arange(n_users), rng.poisson(mean, n_users))
    off, items = user_item_csr(u, rng.integers(0, n_items, u.size), n_users)
    return torch.from_numpy(off).to(dev), torch.from_numpy(items if items.size else np.zeros(1, np.int64)).to(dev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-lib", default=None)
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
        base.invpref_eval_topk.argtypes = _lib.load().invpref_eval_topk.argtypes
        base.invpref_eval_topk.restype = C.c_int
    rng = np.random.default_rng(0)
    # name, n_items, D, b, k, implicit, mask mean, pool mean, scores ascending with item id
    shapes = [("yahoo_implicit_eval", 1000, 40, 1024, 7, True, 20, 0, False),
              ("movielens_eval", 3706, 40, 2048, 30, True, 100, 0, False),
              ("mind_eval", 51283, 40, 256, 40, True, 10, 100, False)]
    shapes += [(f"c5_b{b}_k{k}", 1_000_000, 64, b, k, False, 0, 0, False) for b in (1, 256, 4096, 65536)
               for k in (50, 256)]
    shapes += [("c5_ascending_b4096_k256", 1_000_000, 64, 4096, 256, False, 0, 0, True)]
    out = []
    for name, I, D, b, k, implicit, m_mean, p_mean, asc in shapes:
        n_users = max(b, 2)
        U = torch.randn((n_users, D), device=dev)
        It = torch.randn((I, D), device=dev)
        if asc:                                  # z = <e_0, item row> = i / I: ascending scores
            U.zero_()
            U[:, 0] = 1.0
            It.zero_()
            It[:, 0] = torch.arange(I, device=dev, dtype=torch.float32) / I
        E = torch.zeros((1, D), device=dev)
        hp = HotPath({"Uinv": U, "Iinv": It, "Uenv": U, "Ienv": It, "E": E, "W": E,
                      "b": torch.zeros(1, device=dev)}, implicit, False, False)
        users = torch.from_numpy(rng.permutation(n_users)[:b].astype(np.int64)).to(dev)
        m_off, m_it = lists(rng, n_users, I, m_mean, dev) if m_mean else (None, None)
        p_off, p_it = lists(rng, n_users, I, p_mean, dev) if p_mean else (None, None)
        g_off, g_it = lists(rng, n_users, I, 5, dev)
        top = torch.empty((b, k), dtype=torch.int64, device=dev)
        sc = torch.empty((b, k), dtype=torch.float32, device=dev)
        hits = torch.empty((b, k), dtype=torch.uint8, device=dev)
        ngt = torch.empty(b, dtype=torch.int64, device=dev)
        p = _lib.make_params(hp.params)
        P = _lib.ptr
        evaluator = name.endswith("_eval")

        def call(lib):
            if evaluator:
                rc = lib.invpref_eval_topk(C.byref(hp.desc), C.byref(p), P(users), b, P(m_off), P(m_it), P(p_off),
                                           P(p_it), P(g_off), P(g_it), k, P(top), None, P(hits), P(ngt),
                                           _lib.stream_ptr())
            else:                                # the parent's evaluator without lists = recommend without exclusion
                rc = (lib.invpref_recommend(C.byref(hp.desc), C.byref(p), P(users), b, None, None, k, P(top), P(sc),
                                            _lib.stream_ptr()) if lib is hp.lib else
                      lib.invpref_eval_topk(C.byref(hp.desc), C.byref(p), P(users), b, None, None, None, None, None,
                                            None, k, P(top), P(sc), None, None, _lib.stream_ptr()))
            _lib.check(rc, name)

        r = {"shape": name, "n_items": I, "D": D, "b": b, "k": k}
        t = timed(lambda: call(hp.lib))
        r["us"] = round(t, 2)
        r["users_per_s"] = round(b / (t * 1e-6), 1)
        r["fma_bound_fraction"] = round(b * I * D / fma_per_s / (t * 1e-6), 4)
        if base is not None and (b <= 4096 or evaluator):
            mine = top.clone()
            tb = timed(lambda: call(base), budget_s=0.1)
            r["baseline_us"] = round(tb, 2)
            r["speedup_vs_baseline"] = round(tb / t, 2)
            r["same_items_as_baseline"] = bool(torch.equal(mine, top))
        if b * I * 4 <= (16 << 30):
            def step_by_step():
                rating = torch.sigmoid(U[users] @ It.t()) if implicit else U[users] @ It.t()
                for off, it, value, add in ((m_off, m_it, -1024.0, 0), (p_off, p_it, 1024.0, 1)):
                    if off is not None:
                        _lib.check(hp.lib.invpref_mask_scores(P(rating), b, I, P(users), P(off), P(it),
                                                              C.c_float(value), add, _lib.stream_ptr()), "mask")
                torch.topk(rating, k, dim=1)
            r["step_by_step_us"] = round(timed(step_by_step), 2)
        print(json.dumps(r), flush=True)
        out.append(r)
        del U, It, hp
        torch.cuda.empty_cache()
    res = {"topk_stream": out, **info, "sms": n_sm, "commit": args.commit, "baseline_lib": args.baseline_lib}
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

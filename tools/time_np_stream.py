"""Timing of numpy's global stream drawn on the device (npstream.device_randint) against the host draw, and of the
trainer's cluster() + stat_envs() in its three tie-break modes.  GPU only.   python tools/time_np_stream.py [--no-c5]

Draw sizes: the tie-break draw of one cluster() at C2 (Yahoo!R3, 311 704 from 5!), C3 (MovieLens, 1 M from 2!), C4
(MIND, 4 194 304 from 6!) and C5 (96.5 M from 4!).  Every timing is a host clock around work that ends in a device
synchronise (device_randint synchronises for its state read-back; cluster() reads its diff count, stat_envs() its
histogram); the median of the repetitions is reported after warm-up calls."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench as B  # noqa: E402
from invpref_kdd_2022_b200 import npstream  # noqa: E402

SIZES = {"c2": (311_704, 120), "c3": (1_000_000, 2), "c4": (4_194_304, 720), "c5": (96_500_000, 24)}


def wall_ms(fn, reps, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return round(statistics.median(ts), 3)


def trainer(name, dev):
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    from invpref_kdd_2022_b200.train import ExplicitTrainManager, ImplicitTrainManager
    w = B.WORKLOADS[name]
    N = SIZES[name][0]
    g = torch.Generator(device=dev).manual_seed(5)
    data = torch.stack([torch.randint(0, w["U"], (N,), device=dev, generator=g),
                        torch.randint(0, w["I"], (N,), device=dev, generator=g),
                        torch.randint(0 if w["implicit"] else 1, 2 if w["implicit"] else 6, (N,), device=dev,
                                      generator=g)], 1)
    M = InvPrefImplicit if w["implicit"] else InvPrefExplicit
    T = ImplicitTrainManager if w["implicit"] else ExplicitTrainManager
    model = M(w["U"], w["I"], w["K"], w["D"], w["roe"], w["ree"]).to(dev)
    np.random.seed(0)
    tm = T(model=model, evaluator=None, device=dev, training_data=data, batch_size=w["B"], epochs=1,
           cluster_interval=1, evaluate_interval=1, lr=w["lr"], invariant_coe=1.0, env_aware_coe=1.0, env_coe=1.0,
           L2_coe=1.0, L1_coe=1.0, alpha=None, tie_break_rng="numpy_device")
    del data
    return tm


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--no-c5", action="store_true")
    ap.add_argument("--reps", type=int, default=7)
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": gpu}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    npstream.device_randint(2, 1, dev)                      # builds the jump table
    torch.cuda.synchronize()
    res["jump_table_build_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    res["jump_table_MB"] = round(npstream.jump_table_bytes(dev) / 1e6, 1)
    names = [n for n in SIZES if not (args.no_c5 and n == "c5")]
    draws = {}
    for name in names:
        N, high = SIZES[name]
        out = torch.empty(N, dtype=torch.int64, device=dev)
        np.random.seed(1)
        r = {"n": N, "high": high,
             "numpy_device_ms": wall_ms(lambda: npstream.device_randint(high, N, dev, out=out), args.reps),
             "host_numpy_plus_upload_ms": wall_ms(
                 lambda: out.copy_(torch.from_numpy(np.random.randint(0, high, N))), max(3, args.reps // 2), 1),
             "torch_device_randint_ms": wall_ms(lambda: torch.randint(0, high, (N,), device=dev, out=out), args.reps)}
        draws[name] = r
        del out
    res["draw"] = draws
    cl = {}
    for name in names:
        tm = trainer(name, dev)
        r = {}
        for mode in ("numpy", "device", "numpy_device"):
            tm.tie_break_rng = mode

            def step():
                tm.cluster()
                tm.stat_envs()
            r[f"{mode}_ms"] = wall_ms(step, max(3, args.reps // 2) if mode == "numpy" else args.reps, 1)
        cl[name] = r
        del tm
        torch.cuda.empty_cache()
    res["cluster_plus_stat_envs"] = cl
    print(json.dumps({"np_stream": res}))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- InvPref hot path on B200: train interactions/s (fwd + bwd + Adam) and env re-assignment
samples/s, with the HBM roofline fraction and the reference's CPU path beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c5|c4|c3|c2] [--impl ours|reference]
                    [--dump-outputs DIR]

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for the definitions:
  value      whole-job train interactions/s, inputs + cached sort-segment plans resident in HBM;
  e2e        the same through the public call with HOST (pinned) batch buffers: H2D of the batch, plan
             build, step, D2H of the six losses, every step;
  roofline   algorithmic bytes (SURVEY.md §8d) / CUDA-event time, for the whole fused step and for its
             dominant kernel, against MEASURED_PEAKS.json;
  cluster    env re-assignment samples/s and its roofline;
  cpu_baseline  the oracle's torch-eager port (same ATen op sequence as the reference trainer) timed on
             the box's host cores on a bounded, proportionally scaled sample.
  torch_eager_gpu  the same port on the same GPU at full size (SURVEY.md 8d: the number the kernels must beat).

--dump-outputs DIR writes what the last timed train step returned to its caller -- the six losses and the updated
parameters (a fixed, seeded sample of the table rows) -- as DIR/<name>.npy, so that two builds can be compared
output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# SURVEY.md §8d workloads.  Coefficients: the Yahoo explicit / MovieLens / MIND driver values.
WORKLOADS = {
    "c5": dict(name="synthetic 10M users x 1M items, dim 64, K=4, explicit, B=4194304", U=10_000_000, I=1_000_000,
               D=64, K=4, B=4_194_304, implicit=False, roe=True, ree=False, crw=True, rrw=True, lr=1e-3,
               coef=dict(c_inv=0.007375309563638757, c_ea=7.207790368836971, c_env=7.30272189219841,
                         c_L2=5.105587170019545, c_L1=0.004098813161410509)),
    "c4": dict(name="MIND-shaped synthetic, 50000 x 51283, dim 40, K=6, implicit, B=262144", U=50_000, I=51_283,
               D=40, K=6, B=262_144, N=4_194_304, implicit=True, roe=True, ree=False, crw=True, rrw=False, lr=1e-3,
               coef=dict(c_inv=0.41343891722673093, c_ea=9.833594297680568, c_env=7.521558049068597,
                         c_L2=4.324061954456766, c_L1=0.33322012936680223)),
    "c3": dict(name="MovieLens-shaped synthetic, 6040 x 3706, dim 40, K=2, implicit, B=65536", U=6_040, I=3_706,
               D=40, K=2, B=65_536, N=1_000_000, implicit=True, roe=True, ree=True, crw=False, rrw=True, lr=1e-2,
               coef=dict(c_inv=8.909348155983732, c_ea=1.233057369609993, c_env=8.064376793624795,
                         c_L2=3.4987474005653665, c_L1=0.9355983539586914)),
    "c2": dict(name="Yahoo!R3-shaped explicit, 15400 x 1000, dim 40, K=5, B=131072", U=15_400, I=1_000,
               D=40, K=5, B=131_072, N=311_704, implicit=False, roe=True, ree=False, crw=False, rrw=False, lr=1e-3,
               coef=dict(c_inv=0.007375309563638757, c_ea=7.207790368836971, c_env=7.30272189219841,
                         c_L2=5.105587170019545, c_L1=0.004098813161410509)),
}


def synth_batches(w, nb, seed=20220814, scale=1.0):
    """SURVEY.md §8d generators: mild user skew (r^1.5), hot-item skew (r^3)."""
    U, I, B = max(int(w["U"] * scale), 8), max(int(w["I"] * scale), 8), max(int(w["B"] * scale), 8)
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(nb):
        u = np.floor(U * rng.random(B) ** 1.5).astype(np.int64)
        i = np.floor(I * rng.random(B) ** 3).astype(np.int64)
        y = (rng.integers(0, 2, B) if w["implicit"] else rng.integers(1, 6, B)).astype(np.float32)
        e = rng.integers(0, w["K"], B).astype(np.int64)
        out.append((u, i, y, e))
    return U, I, B, out


def step_bytes(B, D, K, P):
    """SURVEY.md §8d: algorithmic bytes of one train step."""
    return B * (32 * D + 56 + 8 * K) + 24 * P


def cluster_bytes_per_sample(D):
    """SURVEY.md §8d: 16 D + 44."""
    return 16 * D + 44


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the captured kernels (one `ncu --set full` capture
    of this same command, summarised by tools/ncu_summary.py into profiles/ncu_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return {}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_tables(w, dev, U=None, I=None, seed=17373331):
    U, I = U or w["U"], I or w["I"]
    g = torch.Generator(device=dev).manual_seed(seed)
    shp = {"Uinv": (U, w["D"]), "Iinv": (I, w["D"]), "Uenv": (U, w["D"]), "Ienv": (I, w["D"]),
           "E": (w["K"], w["D"]), "W": (w["K"], w["D"]), "b": (w["K"],)}
    out = {}
    for k, s in shp.items():
        std = 0.01 if k not in ("W", "b") else 0.1
        out[k] = torch.randn(s, generator=g, device=dev, dtype=torch.float32) * std
    return out


def dump_outputs(out_dir, hp, loss, users, items, seed=20221014):
    """What one HotPath.train_step returned to its caller: ``losses.npy`` (the six losses, _lib.LOSS_KEYS order) and
    every parameter after the step (call after hp.flush(): lazy user rows are current).  A table of more rows than
    fit 8 MB is sampled -- half of the rows from the step's own batch ``users`` / ``items`` (rows its gradients
    reached), half uniformly, from a fixed seed -- and the sampled row ids go to ``user_rows.npy`` / ``item_rows.npy``:
    at most ~34 MB in all for D <= 64."""
    rng = np.random.default_rng(seed)
    cap = (8 << 20) // (4 * hp.dim)
    arrays = {"losses": loss.cpu().numpy()}
    for side, n, ids in (("user", hp.n_users, users), ("item", hp.n_items, items)):
        rows = np.arange(n) if n <= cap else np.unique(np.concatenate(
            [rng.choice(ids, cap // 2), rng.integers(0, n, cap - cap // 2)]))
        arrays[side + "_rows"] = rows.astype(np.float64)
        sel = torch.from_numpy(rows).to(hp.device)
        for k in (("Uinv", "Uenv") if side == "user" else ("Iinv", "Ienv")):
            arrays[k] = hp.params[k].index_select(0, sel).cpu().numpy()
    for k in ("E", "W", "b"):
        arrays[k] = hp.params[k].cpu().numpy()
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_baseline(w, threads, budget_s=25.0, scale=None, steps=12, warmup=1):
    """The oracle's torch-eager port on the host cores, on a proportionally scaled replica of the
    workload (U, I and B divided by the same factor, so dense-Adam work per interaction is unchanged)."""
    from oracle import invpref_numpy as on
    from oracle import invpref_torch_cpu as ot
    torch.set_num_threads(threads)
    if scale is None:
        scale = min(1.0, 262_144 / w["B"])
    U, I, B, batches = synth_batches(w, 1, scale=scale)
    P = ot.random_params(U, I, w["K"], w["D"])
    hp = on.Hyper(alpha=1.0, lr=w["lr"], use_class_rw=w["crw"], use_rec_rw=w["rrw"], **w["coef"])
    tr = ot.CpuTrainer(P, on.Flags(w["implicit"], w["roe"], w["ree"]), hp)
    u, i, y, e = (torch.from_numpy(a) for a in batches[0])
    wts = torch.rand(B)
    times = []
    t_all = time.perf_counter()
    for s in range(warmup + steps):
        t0 = time.perf_counter()
        tr.train_a_batch(u, i, y, e, wts, 1.0)
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
        if time.perf_counter() - t_all > budget_s and len(times) >= 1:
            break
    t_step = statistics.median(times)
    pidx = torch.randint(0, tr.eps_table.shape[0], (B,))
    t0 = time.perf_counter()
    tr.cluster_a_batch(u, i, y, pidx)
    t_cl = time.perf_counter() - t0
    sample = (f"1/{round(1 / scale)}-scale replica (U={U}, I={I}, B={B}, D={w['D']}, K={w['K']}): "
              f"{len(times)} train_a_batch after {warmup} warm-up; 1 cluster_a_batch")
    return {"value": B / t_step, "unit": "interactions/s", "cores": threads, "kind": "port", "sample": sample,
            "ms_per_step": t_step * 1e3, "cluster_samples_per_s": B / t_cl}


def torch_eager_gpu(w, dev, dbatch, steps=3):
    """SURVEY.md 8d: "also time the reference on the B200 via torch eager -- the number the new kernels must
    beat".  The oracle's torch port issues the reference's op sequence (13 embedding gathers + their dense
    backward, autograd, torch.optim.Adam, six float() syncs per step); here it runs on the same GPU, same batch,
    same shapes.  Baseline only (never the product path)."""
    from oracle import invpref_numpy as on
    from oracle import invpref_torch_cpu as ot
    u, i, y, e, sw = dbatch
    P = {k: v.requires_grad_(True) for k, v in make_tables(w, dev).items()}
    hp = on.Hyper(alpha=1.0, lr=w["lr"], use_class_rw=w["crw"], use_rec_rw=w["rrw"], **w["coef"])
    tr = ot.CpuTrainer(P, on.Flags(w["implicit"], w["roe"], w["ree"]), hp)
    tr.train_a_batch(u, i, y, e, sw, 1.0)                       # warm-up (allocates grads and Adam state)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        tr.train_a_batch(u, i, y, e, sw, 1.0)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    out = {"value": u.numel() / dt, "unit": "interactions/s", "ms_per_step": dt * 1e3, "steps": steps,
           "kind": "port: torch-eager op sequence of the reference, on the same B200, full-size batch"}
    del tr, P
    torch.cuda.empty_cache()
    return out


class _NullEvaluator:
    def evaluate(self):
        return {"mse": 0.0}


def config_leg(name, dev, with_eager=True, seed=17373331, quick=False):
    """One of BASELINE.json's dataset-scale configs (C2 Yahoo explicit, C3 MovieLens, C4 MIND) through the PUBLIC
    trainer API, built as the reference drivers build it: InvPref model + Explicit/ImplicitTrainManager on one
    synthetic epoch of the config's shape (SURVEY.md 8d), train_a_epoch() / cluster() / stat_envs().  Tables and
    interactions are L2-resident: the figure of merit is interactions/s against torch-eager on the same GPU and the
    launches per step (the trainer replays each epoch as one CUDA graph), not the HBM fraction."""
    from invpref_kdd_2022_b200 import _lib
    from invpref_kdd_2022_b200.dataloader import synthetic_interactions
    from invpref_kdd_2022_b200.models import InvPrefExplicit, InvPrefImplicit
    from invpref_kdd_2022_b200.train import ExplicitTrainManager, ImplicitTrainManager
    w = WORKLOADS[name]
    U, I, N, B, K, D = w["U"], w["I"], w["N"], w["B"], w["K"], w["D"]
    data = synthetic_interactions(U, I, N, w["implicit"])
    torch.manual_seed(seed)
    np.random.seed(seed)
    M, T = (InvPrefImplicit, ImplicitTrainManager) if w["implicit"] else (InvPrefExplicit, ExplicitTrainManager)
    c = w["coef"]

    def build(use_graph):
        model = M(U, I, K, D, w["roe"], w["ree"]).to(dev)
        tm = T(model=model, evaluator=_NullEvaluator(), device=dev, training_data=torch.LongTensor(data).to(dev),
               batch_size=B, epochs=1, cluster_interval=1, evaluate_interval=1, lr=w["lr"], invariant_coe=c["c_inv"],
               env_aware_coe=c["c_ea"], env_coe=c["c_env"], L2_coe=c["c_L2"], L1_coe=c["c_L1"], alpha=None,
               use_class_re_weight=w["crw"], use_recommend_re_weight=w["rrw"], use_graph=use_graph)
        tm.stat_envs()
        return tm

    def timed(tm, epochs):
        for _ in range(3):                       # first epoch builds the plans, second captures the graph(s)
            tm.train_a_epoch()
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        t0 = time.perf_counter()
        for _ in range(epochs):
            ld = tm.train_a_epoch()              # one host sync per epoch (the loss rows), as the trainer always does
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / epochs * 1e3
        assert np.isfinite(ld["loss"])
        return wall, (_lib.launch_count() - l0) / (epochs * tm.batch_num)

    epochs = max(4, 60 // max(1, -(-N // B)))
    tm = build(True)
    g_ms, g_launch = timed(tm, epochs)
    steps = tm.batch_num
    tc0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        tm.cluster()
        tm.stat_envs()
    torch.cuda.synchronize()
    cl_ms = (time.perf_counter() - tc0) / reps * 1e3
    tm.tie_break_rng = "device"                  # opt-in: tie-break rows from the device generator (not numpy's stream)
    tm.cluster()
    torch.cuda.synchronize()
    tc0 = time.perf_counter()
    for _ in range(reps):
        tm.cluster()
        tm.stat_envs()
    torch.cuda.synchronize()
    cl_dev_ms = (time.perf_counter() - tc0) / reps * 1e3
    del tm
    if quick:
        p_ms, p_launch = g_ms, g_launch
    else:
        tm = build(False)
        p_ms, p_launch = timed(tm, epochs)
        del tm
    P = 2 * (U + I) * D + 2 * K * D + K
    leg = {"workload": w["name"], "interactions_per_epoch": N, "steps_per_epoch": steps, "global_batch": B, "params": P,
           "value": N / (g_ms * 1e-3), "unit": "interactions/s", "ms_per_step": g_ms / steps, "ms_per_epoch": g_ms,
           "launches_per_step": g_launch, "timing": "wall clock over %d train_a_epoch() calls incl. the per-epoch loss "
           "read-back; epoch = one CUDA-graph launch" % epochs,
           "no_graph": {"value": N / (p_ms * 1e-3), "ms_per_step": p_ms / steps, "launches_per_step": p_launch},
           "cluster": {"value": N / (cl_ms * 1e-3), "unit": "samples/s", "ms": cl_ms,
                       "note": "trainer.cluster() + stat_envs(): host-drawn tie-break indices (numpy stream, as the "
                               "reference) + H2D + one kernel + diff read-back",
                       "device_tie_break_rng": {"value": N / (cl_dev_ms * 1e-3), "ms": cl_dev_ms,
                                                "note": "tie_break_rng='device' (opt-in, not the reference's numpy "
                                                        "stream): no host draw, no H2D"}},
           "roofline_frac_8d": step_bytes(B, D, K, P) * steps / (g_ms * 1e-3) / 1e9 / measured_peaks()[0]}
    if quick:
        del leg["no_graph"]
    torch.cuda.empty_cache()
    if with_eager:
        try:
            sl = slice(0, B)
            t = lambda a, dt=None: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
            u, i = t(data[sl, 0]), t(data[sl, 1])
            y = t(data[sl, 2].astype(np.float32))
            e = torch.randint(0, K, (B,), device=dev)
            sw = torch.rand(B, device=dev)
            eg = torch_eager_gpu(w, dev, (u, i, y, e, sw), steps=5)
            leg["torch_eager_gpu"] = {"value": eg["value"], "ms_per_step": eg["ms_per_step"],
                                      "speedup_of_value": leg["value"] / eg["value"]}
        except Exception as ex:      # noqa: BLE001
            leg["torch_eager_gpu"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:200]}
    return leg


def run_reference(args, w):
    threads = os.cpu_count() or 1
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_baseline(w, threads, budget_s=float("inf"), steps=args.steps, warmup=min(args.warmup, 1))
    scale = min(1.0, 262_144 / w["B"])
    label = w["name"] if scale >= 1.0 else f"1/{round(1 / scale)}-scale replica (U, I and B divided by " \
        f"{round(1 / scale)}: bounded CPU sample) of: " + w["name"]
    line = {"impl": "reference", "metric": "train interactions/sec (fwd+bwd+Adam)", "value": r["value"],
            "unit": "interactions/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": label, "global_batch": max(int(w["B"] * scale), 8),
                       "full_size_global_batch": w["B"], "scale": scale,
                       "params": 2 * (max(int(w["U"] * scale), 8) + max(int(w["I"] * scale), 8)) * w["D"]
                       + 2 * w["K"] * w["D"] + w["K"]},
            "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "cluster": {"value": r["cluster_samples_per_s"], "unit": "samples/s"},
            "e2e": {"value": r["value"], "unit": "interactions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def run_ours_single(args, w):
    from invpref_kdd_2022_b200 import _lib
    from invpref_kdd_2022_b200.engine import HotPath
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    K, D = w["K"], w["D"]
    nb = max(1, min(args.nbatch or (args.steps + args.warmup), args.steps + args.warmup))
    U, I, B, batches = synth_batches(w, nb)
    hp = HotPath(make_tables(w, dev), w["implicit"], w["roe"], w["ree"], lr=w["lr"])
    P = sum(t.numel() for t in hp.params.values())
    dbatches = []
    for (u, i, y, e) in batches:
        u, i, y, e = (torch.from_numpy(a).to(dev) for a in (u, i, y, e))
        cw, sw = hp.stat_envs(e, hp.env_hist(e))
        dbatches.append((u, i, y, e, sw))
    plans = [hp.new_plan(b[0], b[1]) for b in dbatches]
    kw = dict(alpha=1.0, use_class_rw=w["crw"], use_rec_rw=w["rrw"], **w["coef"])
    losses = torch.zeros((args.steps + args.warmup, 6), device=dev)

    def step(s, plan=True):
        b = dbatches[s % nb]
        hp.train_step(b[0], b[1], b[2], b[3], b[4], plan=plans[s % nb] if plan else None, loss_out=losses[s], **kw)

    def timed(lazy):
        """W warm-up + K timed steps.  Lazy mode: the flush that brings every user row up to date is INSIDE
        the timed region, so at the end of it all state is materialised exactly as after K dense steps."""
        hp.set_lazy(lazy)
        for s in range(args.warmup):
            step(s)
        hp.flush()
        torch.cuda.synchronize()
        _lib.profile_enable(args.steps)
        clocks = ClockSampler(dev.index)
        clocks.start()
        l0 = _lib.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        ev0.record()
        for s in range(args.warmup, args.warmup + args.steps):
            step(s)
        hp.flush()
        ev1.record()
        torch.cuda.synchronize()
        launches = _lib.launch_count() - l0
        clk = clocks.stop()
        ms = ev0.elapsed_time(ev1) / args.steps
        phases = np.asarray(_lib.profile_read_all())
        _lib.profile_enable(0)
        assert torch.isfinite(losses).all(), "non-finite loss in the timed region"
        ph = dict(zip(_lib.PHASES, phases.mean(axis=0).tolist())) if len(phases) else {}
        return ms, ph, launches, clk

    peak, peak_src = measured_peaks()
    sbytes = step_bytes(B, D, K, P)
    # unique rows per batch (mean over the distinct batches): what the lazy step actually touches
    n_seg_u = int(round(np.mean([torch.unique(b[0]).numel() for b in dbatches])))
    n_seg_i = int(round(np.mean([torch.unique(b[1]).numel() for b in dbatches])))
    # (1) plain dense Adam: every user row is read and written every step
    d_ms, d_ph, d_launch, d_clk = timed(False)
    dense = {"value": B / (d_ms * 1e-3), "unit": "interactions/s", "ms_per_step": d_ms,
             "roofline_frac": sbytes / (d_ms * 1e-3) / 1e9 / peak, "phase_ms": d_ph, "clocks": d_clk}
    if d_ph.get("sweep_users"):
        sweep_bytes = (U - n_seg_u) * 2 * D * 4 * 6
        a = sweep_bytes / (d_ph["sweep_users"] * 1e-3) / 1e9
        dense["sweep_kernel"] = {"bytes_per_launch": sweep_bytes, "ms_per_launch": d_ph["sweep_users"],
                                 "achieved": a, "frac": a / peak}
    # (2) headline: lazy dense Adam (bit-identical results, tests/test_gpu_lazy.py), flush inside the region
    ms, ph_ms, launches, clk = timed(not args.dense_adam)
    if args.dump_outputs:
        last = args.warmup + args.steps - 1
        dump_outputs(args.dump_outputs, hp, losses[last], batches[last % nb][0], batches[last % nb][1])
    # whole step.  SURVEY.md 8d's convention (B(32D+56+8K) + 24P) charges dense Adam traffic for all P parameters; the
    # lazy path does not move those bytes, so for this leg the fraction is taken over the bytes the step's kernels
    # ACTUALLY have to move (unique-row counts of the batches): user pass (below), item pass (theta/m/v of the unique
    # items 48 D, per interaction the stashed user-row pair 8 D + g-pack 32 + perm/pseg 8), item sweep (untouched
    # items 48 D).  The final flush is timed but its bytes are not counted (a lower bound on the fraction).  The 8d
    # figure is kept for the dense leg only (dense_adam.roofline_frac).
    ub = n_seg_u * (48 * D + 8 * D + 4) + B * (8 * D + 36 + 32)
    ib = n_seg_i * (48 * D + 16) + B * (8 * D + 32 + 8) + (I - n_seg_i) * 48 * D
    step_roof = {"bytes_per_step_actual": ub + ib, "achieved": (ub + ib) / (ms * 1e-3) / 1e9, "unit": "GB/s",
                 "frac": (ub + ib) / (ms * 1e-3) / 1e9 / peak, "unique_users": n_seg_u, "unique_items": n_seg_i,
                 "survey_8d_bytes_per_step": sbytes,
                 "note": "fraction over the bytes the lazy step must move (unique rows of the batch), not over SURVEY.md "
                         "8d's dense-Adam convention (that one: dense_adam.roofline_frac)"}
    # roofline object = the DOMINANT KERNEL: fused user pass.  Its algorithmic bytes per launch: per unique user
    # theta/m/v of two tables read + written (48 D) + the stashed row pair (8 D) + last_step (4); per interaction
    # two item rows (8 D), ids + perm + scalars (36), g-pack write (32).  Timed live by CUDA events recorded
    # between the library's kernels on its stream (invpref_profile_*), averaged over the timed steps.
    roof = {"bound": "hbm", "kernel": "upass_rows (fused forward + losses + user-side segment reduce + Adam)",
            "peak": peak, "peak_source": peak_src, "unit": "GB/s", "traffic": None}
    if ph_ms.get("rows_users"):
        a = ub / (ph_ms["rows_users"] * 1e-3) / 1e9
        roof.update({"achieved": a, "frac": a / peak, "bytes_per_launch": ub, "ms_per_launch": ph_ms["rows_users"],
                     "share_of_step": ph_ms["rows_users"] / ms})
    else:
        roof.update({"kernel": "fused train step (all kernels)", "achieved": step_roof["achieved"],
                     "frac": step_roof["frac"]})
    tr = ncu_traffic().get("upass_rows")
    if tr:
        roof["traffic"] = tr["bytes"]
        roof["traffic_source"] = tr.get("source")
    roof["step"] = step_roof
    roof["phase_ms"] = ph_ms

    # ---- env re-assignment: all nb batches as one slice, as train.py:912-936 does ----
    cu, ci, cy, ce = (torch.cat([b[j] for b in dbatches]) for j in range(4))
    Nc = cu.numel()
    import itertools
    base = torch.Tensor([1e-10 * (1e-1 ** k) for k in range(K)])
    eps = torch.Tensor(list(itertools.permutations(base))).to(dev)                    # train.py:763-769
    pidx = torch.from_numpy(np.random.default_rng(1).integers(0, eps.shape[0], Nc)).to(dev)
    out_e = torch.empty(Nc, dtype=torch.int64, device=dev)       # caller-owned outputs: no allocation inside the timed calls
    out_w = torch.empty(Nc, dtype=torch.float32, device=dev)
    for _ in range(2):
        hp.cluster(cu, ci, cy, pidx, eps, ce, out=out_e)
    torch.cuda.synchronize()
    reps = 7
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    evs[0].record()
    for r_ in range(reps):
        new_e, hist, diff = hp.cluster(cu, ci, cy, pidx, eps, ce, trusted=True, out=out_e)
        hp.stat_envs(new_e, hist, out=out_w)
        evs[r_ + 1].record()
    torch.cuda.synchronize()
    per_rep = [evs[r_].elapsed_time(evs[r_ + 1]) for r_ in range(reps)]
    cms = statistics.median(per_rep)          # per-call CUDA-event times; the median is robust against a stray stall
    cb = cluster_bytes_per_sample(D) * Nc
    cluster = {"value": Nc / (cms * 1e-3), "unit": "samples/s", "samples": Nc, "ms": cms,
               "ms_min_max": [min(per_rep), max(per_rep)], "reps": reps,
               "roofline": {"bound": "hbm", "kernel": "cluster_kernel (+ stat_envs)", "achieved": cb / (cms * 1e-3) / 1e9,
                            "peak": peak, "unit": "GB/s", "frac": cb / (cms * 1e-3) / 1e9 / peak,
                            "bytes_per_launch": cb, "traffic": None}}
    # the same re-assignment over the user-sorted view of the samples (what trainer.cluster() runs: the view is static)
    view = hp.sorted_view(cu, ci, cy)
    for _ in range(2):
        s_new, s_hist, s_diff = hp.cluster_sorted(view, pidx, eps, ce, out=out_e)
    torch.cuda.synchronize()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    evs[0].record()
    for r_ in range(reps):
        s_new, s_hist, s_diff = hp.cluster_sorted(view, pidx, eps, ce, out=out_e)
        hp.stat_envs(s_new, s_hist, out=out_w)
        evs[r_ + 1].record()
    torch.cuda.synchronize()
    s_rep = [evs[r_].elapsed_time(evs[r_ + 1]) for r_ in range(reps)]
    sms = statistics.median(s_rep)
    n_users_seen = int(torch.unique(cu).numel())
    sb_actual = Nc * (8 * D + 12 + 3 * 32 + 8) + n_users_seen * 8 * D      # item rows + sorted ids/score + 3 scattered
    cluster["sorted_view"] = {                                               # sectors + perm; user rows once per user
        "value": Nc / (sms * 1e-3), "unit": "samples/s", "ms": sms, "ms_min_max": [min(s_rep), max(s_rep)],
        "samples_per_user": Nc / max(n_users_seen, 1),
        "bytes_per_launch_actual": sb_actual, "frac_actual_bytes": sb_actual / (sms * 1e-3) / 1e9 / peak,
        "identical_to_unsorted": bool(torch.equal(s_hist, hist) and torch.equal(s_diff, diff)),
        "note": "invpref_cluster_sorted: contiguous runs of the user-sorted samples per 16-lane group; the user rows of "
                "consecutive samples come out of L2.  8d's per-sample convention (16 D + 44) does not apply: fraction "
                "over the bytes this order actually has to move"}
    del view
    ctr = ncu_traffic().get("cluster")
    if ctr:   # captured on ctr["samples"] samples: scale to this launch
        cluster["roofline"]["traffic"] = ctr["bytes"] * Nc / ctr.get("samples", Nc)
        cluster["roofline"]["traffic_source"] = ctr.get("source")

    # ---- e2e: host (pinned) batch -> H2D -> plan build -> step -> D2H of the six losses, every step ----
    hb = [tuple(t.cpu().pin_memory() for t in b) for b in dbatches[:min(nb, 4)]]
    # Two staging sets (batch + plan buffer) and a loader stream: the H2D copy and the sort-segment plan of step
    # s+1 run under the kernels of step s, as a data-loader thread would do.  Every step's inputs still cross
    # PCIe and every step's plan is still built inside the timed region; the per-step loss read-back synchronises.
    stages = [[torch.empty_like(t, device=dev) for t in dbatches[0]] for _ in range(2)]
    plan_bufs = [torch.empty(hp.plan_bytes(B), dtype=torch.uint8, device=dev) for _ in range(2)]
    loader = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    h_loss = torch.empty((2, 6)).pin_memory()
    read_back = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_steps = args.steps                      # same amortisation of the final flush as the device-timed leg
    e2e_losses = []

    def issue_load(s):
        j = s % 2
        with torch.cuda.stream(loader):
            loader.wait_event(consumed[j])          # the step that last read this staging set is done
            for dst, src in zip(stages[j], hb[s % len(hb)]):
                dst.copy_(src, non_blocking=True)
            hp.new_plan(stages[j][0], stages[j][1], out=plan_bufs[j])
            ready[j].record(loader)

    def e2e_step(s):
        j = s % 2
        if s + 1 < e2e_total[0]:
            issue_load(s + 1)
        torch.cuda.current_stream().wait_event(ready[j])
        st = stages[j]
        out = hp.train_step(st[0], st[1], st[2], st[3], st[4], plan=plan_bufs[j], **kw)
        consumed[j].record()
        h_loss[j].copy_(out, non_blocking=True)            # this step's six losses -> pinned host memory
        read_back[j].record()
        if s > 0:                                           # the host reads step s-1's losses while step s runs: every
            read_back[j ^ 1].synchronize()                  # step's result is read, the read never idles the GPU
            e2e_losses.append(float(h_loss[j ^ 1][5]))

    e2e_total = [1]
    for ev in consumed:
        ev.record()
    issue_load(0)
    e2e_step(0)                                           # warm-up
    torch.cuda.synchronize()
    e2e_total[0] = e2e_steps
    t0 = time.perf_counter()
    issue_load(0)
    for s in range(e2e_steps):
        e2e_step(s)
    read_back[(e2e_steps - 1) % 2].synchronize()
    e2e_losses.append(float(h_loss[(e2e_steps - 1) % 2][5]))
    hp.flush()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) / e2e_steps * 1e3
    assert len(e2e_losses) >= e2e_steps and all(np.isfinite(e2e_losses))
    h2d = sum(t.numel() * t.element_size() for t in hb[0])
    e2e = {"value": B / (e2e_ms * 1e-3), "unit": "interactions/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": 24, "steps": e2e_steps,
           "note": "every step: host pinned batch (u,i,y,e,w) copied H2D and its sort-segment plan built on a loader "
                   "stream (overlapping the previous step's kernels), step, its 6 losses copied D2H and read by the "
                   "host one step later (while the next step runs); final flush of the lazy rows inside the region"}

    line = {"metric": "train interactions/sec (fwd+bwd+Adam)", "value": B / (ms * 1e-3), "unit": "interactions/s",
            "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": w["name"], "global_batch": B, "params": P, "distinct_batches": nb,
                       "l2": "inputs larger than L2 (tables %.1f GB + Adam state)" % (P * 4 / 1e9)
                       if P * 4 > 2.5e8 else "tables fit in L2 (no flush): launch-bound config",
                       "parallelism": "1 GPU"},
            "roofline": roof, "adam": "dense" if args.dense_adam else "lazy (bit-identical to dense, flush timed)",
            "dense_adam": dense, "cluster": cluster, "e2e": e2e, "gpu_launches": int(launches), "clocks": clk}
    # second kernel of the step: the item pass (ring rows kernel), same accounting
    if ph_ms.get("rows_items"):
        ia = (ib - (I - n_seg_i) * 48 * D) / (ph_ms["rows_items"] * 1e-3) / 1e9
        roof["item_pass"] = {"kernel": "bwd_rows_ring (item-side segment reduce + Adam)", "achieved": ia,
                             "frac": ia / peak, "bytes_per_launch": ib - (I - n_seg_i) * 48 * D,
                             "ms_per_launch": ph_ms["rows_items"]}
        itr = ncu_traffic().get("item_rows")
        if itr:
            roof["item_pass"]["traffic"] = itr["bytes"]
    if not args.no_cpu_baseline:
        # host-side leg: --steps steps unless its 25 s budget runs out first ("sample" says how many ran)
        line["cpu_baseline"] = cpu_baseline(w, os.cpu_count() or 1, steps=args.steps)
        try:
            line["torch_eager_gpu"] = torch_eager_gpu(w, dev, dbatches[0], steps=args.steps)
            line["torch_eager_gpu"]["speedup_of_value"] = line["value"] / line["torch_eager_gpu"]["value"]
        except Exception as ex:      # noqa: BLE001 -- a baseline leg must never break the bench line
            line["torch_eager_gpu"] = {"unavailable": f"{type(ex).__name__}: {ex}"[:200]}
    if not args.no_config_legs and args.workload == "c5":
        # BASELINE.json configs 2-4 (C1 = Coat on CPU is the reference's own oracle case, parity-tested only)
        del hp, plans, dbatches, stages, plan_bufs, cu, ci, cy, ce, pidx, losses
        torch.cuda.empty_cache()
        line["configs"] = {}
        for name in ("c2", "c3", "c4"):
            try:
                line["configs"][name] = config_leg(name, dev, with_eager=not args.no_cpu_baseline)
            except Exception as ex:      # noqa: BLE001 -- a leg must never break the headline line
                line["configs"][name] = {"unavailable": f"{type(ex).__name__}: {ex}"[:300]}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--nbatch", type=int, default=0,
                    help="distinct synthetic batches cycled through (0 = steps + warmup: every step its own batch)")
    ap.add_argument("--no-config-legs", action="store_true", help="skip the C2/C3/C4 legs of the default line")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the parity_vs_1gpu leg")
    ap.add_argument("--dense-adam", action="store_true", help="headline with plain dense Adam instead of lazy")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the losses and (sampled) parameters of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "ours" or args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs is implemented for the single-GPU path (--impl ours --gpus 1)")
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference(args, w)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback "
                         "(use --impl reference for the CPU baseline)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 or args.gpus > 1:
        from invpref_kdd_2022_b200 import dist_bench
        dist_bench.run(args, w)
        return
    run_ours_single(args, w)


if __name__ == "__main__":
    main()

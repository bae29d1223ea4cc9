#!/usr/bin/env python
"""CUDA-event timing of the fold-in kernel (csrc/foldin.cu) behind ``invpref_fold_in_users`` /
``invpref_fold_in_items``, against a plain-torch fp64 baseline on the same inputs.  GPU only.

    python tools/time_fold_in.py [--repeats R] [--out FILE]

Shapes:
  mind_users / mind_items: implicit, D 40.  The C4 synthetic interactions (4 194 304, bench.py's MIND-shaped config)
      folded in as the histories of its 50 000 users against the 51 283-row item table, and of all 51 283 items
      against the user table.  The item histories are power-law (the longest is reported): the call waits for it.
  c5_users: explicit, D 64.  65 536 users x 64 interactions against the C5 1 M-row item table (256 MB, larger than L2).
  powerlaw_users: explicit, D 64, 65 536 users with power-law history lengths (capped at 200 000) against the C5
      item table; again without the rows of the longest length, and the longest row alone.
The baseline gathers each history into a zero-padded fp64 [rows, L, D] block (rows sorted by length and cut into
blocks that stay under 2 GiB), forms the Gram matrices with ``bmm`` and solves with ``torch.linalg.cholesky`` /
``cholesky_solve``; on the implicit model it runs the same damped Newton iteration (step rule, stopping rule and
Armijo test of the header), vectorised over the rows.  The baseline runs once untimed per shape, then library and
baseline alternate ``--repeats`` times, both timed with CUDA events after an untimed call.  Their results must agree:
the script fails if a row differs by more than 4 ulp32 of its largest entry, or is finite on one side only.
Per shape: milliseconds per call (median), rows per second and the achieved fp64 FMA rate, counted from the shapes as
sum_r n_r * D (D + 1) / 2 per Gram pass plus D^3 / 6 per factorisation, per Newton step.  No share of peak is given:
the project has no measured fp64 peak.  ``recommend_rows`` on the folded users is timed against ``recommend`` at the
same b, D and k.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from invpref_kdd_2022_b200.dataloader import interaction_csr, synthetic_interactions  # noqa: E402
from invpref_kdd_2022_b200.engine import HotPath  # noqa: E402

ARMIJO, HALVINGS = 1e-4, 30


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": out[0], "power_limit_w": float(out[1]), "sm_clock_max_mhz": float(out[2]),
            "sm_clock_mhz_at_query": float(out[3])}


def event_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def hot(U, I, implicit):
    dev = U.device
    E = torch.zeros((1, U.shape[1]), dtype=torch.float32, device=dev)
    return HotPath({"Uinv": U, "Iinv": I, "Uenv": U, "Ienv": I, "E": E, "W": E,
                    "b": torch.zeros(1, dtype=torch.float32, device=dev)}, implicit, False, False)


# ---- plain-torch fp64 baseline ---------------------------------------------------------------------------------------
def _loss_diff(z, dz, y):
    s = torch.sigmoid(z)
    q = s * torch.expm1(dz)
    sp = lambda x: torch.clamp(x, min=0) + torch.log1p(torch.exp(-x.abs()))
    d = torch.where(q > -0.5, torch.log1p(torch.clamp(q, min=-0.5)), sp(z + dz) - sp(z))
    return d - y * dz


def _block(V, ids, y, lens, lam, implicit, max_iter):
    """One padded block: V fp32 table, ids / y padded [R, L] (pad: id 0, mask 0), lens [R] -> fp64 rows [R, D]."""
    R, L = ids.shape
    mask = (torch.arange(L, device=ids.device)[None, :] < lens[:, None]).double()
    Vh = V[ids].double() * mask[..., None]                                      # [R, L, D]
    yh = y.double() * mask
    D = V.shape[1]
    eye = torch.eye(D, dtype=torch.float64, device=V.device) * lam
    if not implicit:
        G = torch.bmm(Vh.transpose(1, 2), Vh) + eye
        return torch.cholesky_solve(torch.bmm(Vh.transpose(1, 2), yh[..., None]), torch.linalg.cholesky(G))[..., 0]
    u = torch.zeros((R, D), dtype=torch.float64, device=V.device)
    live = lens > 0
    for _ in range(max_iter):
        if not bool(live.any()):
            break
        z = torch.bmm(Vh, u[..., None])[..., 0]
        s = torch.sigmoid(z)
        w = s * (1 - s) * mask
        H = torch.bmm(Vh.transpose(1, 2), Vh * w[..., None]) + eye
        g = torch.bmm(Vh.transpose(1, 2), ((s - yh) * mask)[..., None])[..., 0] + lam * u
        dl = -torch.cholesky_solve(g[..., None], torch.linalg.cholesky(H))[..., 0]
        dl = dl * live[:, None]
        conv = dl.abs().amax(1) <= 2.0 ** -30 * torch.clamp(u.abs().amax(1), min=1.0)
        gd, ud, dd = (g * dl).sum(1), (u * dl).sum(1), (dl * dl).sum(1)
        dz = torch.bmm(Vh, dl[..., None])[..., 0]
        t = torch.ones(R, dtype=torch.float64, device=V.device)
        searching = live & ~conv
        for m in range(HALVINGS + 1):
            tm = 2.0 ** -m
            f = (_loss_diff(z, tm * dz, yh) * mask).sum(1) + lam * (tm * ud + 0.5 * tm * tm * dd)
            ok = searching & (f <= ARMIJO * tm * gd)
            t = torch.where(searching, torch.full_like(t, tm), t)
            searching = searching & ~ok
            if not bool(searching.any()):
                break
        t = torch.where(conv, torch.ones_like(t), t)
        u = u + t[:, None] * dl
        live = live & ~conv
    return u


def torch_fold(V, off, ids, y, lam, implicit, max_iter=25, budget=2 << 30):
    lens = (off[1:] - off[:-1])
    order = torch.argsort(lens)
    lens_s = lens[order].cpu().numpy()
    out = torch.zeros((lens.numel(), V.shape[1]), dtype=torch.float64, device=V.device)
    D = V.shape[1]
    r0 = 0
    while r0 < lens_s.size:
        Lmax = max(int(lens_s[r0]), 1)
        R = max(1, int(budget // (Lmax * D * 8 * 3)))
        r1 = min(lens_s.size, r0 + R)
        Lmax = max(int(lens_s[r1 - 1]), 1)
        while r1 - r0 > 1 and (r1 - r0) * Lmax * D * 8 * 3 > budget:
            r1 = r0 + (r1 - r0) // 2
            Lmax = max(int(lens_s[r1 - 1]), 1)
        rows = order[r0:r1]
        st = off[rows]
        pos = st[:, None] + torch.arange(Lmax, device=V.device)[None, :]
        ln = lens[rows]
        valid = torch.arange(Lmax, device=V.device)[None, :] < ln[:, None]
        pos = torch.where(valid, pos, torch.zeros_like(pos))
        out[rows] = _block(V, ids[pos], y[pos], ln, lam, implicit, max_iter)
        r0 = r1
    return out.float()


# ---- shapes ------------------------------------------------------------------------------------------------------
def fma_count(lens, D, steps):
    """sum_r steps_r * (n_r * D (D + 1) / 2 + D^3 / 6)."""
    lens, steps = np.asarray(lens, np.float64), np.asarray(steps, np.float64)
    return float(np.sum(steps * (lens * D * (D + 1) / 2 + D ** 3 / 6)))


def run_shape(name, V, off, ids, y, lam, implicit, fold, repeats, lens_np, with_baseline=True):
    D = V.shape[1]
    rows, iters = fold(off, ids, y, lam, return_iters=True)
    torch.cuda.synchronize()
    steps = np.abs(iters.cpu().numpy())
    res = {"shape": name, "rows": int(off.numel() - 1), "interactions": int(ids.numel()), "D": D,
           "implicit": implicit, "l2": lam, "longest_history": int(lens_np.max()) if lens_np.size else 0,
           "newton_steps_total": int(steps.sum()), "newton_steps_max": int(steps.max()) if steps.size else 0,
           "not_converged": int((iters.cpu().numpy() < 0).sum()), "ours_ms": [], "torch_ms": []}
    base = torch_fold(V, off, ids, y, lam, implicit) if with_baseline else None      # also the baseline's warm-up
    for _ in range(repeats):
        # both sides timed the same way: CUDA events around the calls, each after an untimed call
        res["ours_ms"].append(event_ms(lambda: fold(off, ids, y, lam), 3))
        if with_baseline:
            res["torch_ms"].append(event_ms(lambda: torch_fold(V, off, ids, y, lam, implicit), 1))
    ms = float(np.median(res["ours_ms"]))
    fl = fma_count(lens_np, D, steps)
    res.update(ours_ms_median=ms, rows_per_s=res["rows"] / (ms / 1e3), fp64_fma=fl, fp64_fma_per_s=fl / (ms / 1e3))
    if with_baseline:
        tm = float(np.median(res["torch_ms"]))
        fin = torch.isfinite(rows).all(1)
        if not torch.equal(fin, torch.isfinite(base).all(1)):
            raise AssertionError(f"{name}: library and baseline disagree on which rows are finite")
        err = (rows[fin] - base[fin]).abs().amax(1)
        tol = 2.0 ** -21 * rows[fin].abs().amax(1) + 1e-30                 # 4 ulp32 of the row's largest entry
        if bool((err > tol).any()):
            raise AssertionError(f"{name}: library and baseline differ by {err.max().item()} (tolerance "
                                 f"{tol[err > tol][0].item()})")
        res.update(torch_ms_median=tm, speedup=tm / ms, max_abs_diff=err.max().item() if err.numel() else 0.0,
                   max_abs_row=rows[fin].abs().max().item() if bool(fin.any()) else 0.0)
    print(json.dumps({k: v for k, v in res.items() if not isinstance(v, list)}), flush=True)
    return res, rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default="profiles/r5_fold_in.json")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    info = gpu_info()
    print(json.dumps(info), flush=True)
    out = {"gpu": info, "shapes": []}
    g = torch.Generator(device=dev).manual_seed(5)
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)

    # MIND-shaped implicit, D 40
    U = torch.randn((50_000, 40), generator=g, device=dev) * 0.3
    I = torch.randn((51_283, 40), generator=g, device=dev) * 0.3
    hp = hot(U, I, True)
    data = synthetic_interactions(50_000, 51_283, 4_194_304, True)
    for side, (rr, cc, n_rows) in (("users", (data[:, 0], data[:, 1], 50_000)), ("items", (data[:, 1], data[:, 0], 51_283))):
        off, cols, ys = interaction_csr(rr, cc, data[:, 2], n_rows)
        fold = hp.fold_in_users if side == "users" else hp.fold_in_items
        V = I if side == "users" else U
        r, rows = run_shape(f"mind_{side}", V, t(off), t(cols), t(ys), 1.0, True, fold, args.repeats, np.diff(off))
        out["shapes"].append(r)
        if side == "users":
            k = 50
            users = torch.arange(50_000, device=dev)
            r2 = {"shape": "mind_recommend_rows_vs_recommend", "b": 50_000, "k": k, "D": 40,
                  "recommend_rows_ms": event_ms(lambda: hp.recommend_rows(rows, k), 3),
                  "recommend_ms": event_ms(lambda: hp.recommend(users, k), 3)}
            print(json.dumps(r2), flush=True)
            out["shapes"].append(r2)
    del hp, U, I

    # C5-shaped explicit, D 64, 1 M-row item table
    I = torch.randn((1_000_000, 64), generator=g, device=dev) * 0.3
    U = torch.randn((1024, 64), generator=g, device=dev) * 0.3
    hp = hot(U, I, False)
    rng = np.random.default_rng(7)
    b = 65_536
    off = np.arange(b + 1, dtype=np.int64) * 64
    ids = rng.integers(0, 1_000_000, b * 64)
    ys = rng.integers(1, 6, b * 64).astype(np.float32)
    r, rows = run_shape("c5_users", I, t(off), t(ids), t(ys), 1.0, False, hp.fold_in_users, args.repeats, np.diff(off))
    out["shapes"].append(r)
    r2 = {"shape": "c5_recommend_rows_vs_recommend", "b": 4096, "k": 50, "D": 64}
    hp_u = hot(rows[:4096].contiguous(), I, False)          # the folded rows as a user table: recommend at equal b
    users = torch.arange(4096, device=dev)
    r2["recommend_rows_ms"] = event_ms(lambda: hp.recommend_rows(rows[:4096], 50), 3)
    r2["recommend_ms"] = event_ms(lambda: hp_u.recommend(users, 50), 3)
    a, _ = hp.recommend_rows(rows[:4096], 50)
    b_, _ = hp_u.recommend(users, 50)
    r2["same_items"] = bool(torch.equal(a, b_))
    print(json.dumps(r2), flush=True)
    out["shapes"].append(r2)

    # power-law history lengths, explicit, D 64: with and without the longest row
    lens = np.minimum(np.floor(1.0 / (1.0 - rng.random(b)) ** 1.2).astype(np.int64), 200_000)
    off = np.zeros(b + 1, np.int64)
    off[1:] = np.cumsum(lens)
    n = int(off[-1])
    ids = rng.integers(0, 1_000_000, n)
    ys = rng.integers(1, 6, n).astype(np.float32)
    r, _ = run_shape("powerlaw_users", I, t(off), t(ids), t(ys), 1.0, False, hp.fold_in_users, args.repeats, lens)
    out["shapes"].append(r)
    j = int(np.argmax(lens))
    keep = np.flatnonzero(lens < lens[j])                   # every row of the longest length left out
    off2 = np.zeros(keep.size + 1, np.int64)
    off2[1:] = np.cumsum(lens[keep])
    sel = np.concatenate([np.arange(off[i], off[i + 1]) for i in keep])
    r, _ = run_shape("powerlaw_users_without_longest", I, t(off2), t(ids[sel]), t(ys[sel]), 1.0, False,
                     hp.fold_in_users, args.repeats, lens[keep], with_baseline=False)
    r["rows_left_out"] = int(b - keep.size)
    out["shapes"].append(r)
    one = np.array([0, lens[j]], np.int64)
    r, _ = run_shape("powerlaw_longest_row_alone", I, t(one), t(ids[off[j]:off[j + 1]]), t(ys[off[j]:off[j + 1]]), 1.0,
                     False, hp.fold_in_users, args.repeats, lens[j:j + 1], with_baseline=False)
    out["shapes"].append(r)

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()

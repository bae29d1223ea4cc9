"""GPU, the EM re-assignment (cluster.cu) against an exact reference: every instantiation of the plain and the
user-sorted kernel, the tie-break table, the steady state of the staging ring, env_hist and stat_envs.

Why the inputs look the way they do:

  * Exactness.  Every table entry is a small integer times 2^-3 in [-1, 1].  Every product and partial sum the kernel
    forms (Uinv . Iinv, (Uenv * Ienv) * E, up to D = 256) is then a multiple of 2^-9 below 2^20 ulps: exact in fp32 in
    any summation order.  So z1 and every zk equal the fp64 per-pair tables Z1 = Uinv Iinv^T and
    ZK = einsum(ud, id, kd -> uik), and the explicit distance ((z1 + zk) - y)^2 + eps[pidx] can be restated in numpy fp32
    with the kernel's three roundings (add, subtract, square, add).  new_envs, hist and diff must then be EQUAL, with no
    near-tie exemption: the tie-break table (1e-10 * 0.1^k, train.py:763-769) only decides where distances agree to
    ~1e-10, which the tolerance-based tests elsewhere have to exempt.
  * Explicit regimes, mixed in one batch: (A) users whose env-aware row is zero and y = z1, so all K distances are
    exactly 0 and the eps row alone decides (table indexing, the smem table for K <= 6 and the global one for K = 7, 8,
    every row of K!); (B) y = z1 + zk* + delta with delta in {1, 3} 2^-12, 2^-8, 2^-6: distances near 6e-8 .. 2.4e-4,
    where only some eps values survive the fp32 add and the first minimum among the collapsed ones decides; (C) two E
    rows equal on the dims that a quarter of the items use: exact ties on a subset of k, with and without the
    tie-break table; (D) y = z1 + zk* or a rating: clear margins.  A second model (E) scales chosen E rows by 2^80 (still
    dyadic; a nonzero zk is at least 2^-9, so |r| >= 2^71): r^2 overflows for those k only, and y = 2^100 makes every k +inf, which must resolve to k = 0 past the
    +inf padding lanes of K = 3, 5, 7.
  * Implicit: sigmoid and log are not bit-reproducible, so equality is asserted on the samples whose answer does not
    depend on ulps, and each such regime must cover its share of the batch: saturated samples (z1, zk >= 64 with y = 1,
    or zk <= -96 with y = 0: the distance is +-0 for every k and the eps row decides), ties between the two equal E rows
    at a distance >= 2^-3 (eps is absorbed: the lower k wins), and a margin of 1e-3 relative (1e-5 absolute) against
    an fp64 restatement.  The rest must still agree between the two kernels bit for bit.
  * Batch sizes.  The grid is capped at 148 * 16 CTAs of 16 groups, so a group handles samples S = 37 888 apart.  The
    ring has ST = 3 slots (2 for VEC * NV = 16); a slot is re-filled in the loop only when a group has more than ST
    samples, the ids are loaded two iterations ahead and the scalars one.  Every instantiation therefore runs at
    B = (ST + 2) S + 5; the sizes 1, 16, 17, S - 1, S, S + 1, ST S, ST S + 1 and one of ~10^6 with a ragged tail run
    on three geometries.  The user-sorted kernel gives each group ceil(B / S) consecutive samples of the sorted view;
    users are drawn from a power law (runs longer than 10^4, every fifth user absent), so runs cross group bounds.
  * Every call runs with the tie-break table present and absent, crossed with the old environments (and so the diff
    count) present and absent, into one reused ``out=`` tensor that is pre-filled with -1 so a missing write shows.

Also here: the trainer's ``sorted_cluster=True`` path against the default one, and a NaN distance (a diverged
explicit model), which must give the first NaN environment as torch.argmin / np.argmin do.
"""
import re
from collections import Counter

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

from oracle import invpref_numpy as on

pytestmark = pytest.mark.gpu

S = 148 * 16 * 16                   # grid stride of the plain kernel: CTAs (launch_cluster's cap) x groups per CTA
U, I = 3000, 61                     # every fifth user has no sample (ABSENT), user 0 has > 10^4 at B >= 10^6
Q = 0.125                           # table entries are integers times Q


def _dev():
    return torch.device("cuda:0")


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


def stages(D, K):
    """cluster.cu cl_stages: ring depth."""
    vec, nv, _ = geometry(D, K)
    return 3 if vec * nv <= 8 else 2


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


# Every (VEC, NV, KT, DX) instantiation of cluster_kernel / cluster_sorted_kernel and a (D, K) that dispatches to it.
# K = 1 (one-row eps table), K = 3, 5, 7 (+inf padding lanes), K = 7, 8 (eps table in global memory), and the variants
# with E in shared memory (KT * VEC * NV > 32: (4, 2) with KT 6 / 8, (4, 4) with KT >= 4).
INSTANCES = [
    ((4, 1, 2, 0), 64, 1), ((4, 1, 4, 0), 40, 3), ((4, 1, 6, 0), 64, 5), ((4, 1, 8, 0), 44, 7),
    ((4, 2, 2, 0), 68, 2), ((4, 2, 4, 0), 96, 4), ((4, 2, 6, 0), 124, 6), ((4, 2, 8, 0), 128, 8),
    ((4, 4, 2, 0), 132, 2), ((4, 4, 4, 0), 200, 3), ((4, 4, 6, 0), 252, 6), ((4, 4, 8, 0), 256, 8),
    ((2, 1, 2, 0), 30, 1), ((2, 1, 4, 0), 14, 4), ((2, 1, 6, 0), 10, 5), ((2, 1, 8, 0), 6, 8),
    ((2, 2, 2, 0), 34, 2), ((2, 2, 4, 0), 50, 3), ((2, 2, 6, 0), 62, 6), ((2, 2, 8, 0), 46, 7),
    ((1, 4, 2, 0), 3, 2), ((1, 4, 4, 0), 33, 4), ((1, 4, 6, 0), 63, 5), ((1, 4, 8, 0), 33, 8),
    ((4, 1, 2, 64), 64, 2), ((4, 1, 4, 64), 64, 4), ((4, 1, 6, 64), 64, 6), ((4, 1, 8, 64), 64, 8),
    ((4, 1, 2, 40), 40, 2), ((4, 1, 4, 40), 40, 4), ((4, 1, 5, 40), 40, 5), ((4, 1, 6, 40), 40, 6),
    ((4, 1, 8, 40), 40, 8),
]


def _case_id(v):
    return "x".join(map(str, v)) if isinstance(v, tuple) else str(v)


def _kernel_name(inst, sorted_):
    return f"cluster_{'sorted_' if sorted_ else ''}kernel<{', '.join(map(str, inst))}>"


def _dup_pair(K):
    """The two E rows that are equal on the dims [0, h): (1, 3) from K = 4 on."""
    return None if K == 1 else ((0, 1) if K == 2 else ((0, 2) if K == 3 else (1, 3)))


def _ints(rng, shape, lim=8):
    return rng.integers(-lim, lim + 1, shape).astype(np.float64) * Q


def _tables(D, K, seed, implicit=False):
    """Dyadic tables.  Users u % 8 == 0 have a zero env-aware row (zk = 0 for every k); items i % 4 == 0 have a zero
    env-aware row on the dims [h, D), where the duplicated E rows differ.  implicit: users u % 8 == 1 and items
    i % 8 == 1 (i % 8 == 2) carry +-8 on dim 0 only, with E[:, 0] in {1.5, 2}: saturated sigmoids."""
    rng = np.random.default_rng(seed)
    h = max(1, D // 2)
    T = {"Uinv": _ints(rng, (U, D)), "Iinv": _ints(rng, (I, D)), "Uenv": _ints(rng, (U, D)),
         "Ienv": _ints(rng, (I, D)), "E": _ints(rng, (K, D)), "W": np.zeros((K, D)), "b": np.zeros(K)}
    T["Uenv"][::8] = 0.0
    T["Ienv"][::4, h:] = 0.0
    if implicit:
        T["E"][:, 0] = rng.choice([1.5, 2.0], K)
        e0 = np.zeros(D)
        e0[0] = 8.0
        T["Uinv"][1::8] = e0
        T["Uenv"][1::8] = e0
        T["Iinv"][1::8] = e0
        T["Ienv"][1::8] = e0
        T["Ienv"][2::8] = -e0
    pair = _dup_pair(K)
    if pair is not None:
        a, b = pair
        T["E"][b, :h] = T["E"][a, :h]
        T["E"][b, h:] = T["E"][a, h:] + Q
    return T


def _pair_tables(T):
    """Z1 [U, I] and ZK [U, I, K] in fp64: exact for these tables."""
    Z1 = T["Uinv"] @ T["Iinv"].T
    K = T["E"].shape[0]
    ZK = np.empty((U, I, K))
    for s in range(0, U, 250):
        ZK[s:s + 250] = np.einsum("ud,id,kd->uik", T["Uenv"][s:s + 250], T["Ienv"], T["E"], optimize=True)
    assert np.array_equal(Z1.astype(np.float32), Z1) and np.array_equal(ZK.astype(np.float32), ZK)
    return Z1, ZK


PRESENT = np.flatnonzero(np.arange(U) % 5 != 4)
ZERO_ENV_USERS = PRESENT[PRESENT % 8 == 0]


def _power_law(rng, pool, n):
    return pool[np.floor(len(pool) * rng.random(n) ** 3).astype(np.int64)]


def _ids(rng, N):
    return _power_law(rng, PRESENT, N), rng.integers(0, I, N)


def _explicit_scores(rng, u, i, Z1, ZK, scaled=()):
    """Per-sample regimes A-D (module docstring); with scaled E rows (model E) the regimes are all-inf (y = 2^100), a
    rating, and y = z1 + zk* for an unscaled k*."""
    N, K = len(u), ZK.shape[2]
    reg = rng.integers(0, 4, N)
    a = reg == 0
    u = u.copy()
    u[a] = _power_law(rng, ZERO_ENV_USERS, int(a.sum()))
    z1, zk = Z1[u, i], ZK[u, i]
    free = [k for k in range(K) if k not in scaled] or [None]
    ks = np.asarray(free)[rng.integers(0, len(free), N)]
    zs = zk[np.arange(N), ks] if free[0] is not None else np.zeros(N)
    rating = rng.integers(1, 6, N).astype(np.float64)
    if scaled:                          # K = 1: no unscaled row, regime 2 is a rating as well
        y = np.where(reg == 0, 2.0 ** 100, np.where((reg == 1) | (free[0] is None), rating, z1 + zs))
    else:
        delta = rng.choice([1.0, 3.0, 16.0, 64.0], N) * rng.choice([-1.0, 1.0], N) * 2.0 ** -12
        y = np.select([reg == 0, reg == 1, reg == 2], [z1, z1 + zs + delta, z1 + zs], rating)
    assert np.array_equal(y.astype(np.float32), y)
    return u, y.astype(np.float32)


def _explicit_dist(z1, zk, y):
    """((z1 + zk) - y)^2 in fp32, one rounding per operation as in the kernel (and in torch)."""
    with np.errstate(over="ignore", invalid="ignore"):
        r = (z1.astype(np.float32)[:, None] + zk.astype(np.float32)) - y[:, None]
        return r * r


def _argmin_eps(d, eps_rows):
    with np.errstate(invalid="ignore"):
        return np.argmin(d if eps_rows is None else d + eps_rows, axis=1).astype(np.int64)


def _hot(T, implicit):
    from invpref_kdd_2022_b200.engine import HotPath
    return HotPath({k: torch.tensor(v.astype(np.float32), device=_dev()) for k, v in T.items()}, implicit, False, True)


def _run_all(hp, inst, u, i, y, old, pidx, eps, want, tag, mask=None, check_names=True):
    """Plain and user-sorted kernel, tie-break table (pidx, eps) present / absent x old environments present / absent,
    all into one reused out= tensor pre-filled with -1.  want[tb]: expected environments with (tb = True) and without
    the table; mask: the samples whose expectation is defined (None: all).  The two kernels must agree everywhere."""
    K, N = hp.n_envs, len(u)
    du, di, dy = (torch.tensor(a, device=_dev()) for a in (u, i, y))
    dold, dp = torch.tensor(old, device=_dev()), torch.tensor(pidx, device=_dev())
    view = hp.sorted_view(du, di, dy)
    out = torch.empty(N, dtype=torch.int64, device=_dev())
    for tb in (True, False):
        for od in (True, False):
            args = (dp if tb else None, eps if tb else None, dold if od else None)
            got = {}
            for sorted_ in (False, True):
                out.fill_(-1)
                fn = ((lambda: hp.cluster_sorted(view, *args, out=out)) if sorted_ else
                      (lambda: hp.cluster(du, di, dy, *args, trusted=True, out=out)))
                if check_names and tb and od:
                    (new, hist, diff), names = _launched(fn)
                    _assert_ran(names, [(_kernel_name(inst, sorted_), 1)], (tag, sorted_))
                else:
                    new, hist, diff = fn()
                assert new is out
                g = new.cpu().numpy()
                c = (tag, "sorted" if sorted_ else "plain", "eps" if tb else "no eps", "old" if od else "no old")
                assert ((g >= 0) & (g < K)).all(), (c, int((g < 0).sum()))
                w, m = want[tb], (slice(None) if mask is None else mask)
                bad = np.flatnonzero(g[m] != w[m])
                assert len(bad) == 0, (c, len(bad), bad[:8])
                assert np.array_equal(hist.cpu().numpy(), np.bincount(g, minlength=K)), c
                assert int(diff) == (int((g != old).sum()) if od else 0), c
                got[sorted_] = g
            assert np.array_equal(got[False], got[True]), (tag, tb, od)


def _explicit_case(inst, D, K, N, seed, scaled=(), check_names=True):
    """Model A-D (scaled = ()) or model E (scaled: E rows multiplied by 2^80) on N samples.  Returns the fp32 distances
    without the table, and the data drawn."""
    tag = (inst, D, K, N, "E" if scaled else "A-D")
    T = _tables(D, K, seed)
    Z1, ZK = _pair_tables(T)
    for k in scaled:
        T["E"][k] *= 2.0 ** 80
        ZK[:, :, k] *= 2.0 ** 80
    rng = np.random.default_rng(seed + 1)
    u, i = _ids(rng, N)
    u, y = _explicit_scores(rng, u, i, Z1, ZK, scaled)
    eps_np = on.init_eps(K)
    pidx = rng.integers(0, eps_np.shape[0], N)
    old = rng.integers(0, K, N)
    d = _explicit_dist(Z1[u, i], ZK[u, i], y)
    want = {True: _argmin_eps(d, eps_np[pidx]), False: _argmin_eps(d, None)}
    hp = _hot(T, False)
    assert geometry(D, K)[:2] == inst[:2] and (inst[3] > 0 or geometry(D, K)[2] == inst[2])
    _run_all(hp, inst, u, i, y, old, pidx, torch.tensor(eps_np, device=_dev()), want, tag, check_names=check_names)
    return d, want, u, pidx, eps_np


def _check_explicit_coverage(d, want, pidx, eps_np, K, tag):
    """Each regime of the batch is present in the share it was drawn with."""
    dmin = d.min(1)
    nmin = (d == dmin[:, None]).sum(1)
    assert (d == 0).all(1).mean() > 0.2, tag                                          # A
    assert ((dmin > 0) & (dmin < 2.0 ** -10)).mean() > 0.15, tag                     # B
    if K >= 2:
        assert ((dmin > 0) & (nmin >= 2)).mean() > 0.01, tag                          # C
        assert (want[True] != want[False]).mean() > 0.1, tag                          # the table decides
        de = d + eps_np[pidx]
        if K >= 4:                                                                    # eps absorbed in the add
            collapsed = (de == de.min(1)[:, None]).sum(1) >= 2
            assert (collapsed & (dmin > 0)).sum() > 100, tag


def _check_inf_coverage(d, K, tag):
    inf = np.isinf(d)
    assert inf.all(1).mean() > 0.2, tag
    if K >= 2:
        assert (inf.any(1) & ~inf.all(1)).mean() > 0.2, tag


def _scaled_rows(K):
    return tuple(k for k in range(K) if k % 3 == 1) or (0,)


@pytest.mark.parametrize("inst,D,K", INSTANCES, ids=_case_id)
def test_every_instantiation_exact(inst, D, K):
    """Explicit models A-D and E at B = (ST + 2) S + 5: every group re-fills each ring slot in the loop."""
    N = (stages(D, K) + 2) * S + 5
    d, want, _, pidx, eps_np = _explicit_case(inst, D, K, N, 1000 * D + K)
    _check_explicit_coverage(d, want, pidx, eps_np, K, (inst, "A-D"))
    d, _, _, _, _ = _explicit_case(inst, D, K, N, 2000 * D + K, scaled=_scaled_rows(K))
    _check_inf_coverage(d, K, (inst, "E"))


def _implicit_ref(z1, zk, y):
    """BCE distance in fp64 with the reference's clamp of log at -100."""
    sig = lambda x: 1.0 / (1.0 + np.exp(-x))
    with np.errstate(over="ignore", divide="ignore"):
        s = sig(z1)[:, None] * sig(zk)
        yy = y.astype(np.float64)[:, None]
        return -(yy * np.maximum(np.log(s), -100.0) + (1.0 - yy) * np.maximum(np.log1p(-s), -100.0))


@pytest.mark.parametrize("inst,D,K", INSTANCES, ids=_case_id)
def test_every_instantiation_implicit_where_decidable(inst, D, K):
    """Implicit model: saturated samples (eps decides), duplicated-row ties at d >= 2^-3 (the lower k), margins of
    1e-3; every regime must cover its share, and the two kernels agree everywhere."""
    N = (stages(D, K) + 2) * S + 5
    seed = 3000 * D + K
    T = _tables(D, K, seed, implicit=True)
    Z1, ZK = _pair_tables(T)
    rng = np.random.default_rng(seed + 1)
    u, i = _ids(rng, N)
    reg = rng.integers(0, 4, N)
    sat_users = PRESENT[PRESENT % 8 == 1]
    u[reg <= 1] = _power_law(rng, sat_users, int((reg <= 1).sum()))
    i[reg == 0] = 8 * rng.integers(0, (I - 2) // 8 + 1, int((reg == 0).sum())) + 1       # z1, zk >= 64, y = 1
    i[reg == 1] = 8 * rng.integers(0, (I - 3) // 8 + 1, int((reg == 1).sum())) + 2       # zk <= -96, y = 0
    y = np.where(reg == 0, 1.0, np.where(reg == 1, 0.0, rng.integers(0, 2, N))).astype(np.float32)
    z1, zk = Z1[u, i], ZK[u, i]
    sat = ((z1 >= 20) & (zk >= 20).all(1) & (y == 1)) | ((zk <= -90).all(1) & (y == 0))
    assert sat[reg <= 1].all(), (inst, "saturation")
    d = _implicit_ref(z1, zk, y)
    srt = np.sort(d, 1)
    dmin = srt[:, 0]
    nmin = (d == dmin[:, None]).sum(1)
    nxt = np.where(nmin < K, np.take_along_axis(srt, np.minimum(nmin, K - 1)[:, None], 1)[:, 0], np.inf)
    margin = (nxt - dmin >= np.maximum(1e-3 * dmin, 1e-5)) & (dmin < 50) & ~sat     # far from the log clamp
    tie = margin & (nmin >= 2) & (dmin >= 0.125)
    uniq = margin & (nmin == 1)
    eps_np = on.init_eps(K)
    pidx = rng.integers(0, eps_np.shape[0], N)
    old = rng.integers(0, K, N)
    first = np.argmin(d, 1)
    want = {True: np.where(sat, np.argmin(eps_np[pidx], 1), first), False: np.where(sat, 0, first)}
    assert sat.mean() > 0.45 and uniq.mean() > 0.12, (inst, sat.mean(), uniq.mean())
    if K >= 2:
        assert tie.mean() > 0.05, (inst, tie.mean())
    hp = _hot(T, True)
    _run_all(hp, inst, u, i, y, old, pidx, torch.tensor(eps_np, device=_dev()), want, (inst, "implicit"),
             mask=sat | tie | uniq)


# (instantiation, D, K) of the batch-size sweep: exact D = 64 K = 4; D = 256 K = 8 (ST = 2, E in shared memory,
# global eps table); D = 33 K = 5 (VEC = 1, padding lanes)
SIZE_GEOMS = [((4, 1, 4, 64), 64, 4), ((4, 4, 8, 0), 256, 8), ((1, 4, 6, 0), 33, 5)]


def _sizes(st):
    return [1, 16, 17, S - 1, S, S + 1, st * S, st * S + 1, 27 * S + 12345]


@pytest.mark.parametrize("inst,D,K", SIZE_GEOMS, ids=_case_id)
@pytest.mark.parametrize("j", range(9))
def test_batch_sizes_around_the_stride(inst, D, K, j):
    N = _sizes(stages(D, K))[j]
    d, want, u, pidx, eps_np = _explicit_case(inst, D, K, N, 7 * N + D, check_names=(j == 0))
    if N >= 10 ** 6:
        per = -(-N // S)
        assert 2 <= per <= 30
        su = np.sort(u)
        assert np.bincount(u).max() > 10 ** 4 and len(np.unique(u)) < u.max() + 1
        bounds = np.arange(per, N, per)
        assert (su[bounds - 1] == su[bounds]).sum() > 1000            # group bounds inside a user's run
        _check_explicit_coverage(d, want, pidx, eps_np, K, (inst, N))


@pytest.mark.parametrize("K", range(1, 9))
@pytest.mark.parametrize("N", [1, 2, S + 1, 3 * 10 ** 6 + 7])
def test_env_hist_and_stat_envs_exact(K, N):
    """Histogram against np.bincount, class and sample weights against oracle.stat_envs, with the
    min(cnt + 1, N - 1) cap (it binds at N = 1, 2 and for K = 1)."""
    T = {"Uinv": np.zeros((1, 4)), "Iinv": np.zeros((1, 4)), "Uenv": np.zeros((1, 4)), "Ienv": np.zeros((1, 4)),
         "E": np.zeros((K, 4)), "W": np.zeros((K, 4)), "b": np.zeros(K)}
    hp = _hot(T, False)
    rng = np.random.default_rng(N + K)
    envs = np.minimum(np.floor(K * rng.random(N) ** 2), K - 1).astype(np.int64)     # skewed: some counts differ a lot
    de = torch.tensor(envs, device=_dev())
    hist = hp.env_hist(de)
    cnt, cw, sw = on.stat_envs(envs, K, N)
    assert np.array_equal(hist.cpu().numpy(), cnt), (K, N)
    out = torch.full((N,), -1.0, device=_dev())
    cw_d, sw_d = hp.stat_envs(de, hist, out=out)
    assert sw_d is out
    assert np.array_equal(cw_d.cpu().numpy(), cw), (K, N, cw_d.cpu().numpy(), cw)
    assert np.array_equal(sw_d.cpu().numpy(), sw), (K, N)


@pytest.mark.parametrize("inst,D,K,nan_rows", [((4, 1, 4, 64), 64, 4, (2,)), ((4, 4, 8, 0), 256, 8, (3, 6))],
                         ids=_case_id)
def test_nan_distance_gives_the_first_nan_environment(inst, D, K, nan_rows):
    """An explicit model with non-finite E rows (a diverged run): np.argmin / torch.argmin return the first NaN
    distance.  Users u % 7 == 3 have a NaN env-aware row and some scores are NaN: every k is NaN there, k = 0 wins."""
    N = 3 * S + 11
    T = _tables(D, K, D + K)
    Z1, ZK = _pair_tables(T)
    nan_users = np.arange(U) % 7 == 3
    for k in nan_rows:
        T["E"][k, D // 3] = np.nan
        ZK[:, :, k] = np.nan
    T["Uenv"][nan_users, 0] = np.nan
    ZK[nan_users] = np.nan
    rng = np.random.default_rng(5)
    u, i = _ids(rng, N)
    y = rng.integers(1, 6, N).astype(np.float32)
    y[rng.random(N) < 0.05] = np.nan
    d = _explicit_dist(Z1[u, i], ZK[u, i], y)
    eps_np = on.init_eps(K)
    pidx = rng.integers(0, eps_np.shape[0], N)
    want = {True: _argmin_eps(d, eps_np[pidx]), False: _argmin_eps(d, None)}
    assert (want[False] == nan_rows[0]).mean() > 0.5 and (want[False] == 0).mean() > 0.1
    hp = _hot(T, False)
    _run_all(hp, inst, u, i, y, rng.integers(0, K, N), pidx, torch.tensor(eps_np, device=_dev()), want, (inst, "nan"))


def test_trainer_sorted_cluster_matches_the_default():
    """ExplicitTrainManager.cluster() with sorted_cluster=True against the default path, on 4 S + 1234 interactions
    (five samples per group of the sorted kernel), twice with an epoch in between, each time with the reference's
    numpy tie-break stream in the same state: environments, diff counts, class and sample weights identical."""
    from invpref_kdd_2022_b200.models import InvPrefExplicit
    from invpref_kdd_2022_b200.train import ExplicitTrainManager

    class NullEvaluator:
        def evaluate(self):
            return {"mse": 0.0}

    dev = _dev()
    K, D, N = 4, 64, 4 * S + 1234
    rng = np.random.default_rng(11)
    u, i = _ids(rng, N)
    data = np.stack([u, i, rng.integers(1, 6, N)], axis=1).astype(np.int64)
    torch.manual_seed(3)
    np.random.seed(3)
    model = InvPrefExplicit(U, I, K, D, True, False).to(dev)
    tm = ExplicitTrainManager(model=model, evaluator=NullEvaluator(), device=dev,
                              training_data=torch.LongTensor(data).to(dev), batch_size=1 << 15, epochs=3,
                              cluster_interval=1, evaluate_interval=1, lr=1e-2, invariant_coe=0.8, env_aware_coe=1.7,
                              env_coe=1.1, L2_coe=0.6, L1_coe=0.03, alpha=1.3, use_class_re_weight=True,
                              use_recommend_re_weight=True)
    assert not tm.sorted_cluster
    tm.stat_envs()
    diffs = []
    for r in range(2):
        tm.train_a_epoch()
        old = tm.envs
        got = {}
        for sorted_ in (False, True):
            tm.sorted_cluster = sorted_
            tm.envs = old
            np.random.seed(100 + r)
            diff = tm.cluster()
            cnt = tm.stat_envs()
            got[sorted_] = (tm.envs.cpu().numpy(), diff, cnt, tm.class_weights.cpu().numpy(),
                            tm.sample_weights.cpu().numpy())
        a, b = got[False], got[True]
        assert np.array_equal(a[0], b[0]) and a[1] == b[1] and a[2] == b[2], r
        assert np.array_equal(a[3], b[3]) and np.array_equal(a[4], b[4]), r
        assert a[1] == int((a[0] != old.cpu().numpy()).sum())
        diffs.append(a[1])
    assert tm._cl_view is not None and all(d > 0 for d in diffs), diffs

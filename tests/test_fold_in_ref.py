"""CPU: the fp64 fold-in references the GPU tests compare against (tests/_foldin_ref.py), checked against scipy and
numpy solvers, and dataloader.interaction_csr against a brute-force grouping."""
import numpy as np
import pytest
from scipy import optimize

import _foldin_ref as ref
from invpref_kdd_2022_b200 import dataloader


def _problem(kind, n, D, seed, scale=0.3):
    rng = np.random.default_rng(seed)
    V = rng.normal(0, scale, (n, D)).astype(np.float32).astype(np.float64)
    if kind == "random":
        y = (rng.random(n) < 0.5).astype(np.float64)
    elif kind == "separable":                    # labels a hyperplane separates exactly: only l2 keeps u finite
        w = rng.normal(size=D)
        y = (V @ w > 0).astype(np.float64)
    elif kind == "fractional":
        y = rng.random(n).astype(np.float32).astype(np.float64)
    elif kind == "positive":
        y = np.ones(n)
    else:                                        # row norms of 30: saturated sigmoids, slow curvature
        V *= 30.0 / np.linalg.norm(V, axis=1, keepdims=True)
        y = (rng.random(n) < 0.5).astype(np.float64)
    return V, y


@pytest.mark.parametrize("kind", ["random", "separable", "fractional", "positive", "large"])
@pytest.mark.parametrize("D,n,lam", [(3, 40, 1.0), (8, 200, 1e-2), (17, 30, 1e-3), (40, 500, 1.0)])
def test_newton_reaches_the_scipy_minimiser(kind, D, n, lam):
    V, y = _problem(kind, n, D, seed=D * 1000 + n)
    u, it = ref.newton(V, y, lam, max_iter=200)
    assert 1 <= it <= 200
    res = optimize.minimize(ref.objective, np.zeros(D), args=(V, y, lam), jac=ref.gradient, hess=ref.hessian,
                            method="trust-exact", options={"gtol": 1e-13, "maxiter": 2000})
    kappa = ref.condition(V, y, lam, u, implicit=True)
    scale = max(1.0, np.abs(u).max())
    # both stop at the same optimum: the distance is what the smaller of the two gradients allows, times 1 / l2
    gmin = min(np.abs(ref.gradient(u, V, y, lam)).max(), np.abs(ref.gradient(res.x, V, y, lam)).max())
    assert np.abs(u - res.x).max() <= 1e-9 * kappa * scale + 10 * np.abs(ref.gradient(res.x, V, y, lam)).max() / lam
    assert np.abs(ref.gradient(u, V, y, lam)).max() <= 1e-9 * max(1.0, lam * scale) + gmin * 10


@pytest.mark.parametrize("seed", [1134, 2570])
def test_backtracking_engages(seed):
    V, y, lam = ref.damped_problem(seed)
    steps = []
    u, it = ref.newton(V, y, lam, max_iter=100, steps=steps)
    assert 1 <= it <= 100 and min(steps) < 1.0
    res = optimize.minimize(ref.objective, np.zeros(V.shape[1]), args=(V, y, lam), jac=ref.gradient,
                            hess=ref.hessian, method="trust-exact", options={"gtol": 1e-12, "maxiter": 2000})
    assert ref.objective(u, V, y, lam) <= res.fun + 1e-12 * abs(res.fun)


def test_first_step():
    V, y = _problem("random", 60, 8, seed=5)
    u1, it1 = ref.newton(V, y, 1e-2, max_iter=1)
    assert it1 == -1
    g = ref.gradient(np.zeros(8), V, y, 1e-2)
    assert np.allclose(u1, np.linalg.solve(ref.hessian(np.zeros(8), V, y, 1e-2), -g), rtol=1e-14, atol=0)
    assert ref.objective(u1, V, y, 1e-2) < ref.objective(np.zeros(8), V, y, 1e-2)


def test_empty_history_is_zero():
    u, it = ref.newton(np.zeros((0, 5)), np.zeros(0), 1.0)
    assert it == 0 and not u.any()


@pytest.mark.parametrize("D,n,lam", [(1, 1, 1e-3), (3, 2, 1.0), (17, 16, 1e-3), (40, 41, 1e3), (64, 1000, 1.0)])
def test_explicit_closed_form_matches_least_squares(D, n, lam):
    rng = np.random.default_rng(n + D)
    V = rng.normal(0, 0.3, (n, D)).astype(np.float32).astype(np.float64)
    y = rng.integers(1, 6, n).astype(np.float64)
    u = ref.explicit(V, y, lam)
    A = np.vstack([V, np.sqrt(lam) * np.eye(D)])
    want = np.linalg.lstsq(A, np.concatenate([y, np.zeros(D)]), rcond=None)[0]
    kappa = ref.condition(V, y, lam)
    assert np.abs(u - want).max() <= 64 * (D + n) * kappa * 2.0 ** -53 * max(1.0, np.abs(want).max())


@pytest.mark.parametrize("seed", range(4))
def test_interaction_csr_groups_stably(seed):
    rng = np.random.default_rng(seed)
    n_rows, n = 37, 500
    rows = rng.integers(0, n_rows, n)
    rows[:5] = 3                                              # duplicates of a (row, col) pair are kept
    cols = rng.integers(0, 90, n)
    cols[:5] = 11
    scores = rng.random(n).astype(np.float32)
    off, c, s = dataloader.interaction_csr(rows, cols, scores, n_rows)
    assert off.dtype == np.int64 and c.dtype == np.int64 and s.dtype == np.float32
    assert off[0] == 0 and off[-1] == n and len(off) == n_rows + 1
    for r in range(n_rows):
        idx = [p for p in range(n) if rows[p] == r]
        assert list(c[off[r]:off[r + 1]]) == list(cols[idx])
        assert list(s[off[r]:off[r + 1]]) == list(scores[idx])
    off, c, s = dataloader.interaction_csr([], [], [], 4)
    assert list(off) == [0] * 5 and c.size == 0 and s.size == 0
    with pytest.raises(IndexError):
        dataloader.interaction_csr([4], [0], [1.0], 4)

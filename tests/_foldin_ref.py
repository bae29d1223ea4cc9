"""numpy fp64 restatement of the fold-in (include/invpref_b200.h, invpref_fold_in_users): the explicit ridge solve and
the implicit damped Newton iteration with the library's step rule, stopping rule and Armijo test."""
import numpy as np

ARMIJO = 1e-4
HALVINGS = 30


def sigmoid2(z):
    """(sigmoid(z), 1 - sigmoid(z)) without cancellation."""
    e = np.exp(-np.abs(z))
    inv = 1.0 / (1.0 + e)
    return np.where(z >= 0, inv, e * inv), np.where(z >= 0, e * inv, inv)


def softplus(z):
    return np.maximum(z, 0.0) + np.log1p(np.exp(-np.abs(z)))


def objective(u, V, y, lam):
    z = V @ u
    return float(np.sum(softplus(z) - y * z) + 0.5 * lam * u @ u)


def gradient(u, V, y, lam):
    s, _ = sigmoid2(V @ u)
    return V.T @ (s - y) + lam * u


def hessian(u, V, y, lam):
    s, sm = sigmoid2(V @ u)
    return (V * (s * sm)[:, None]).T @ V + lam * np.eye(V.shape[1])


def loss_diff(z, dz, y):
    """softplus(z + dz) - softplus(z) - y dz, as the library forms it."""
    s, _ = sigmoid2(z)
    with np.errstate(over="ignore"):
        q = s * np.expm1(dz)
    with np.errstate(invalid="ignore", divide="ignore"):
        d = np.where(q > -0.5, np.log1p(np.maximum(q, -0.5)), softplus(z + dz) - softplus(z))
    return d - y * dz


def explicit(V, y, lam):
    """argmin 1/2 |V u - y|^2 + lam/2 |u|^2 (fp64)."""
    V, y = np.asarray(V, np.float64), np.asarray(y, np.float64)
    D = V.shape[1]
    return np.linalg.solve(V.T @ V + lam * np.eye(D), V.T @ y)


def newton(V, y, lam, max_iter=25, steps=None):
    """The library's damped Newton iteration in fp64 -> (u, iters).  ``steps``: a list that receives the step
    length t of every damped step."""
    V, y = np.asarray(V, np.float64), np.asarray(y, np.float64)
    D = V.shape[1]
    u = np.zeros(D)
    if V.shape[0] == 0:
        return u, 0
    for it in range(1, max_iter + 1):
        g = gradient(u, V, y, lam)
        dl = np.linalg.solve(hessian(u, V, y, lam), -g)
        gd, ud, dd = g @ dl, u @ dl, dl @ dl
        if np.abs(dl).max() <= 2.0 ** -30 * max(1.0, np.abs(u).max()):
            return u + dl, it
        z, dz = V @ u, V @ dl
        for m in range(HALVINGS + 1):
            t = 2.0 ** -m
            if np.sum(loss_diff(z, t * dz, y)) + lam * (t * ud + 0.5 * t * t * dd) <= ARMIJO * t * gd:
                break
        if steps is not None:
            steps.append(t)
        u = u + t * dl
    return u, -max_iter


def condition(V, y, lam, u=None, implicit=False):
    """2-norm condition number of the system matrix at u (the optimum)."""
    V = np.asarray(V, np.float64)
    H = hessian(u, V, y, lam) if implicit else V.T @ V + lam * np.eye(V.shape[1])
    return float(np.linalg.cond(H))


def damped_problem(seed=1134):
    """A small implicit history on which the iteration backtracks (some step t < 1): found by a search over random
    problems; Newton from u = 0 on logistic losses rarely overshoots."""
    rng = np.random.default_rng(seed)
    D, n, lam = int(rng.integers(1, 6)), int(rng.integers(1, 12)), 10.0 ** rng.uniform(-4, 0)
    V = (rng.normal(0, 1, (n, D)) * 10.0 ** rng.uniform(0, 1.5)).astype(np.float32)
    y = (rng.random(n) if seed % 2 else (rng.random(n) < 0.5) * 1.0).astype(np.float32)
    return V, y, lam

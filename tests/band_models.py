"""A synthetic trajectory model whose KKT half bandwidth is chosen by its sizes and a coupling knob, so the suite can reach
every template bound of the banded factor kernels (csrc/dto_kkt.cu, `dto_kkt_bw_bound`) and the first bandwidth past each.

`build_band(api, n, m, T, coupling=k)` takes the `api` namespace like the builders of examples/models.py, so the same
definition gives the CPU oracle's model (`oracle.api`) and the product's (`dto_b200`). Explicit dynamics

    x_{t+1} = x_t + h (A (x_t o x_t) + 0.2 sin(x_{t,i+1}) x_{t,i} + Bm u_t)

with A banded: A_ij != 0 for |i - j| <= k (k >= n - 1: dense), and control i (mod m) driving state i. The sin(x_{i+1}) x_i
term and the cost's x_0 u_0 term put cross entries into H, and the cost's double well sum(x^4/4 - x^2/2) makes H indefinite
near x = 0. The start and end states are fixed by constraints as in the pendulum builder (`ends=False`: free, which
narrows the band to about 2n). `u_bnd` adds |u| <= u_bnd bounds (the native solver's interior-point mode).

BAND_CASES lists the half bandwidths `kkt.analyze` gives these models, in the exact-Hessian mode and in the knot-block mode
(None: refused, bandwidth > 31). They do not depend on T.
"""
from __future__ import annotations

import numpy as np

from examples.models import arr, dot, sin


def state_matrix(n, coupling):
    A = np.zeros((n, n))
    for i in range(n):
        for j in range(n):
            if abs(i - j) <= coupling:
                A[i, j] = (0.3 if i == j else 0.15 / abs(i - j)) * (-1.0) ** (i + j)
    return A


def build_band(api, n, m, T, *, coupling, evaluate_hessian=True, u_bnd=None, ends=True):
    h = 0.1
    A = state_matrix(n, coupling)

    def f(x, u):
        out = []
        for i in range(n):
            v = 0.0
            for j in range(n):
                if A[i, j] != 0.0:
                    v = v + float(A[i, j]) * x[j] * x[j]
            v = v + 0.2 * sin(x[(i + 1) % n]) * x[i] + u[i % m]
            out.append(v)
        return arr(*out)

    def dyn(y, x, u, w):
        return y - (x + h * f(x, u))

    x1 = np.array([0.1 * (i + 1) for i in range(n)])
    xT = np.array([0.5 * (-1.0) ** i for i in range(n)])
    # a double well in every state: H is indefinite near x = 0, so the solver's inertia correction has work to do
    ot = lambda x, u, w: sum(0.25 * xi * xi * xi * xi - 0.5 * xi * xi for xi in x) + 0.5 * dot(u, u) + 0.1 * x[0] * u[0]  # noqa: E731
    oT = lambda x, u, w: dot(x, x)                                                  # noqa: E731
    c1 = lambda x, u, w: x - x1                                                     # noqa: E731
    cT = lambda x, u, w: x - xT                                                     # noqa: E731
    dt = api.Dynamics(dyn, n, n, m, num_parameter=0, evaluate_hessian=evaluate_hessian)
    ct = api.Cost(ot, n, m, num_parameter=0, evaluate_hessian=evaluate_hessian)
    cTc = api.Cost(oT, n, 0, num_parameter=0, evaluate_hessian=evaluate_hessian)
    con1 = api.Constraint(c1, n, m, evaluate_hessian=evaluate_hessian)
    conT = api.Constraint(cT, n, 0, evaluate_hessian=evaluate_hessian)
    bnd = api.Bound(n, m) if u_bnd is None else api.Bound(n, m, action_lower=[-u_bnd] * m, action_upper=[u_bnd] * m)
    if ends:
        constraints = [con1] + [api.Constraint() for _ in range(2, T)] + [conT]
    else:
        constraints = [api.Constraint() for _ in range(T)]
    return dict(
        name=f"band_n{n}_m{m}_k{coupling}" + ("" if ends else "_free"), T=T, n=n, m=m,
        dynamics=[dt] * (T - 1),
        objective=[ct] * (T - 1) + [cTc],
        constraints=constraints,
        bounds=[bnd] * (T - 1) + [api.Bound(n, 0)],
        general=None, evaluate_hessian=evaluate_hessian, x1=x1, xT=xT,
    )


T_BAND = 5

# (n, m, coupling, ends) -> (half bandwidth with the exact Hessian, half bandwidth with knot blocks)
BAND_CASES = {
    (3, 1, 2, False): (6, 6),
    (3, 1, 0, True): (7, 7),
    (4, 2, 1, False): (8, 9),
    (3, 2, 0, True): (9, 7),
    (4, 1, 1, True): (10, 10),
    (6, 1, 5, False): (12, 12),
    (6, 2, 5, False): (12, 13),
    (5, 1, 1, True): (13, 14),
    (5, 3, 1, True): (15, 15),
    (8, 1, 7, False): (16, 16),
    (7, 1, 6, True): (20, 20),
    (7, 2, 6, True): (21, 20),
    (10, 2, 9, False): (20, 21),
    (15, 2, 14, False): (30, 31),
    (11, 2, 4, True): (31, None),
    (11, 1, 10, True): (32, None),
}

# knot blocks of 17 variables (k_qn_update with 32 lanes) in a knot-block KKT matrix of half bandwidth 31
QN_BAND = (15, 2, 14, False)


def band_kwargs(key, T=T_BAND):
    n, m, coupling, ends = key
    return dict(n=n, m=m, T=T, coupling=coupling, ends=ends)


def case_id(key):
    n, m, coupling, ends = key
    return f"n{n}m{m}k{coupling}" + ("" if ends else "free")

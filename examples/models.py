"""Model zoo: the reference's example/test problem definitions, written once as plain
python functions that work both on symbols (tracing) and floats (roll-outs).

Each `build_*` takes an `api` namespace exposing the reference's element
constructors (Dynamics, Cost, Constraint, GeneralConstraint, Bound) -- either the
CPU oracle (`oracle.api`) or the B200 product package -- so parity tests feed the
very same problem definition to both sides.

Sources (relative to /root/reference):
  pendulum  examples/pendulum/pendulum.jl:22-77
  cartpole  examples/cartpole/cartpole.jl:19-95
  acrobot   examples/acrobot/acrobot.jl:19-118
  car       examples/car/car.jl:19-60
  test models: test/dynamics.jl:8-19, test/objective.jl:6-9, test/constraints.jl:13-17,
               test/hessian_lagrangian.jl:12-123, test/solve.jl:149-172,239-274
"""
from __future__ import annotations

import math

import numpy as np
import sympy as sp


def _sym(x) -> bool:
    return isinstance(x, sp.Basic)


def sin(x):
    return sp.sin(x) if _sym(x) else math.sin(x)


def cos(x):
    return sp.cos(x) if _sym(x) else math.cos(x)


def tan(x):
    return sp.tan(x) if _sym(x) else math.tan(x)


def dot(a, b):
    s = 0.0
    for p, q in zip(a, b):
        s = s + p * q
    return s


def ifelse(cond, a, b):
    """IfElse.ifelse (imported by the reference, src/DirectTrajectoryOptimization.jl:5): symbolic when the
    condition is, plain python otherwise."""
    if _sym(cond):
        return sp.Piecewise((a, cond), (b, True))
    return a if cond else b


def arr(*v):
    return np.array(v, dtype=object)


def cat(*vs):
    out = []
    for v in vs:
        out.extend(list(v))
    return np.array(out, dtype=object)


# ----------------------------------------------------------------------------
# pendulum (examples/pendulum/pendulum.jl)
# ----------------------------------------------------------------------------
def pendulum(x, u, w):
    mass, length_com, gravity, damping = 1.0, 0.5, 9.81, 0.1
    return arr(
        x[1],
        (u[0] / ((mass * length_com * length_com))
         - gravity * sin(x[0]) / length_com
         - damping * x[1] / (mass * length_com * length_com)),
    )


def pendulum_midpoint(y, x, u, w):
    h = 0.05
    return y - (x + h * pendulum(0.5 * (x + y), u, w))


def build_pendulum(api, T=11, evaluate_hessian=True, u_bnd=None):
    """`u_bnd` (not in the example): |u| <= u_bnd as Bound(action_lower, action_upper) -- the unconstrained swing-up peaks at
    |u| = 18.6, so e.g. 15 makes the bounds active. Bounds live on the host: the model library is the same."""
    n, m = 2, 1
    dt = api.Dynamics(pendulum_midpoint, n, n, m, num_parameter=0, evaluate_hessian=evaluate_hessian)
    x1 = np.array([0.0, 0.0])
    xT = np.array([math.pi, 0.0])
    ot = lambda x, u, w: 0.1 * dot(x[0:2], x[0:2]) + 0.1 * dot(u, u)
    oT = lambda x, u, w: 0.1 * dot(x[0:2], x[0:2])
    ct = api.Cost(ot, n, m, num_parameter=0, evaluate_hessian=evaluate_hessian)
    cT = api.Cost(oT, n, 0, num_parameter=0, evaluate_hessian=evaluate_hessian)
    c1 = lambda x, u, w: x - x1
    cT_ = lambda x, u, w: x - xT
    con1 = api.Constraint(c1, n, m, evaluate_hessian=evaluate_hessian)
    conT = api.Constraint(cT_, n, m, evaluate_hessian=evaluate_hessian)
    return dict(
        fns=dict(dyn=pendulum_midpoint, cost=[ot] * (T - 1) + [oT], con=[c1] + [None] * (T - 2) + [cT_], general=None),
        name="pendulum", T=T, n=n, m=m,
        dynamics=[dt] * (T - 1),
        objective=[ct] * (T - 1) + [cT],
        constraints=[con1] + [api.Constraint() for _ in range(2, T)] + [conT],
        bounds=[api.Bound(n, m) if u_bnd is None else api.Bound(n, m, action_lower=[-u_bnd], action_upper=[u_bnd])] * (T - 1) + [api.Bound(n, 0)],
        general=None, evaluate_hessian=evaluate_hessian, x1=x1, xT=xT,
    )


# ----------------------------------------------------------------------------
# cartpole (examples/cartpole/cartpole.jl)
# ----------------------------------------------------------------------------
def cartpole(x, u, w):
    mc, mp, l, g = 1.0, 0.2, 0.5, 9.81
    q = x[0:2]
    qd = x[2:4]
    s = sin(q[1])
    c = cos(q[1])
    H = np.array([[mc + mp, mp * l * c], [mp * l * c, mp * l ** 2]], dtype=object)
    Hinv = 1.0 / (H[0, 0] * H[1, 1] - H[0, 1] * H[1, 0]) * np.array(
        [[H[1, 1], -H[0, 1]], [-H[1, 0], H[0, 0]]], dtype=object)
    C = np.array([[0, -mp * qd[1] * l * s], [0, 0]], dtype=object)
    G = arr(0, mp * g * l * s)
    B = arr(1, 0)
    qdd = -Hinv @ (C @ qd + G - B * u[0])
    return cat(qd, qdd)


def cartpole_rk3_explicit(x, u, w):
    h = 0.05
    k1 = h * cartpole(x, u, w)
    k2 = h * cartpole(x + 0.5 * k1, u, w)
    k3 = h * cartpole(x - k1 + 2.0 * k2, u, w)
    return x + (k1 + 4.0 * k2 + k3) / 6.0


def cartpole_rk3_implicit(y, x, u, w):
    return y - cartpole_rk3_explicit(x, u, w)


def build_cartpole(api, T=101, evaluate_hessian=True, parameterized=True, u_bnd=3.0):
    """`parameterized=True` is BASELINE config 2: start/goal enter through an 8-vector of
    per-problem parameters w = [x1; xT] seen by every knot (SURVEY Q10); False is the
    example verbatim (constants captured in the closures). `u_bnd`: |u| <= u_bnd as the example's
    Bound(action_lower, action_upper); None leaves the controls free (equality constraints only). Bounds
    live on the host: the model library is the same."""
    n, m = 4, 1
    nw = 8 if parameterized else 0
    x1 = np.array([0.0, 0.0, 0.0, 0.0])
    xT = np.array([0.0, math.pi, 0.0, 0.0])
    Q, R, Qf = 1.0e-2, 1.0e-1, 1.0e2
    dt = api.Dynamics(cartpole_rk3_implicit, n, n, m, num_parameter=nw, evaluate_hessian=evaluate_hessian)
    if parameterized:
        ot = lambda x, u, w: 0.5 * Q * dot(x - w[4:8], x - w[4:8]) + 0.5 * R * dot(u, u)
        oT = lambda x, u, w: 0.5 * Qf * dot(x - w[4:8], x - w[4:8])
        c1 = lambda x, u, w: x - w[0:4]
        cT = lambda x, u, w: x - w[4:8]
    else:
        ot = lambda x, u, w: 0.5 * Q * dot(x - xT, x - xT) + 0.5 * R * dot(u, u)
        oT = lambda x, u, w: 0.5 * Qf * dot(x - xT, x - xT)
        c1 = lambda x, u, w: x - x1
        cT = lambda x, u, w: x - xT
    ct = api.Cost(ot, n, m, num_parameter=nw, evaluate_hessian=evaluate_hessian)
    cTc = api.Cost(oT, n, 0, num_parameter=nw, evaluate_hessian=evaluate_hessian)
    bndt = api.Bound(n, m) if u_bnd is None else api.Bound(n, m, action_lower=[-u_bnd], action_upper=[u_bnd])
    con1 = api.Constraint(c1, n, m, num_parameter=nw, evaluate_hessian=evaluate_hessian)
    conT = api.Constraint(cT, n, 0, num_parameter=nw, evaluate_hessian=evaluate_hessian)
    return dict(
        fns=dict(dyn=cartpole_rk3_implicit, cost=[ot] * (T - 1) + [oT], con=[c1] + [None] * (T - 2) + [cT], general=None),
        name="cartpole", T=T, n=n, m=m,
        dynamics=[dt] * (T - 1),
        objective=[ct] * (T - 1) + [cTc],
        constraints=[con1] + [api.Constraint() for _ in range(2, T)] + [conT],
        bounds=[bndt] * (T - 1) + [api.Bound(n, 0)],
        general=None, evaluate_hessian=evaluate_hessian, x1=x1, xT=xT,
        num_parameter=nw, shared_parameters=parameterized,
    )


# ----------------------------------------------------------------------------
# acrobot (examples/acrobot/acrobot.jl, test/hessian_lagrangian.jl)
# ----------------------------------------------------------------------------
def acrobot(x, u, w):
    mass1, inertia1, length1, lengthcom1 = 1.0, 0.33, 1.0, 0.5
    mass2, inertia2, length2, lengthcom2 = 1.0, 0.33, 1.0, 0.5
    gravity, friction1, friction2 = 9.81, 0.1, 0.1

    def Minv(x, w):
        a = (inertia1 + inertia2 + mass2 * length1 * length1
             + 2.0 * mass2 * length1 * lengthcom2 * cos(x[1]))
        b = inertia2 + mass2 * length1 * lengthcom2 * cos(x[1])
        c = inertia2
        return 1.0 / (a * c - b * b) * np.array([[c, -b], [-b, a]], dtype=object)

    def tau(x, w):
        a = (-1.0 * mass1 * gravity * lengthcom1 * sin(x[0])
             - mass2 * gravity * (length1 * sin(x[0])
                                  + lengthcom2 * sin(x[0] + x[1])))
        b = -1.0 * mass2 * gravity * lengthcom2 * sin(x[0] + x[1])
        return arr(a, b)

    def C(x, w):
        a = -2.0 * mass2 * length1 * lengthcom2 * sin(x[1]) * x[3]
        b = -1.0 * mass2 * length1 * lengthcom2 * sin(x[1]) * x[3]
        c = mass2 * length1 * lengthcom2 * sin(x[1]) * x[2]
        d = 0.0
        return np.array([[a, b], [c, d]], dtype=object)

    def B(x, w):
        return arr(0.0, 1.0)

    q = x[0:2]
    v = x[2:4]
    qdd = Minv(q, w) @ (-1.0 * (C(x, w) @ v) + tau(q, w) + B(q, w) * u[0] - arr(friction1, friction2) * v)
    return arr(x[2], x[3], qdd[0], qdd[1])


def acrobot_midpoint(y, x, u, w):
    h = 0.05
    return y - (x + h * acrobot(0.5 * (x + y), u, w))


def build_acrobot(api, T=101, evaluate_hessian=True, stage_endpoint_constraints=True):
    """examples/acrobot/acrobot.jl with every Hessian enabled (BASELINE config 3)."""
    n, m = 4, 1
    dt = api.Dynamics(acrobot_midpoint, n, n, m, num_parameter=0, evaluate_hessian=evaluate_hessian)
    x1 = np.array([0.0, 0.0, 0.0, 0.0])
    xT = np.array([math.pi, 0.0, 0.0, 0.0])
    ot = lambda x, u, w: 0.1 * dot(x[2:4], x[2:4]) + 0.1 * dot(u, u)
    oT = lambda x, u, w: 0.1 * dot(x[2:4], x[2:4])
    ct = api.Cost(ot, n, m, num_parameter=0, evaluate_hessian=evaluate_hessian)
    cT = api.Cost(oT, n, 0, num_parameter=0, evaluate_hessian=evaluate_hessian)
    c1 = lambda x, u, w: x - x1
    cT_ = lambda x, u, w: x - xT
    con_fns = [None] * T
    if stage_endpoint_constraints:
        con_fns = [c1] + [None] * (T - 2) + [cT_]
        cons = ([api.Constraint(c1, n, m, evaluate_hessian=evaluate_hessian)]
                + [api.Constraint() for _ in range(2, T)]
                + [api.Constraint(cT_, n, 0, evaluate_hessian=evaluate_hessian)])
        bounds = [api.Bound(n, m)] * (T - 1) + [api.Bound(n, 0)]
    else:  # test/solve.jl: end points pinned through bounds
        cons = [api.Constraint() for _ in range(T)]
        bounds = ([api.Bound(n, m, state_lower=x1, state_upper=x1)] + [api.Bound(n, m)] * (T - 2)
                  + [api.Bound(n, 0, state_lower=xT, state_upper=xT)])
    return dict(
        fns=dict(dyn=acrobot_midpoint, cost=[ot] * (T - 1) + [oT], con=con_fns, general=None),
        name="acrobot", T=T, n=n, m=m,
        dynamics=[dt] * (T - 1), objective=[ct] * (T - 1) + [cT], constraints=cons, bounds=bounds,
        general=None, evaluate_hessian=evaluate_hessian, x1=x1, xT=xT,
    )


def build_acrobot_hessian_test(api):
    """test/hessian_lagrangian.jl:97-128 -- T=3, nonlinear stage constraints, all Hessians."""
    T, n, m = 3, 4, 1
    dt = api.Dynamics(acrobot_midpoint, n, n, m, num_parameter=0, evaluate_hessian=True)
    x1 = np.array([0.0, 0.0, 0.0, 0.0])
    xT = np.array([0.0, math.pi, 0.0, 0.0])
    ot = lambda x, u, w: 0.1 * dot(x[2:4], x[2:4]) + 0.1 * dot(u, u)
    oT = lambda x, u, w: 0.1 * dot(x[2:4], x[2:4])
    objt = api.Cost(ot, n, m, num_parameter=0, evaluate_hessian=True)
    objT = api.Cost(oT, n, 0, num_parameter=0, evaluate_hessian=True)

    def ct(x, u, w):
        sx2 = 0.0
        for xi in x:
            sx2 = sx2 + xi ** 2
        return cat([-5.0 - cos(ui) * sx2 for ui in u], [cos(xi) * tan(u[0]) - 5.0 for xi in x])

    def cT(x, u, w):
        return arr(*[sin(xi ** 3.0) for xi in x])

    cont = api.Constraint(ct, n, m, num_parameter=0, indices_inequality=list(range(1, m + n + 1)),
                          evaluate_hessian=True)
    conT = api.Constraint(cT, n, 0, num_parameter=0, evaluate_hessian=True)
    bounds = ([api.Bound(n, m, state_lower=x1, state_upper=x1)] + [api.Bound(n, m)] * (T - 2)
              + [api.Bound(n, 0, state_lower=xT, state_upper=xT)])
    return dict(
        name="acrobot_hessian_test", T=T, n=n, m=m,
        dynamics=[dt] * (T - 1), objective=[objt] * (T - 1) + [objT],
        constraints=[cont] * (T - 1) + [conT], bounds=bounds, general=None, evaluate_hessian=True,
        ot=ot, oT=oT, ct=ct, cT=cT,
    )


# ----------------------------------------------------------------------------
# car (examples/car/car.jl)
# ----------------------------------------------------------------------------
def car(x, u, w):
    return arr(u[0] * cos(x[2]), u[0] * sin(x[2]), u[1])


def car_midpoint(y, x, u, w):
    h = 0.1
    return y - (x + h * car(0.5 * (x + y), u, w))


P_OBS = (0.5, 0.5)
R_OBS = 0.1


def car_obs(x, u, w):
    e = x[0:2] - np.array(P_OBS)
    return arr(R_OBS ** 2.0 - dot(e, e))


def build_car(api, T=51, evaluate_hessian=True, obstacle="general"):
    """obstacle='stage' is the example verbatim (one inequality per knot);
    obstacle='general' is BASELINE config 4: the same T inequalities expressed as ONE
    GeneralConstraint over the whole z (exercises the general path + Hessian scatter)."""
    n, m = 3, 2
    dt = api.Dynamics(car_midpoint, n, n, m, num_parameter=0, evaluate_hessian=evaluate_hessian)
    x1 = np.array([0.0, 0.0, 0.0])
    xT = np.array([1.0, 1.0, 0.0])
    ot = lambda x, u, w: 0.0 * dot(x - xT, x - xT) + 1.0 * dot(u, u)
    oT = lambda x, u, w: 0.0 * dot(x - xT, x - xT)
    ct = api.Cost(ot, n, m, num_parameter=0, evaluate_hessian=evaluate_hessian)
    cT = api.Cost(oT, n, 0, num_parameter=0, evaluate_hessian=evaluate_hessian)
    al, au = -0.5 * np.ones(m), 0.5 * np.ones(m)
    bounds = ([api.Bound(n, m, state_lower=x1, state_upper=x1, action_lower=al, action_upper=au)]
              + [api.Bound(n, m, action_lower=al, action_upper=au)] * (T - 2)
              + [api.Bound(n, 0, state_lower=xT, state_upper=xT)])
    general = None
    gen_fn, con_fns = None, [None] * T
    if obstacle == "stage":
        con_fns = [car_obs] * T
        cont = api.Constraint(car_obs, n, m, num_parameter=0, indices_inequality=[1],
                              evaluate_hessian=evaluate_hessian)
        conT = api.Constraint(car_obs, n, 0, num_parameter=0, indices_inequality=[1],
                              evaluate_hessian=evaluate_hessian)
        cons = [cont] * (T - 1) + [conT]
    else:
        cons = [api.Constraint() for _ in range(T)]
        nz = T * n + (T - 1) * m

        def g(z, w):
            rows = []
            for t in range(T):
                o = t * (n + m)
                rows.append(car_obs(z[o:o + n], None, w)[0])
            return arr(*rows)

        gen_fn = g
        general = api.GeneralConstraint(g, nz, 0, indices_inequality=list(range(1, T + 1)),
                                        evaluate_hessian=evaluate_hessian)
    return dict(
        fns=dict(dyn=car_midpoint, cost=[ot] * (T - 1) + [oT], con=con_fns, general=gen_fn),
        name="car", T=T, n=n, m=m,
        dynamics=[dt] * (T - 1), objective=[ct] * (T - 1) + [cT], constraints=cons, bounds=bounds,
        general=general, evaluate_hessian=evaluate_hessian, x1=x1, xT=xT,
    )


# ----------------------------------------------------------------------------
# small test models
# ----------------------------------------------------------------------------
def test_pendulum(z, u, w):
    """test/dynamics.jl:8-14"""
    mass, lc, gravity, damping = 1.0, 1.0, 9.81, 0.1
    return arr(z[1], (u[0] / ((mass * lc * lc)) - gravity * sin(z[0]) / lc - damping * z[1] / (mass * lc * lc)))


def test_euler_implicit(y, x, u, w):
    """test/dynamics.jl:16-19"""
    h = 0.1
    return y - (x + h * test_pendulum(y, u, w))


def build_linear_general(api, T=11, reference_exact=False):
    """test/solve.jl:227-296 flavour: double integrator, linear GeneralConstraint pinning
    the end points over the whole z; every Hessian enabled (general/dynamics ones are empty).
    reference_exact=True is the test verbatim: A = [1 1; 0 1], B = [0; 1], x1 pinned by a Bound, only xT by the
    GeneralConstraint."""
    n, m = 2, 1
    h = 0.1

    if reference_exact:
        h = 1.0

    def dyn(y, x, u, w):
        A = np.array([[1.0, h], [0.0, 1.0]], dtype=object)
        Bm = arr(0.0, h)
        return y - (A @ x + Bm * u[0])

    dt = api.Dynamics(dyn, n, n, m, evaluate_hessian=True)
    ot = lambda x, u, w: 0.1 * dot(x, x) + 0.1 * dot(u, u)
    oT = lambda x, u, w: 0.1 * dot(x, x)
    ct = api.Cost(ot, n, m, evaluate_hessian=True)
    cT = api.Cost(oT, n, 0, evaluate_hessian=True)
    x1 = np.array([0.0, 0.0])
    xT = np.array([1.0, 0.0])
    nz = T * n + (T - 1) * m
    if reference_exact:
        gc = api.GeneralConstraint(lambda z, w: z[nz - n:nz] - xT, nz, 0, evaluate_hessian=True)
        bounds = [api.Bound(n, m, state_lower=x1, state_upper=x1)] + [api.Bound(n, m)] * (T - 2) + [api.Bound(n, 0)]
    else:
        gc = api.GeneralConstraint(lambda z, w: cat(z[0:n] - x1, z[nz - n:nz] - xT), nz, 0, evaluate_hessian=True)
        bounds = [api.Bound(n, m)] * (T - 1) + [api.Bound(n, 0)]
    return dict(
        name="linear_general", T=T, n=n, m=m,
        dynamics=[dt] * (T - 1), objective=[ct] * (T - 1) + [cT],
        constraints=[api.Constraint() for _ in range(T)],
        bounds=bounds,
        general=gc, evaluate_hessian=True, x1=x1, xT=xT,
    )


def build_heterogeneous(api, evaluate_hessian=True):
    """Not from the reference's examples: a deliberately irregular problem that exercises what the
    reference's data model allows (SURVEY Q1, Q10, Q11): state/action dims change along the horizon,
    every knot has its own Dynamics/Cost object, per-knot parameter vectors of different lengths in the
    reference's vcat layout, nonlinear stage constraints with inequalities on some knots only, and a
    nonlinear GeneralConstraint coupling distant knots."""
    nx = [2, 2, 3, 3, 2, 2]
    nu = [1, 2, 1, 1, 1, 0]
    nw = [0, 1, 2, 0, 1, 1]
    T = len(nx)

    def make_dyn(t):
        n0, m0, n1 = nx[t], nu[t], nx[t + 1]

        def f(y, x, u, w):
            out = []
            for i in range(n1):
                xi = x[i % n0]
                uj = u[i % m0]
                p = w[0] if nw[t] > 0 else 0.3
                out.append(y[i] - (xi + 0.1 * (sin(xi * uj) + p * cos(y[i]) * x[(i + 1) % n0] ** 2 - 0.5 * uj)))
            return arr(*out)

        return api.Dynamics(f, n1, n0, m0, num_parameter=nw[t], evaluate_hessian=evaluate_hessian)

    def make_cost(t):
        def c(x, u, w):
            v = 0.0
            for i in range(nx[t]):
                v = v + (0.5 + 0.1 * i) * x[i] ** 2 + 0.01 * x[i] ** 4
            for j in range(nu[t]):
                v = v + 0.2 * u[j] ** 2 + 0.05 * u[j] * x[0]
            if nw[t] > 0:
                v = v + w[nw[t] - 1] * x[0]
            return v

        return api.Cost(c, nx[t], nu[t], num_parameter=nw[t], evaluate_hessian=evaluate_hessian)

    def make_con(t):
        if t in (1, 4):
            return api.Constraint()
        if t == 2:
            return api.Constraint(lambda x, u, w: arr(x[0] * x[1] - w[1], sin(u[0]) + x[2] ** 2 - 1.0), nx[t], nu[t],
                                  num_parameter=nw[t], indices_inequality=[2], evaluate_hessian=evaluate_hessian)
        if t == T - 1:
            return api.Constraint(lambda x, u, w: arr(x[0] ** 2 + x[1] ** 2 - 1.0), nx[t], 0, num_parameter=nw[t],
                                  evaluate_hessian=evaluate_hessian)
        return api.Constraint(lambda x, u, w: arr(x[0] - 0.1 * u[0], x[1] * u[0]), nx[t], nu[t], num_parameter=nw[t],
                              indices_inequality=[1, 2], evaluate_hessian=evaluate_hessian)

    nz = sum(nx) + sum(nu)
    npar = sum(nw)

    def g(z, w):
        return arr(z[0] * z[nz - 1] - 0.5, sin(z[3]) * z[7] + w[npar - 1] * z[1] ** 2, z[2] + z[5])

    general = api.GeneralConstraint(g, nz, npar, indices_inequality=[2], evaluate_hessian=evaluate_hessian)
    return dict(
        name="heterogeneous", T=T, n=None, m=None, nx=nx, nu=nu, nw=nw,
        dynamics=[make_dyn(t) for t in range(T - 1)], objective=[make_cost(t) for t in range(T)],
        constraints=[make_con(t) for t in range(T)],
        bounds=[api.Bound(nx[t], nu[t]) for t in range(T)], general=general, evaluate_hessian=evaluate_hessian,
    )


def build_user_jacobian(api, T=11, nonlinear=False):
    """test/solve.jl:140-225: double integrator whose dynamics Jacobian is SUPPLIED by the user
    (second Dynamics constructor, src/dynamics.jl:59-101): dense column-major pattern, no Hessian, state
    end points pinned by bounds. `nonlinear=True` (not in the reference) makes f and the user Jacobian
    state dependent and the Jacobian deliberately NOT the exact derivative (entry (2,1) is scaled by 3),
    so a parity test can tell "lowered the user's expressions" from "differentiated f"."""
    n, m = 2, 1

    def f(y, x, u, w):
        A = np.array([[1.0, 1.0], [0.0, 1.0]], dtype=object)
        Bm = arr(0.0, 1.0)
        r = y - (A @ x + Bm * u[0])
        if nonlinear:
            r = r - arr(0.0, 0.1 * sin(x[0]) * u[0])
        return r

    def fz(J, y, x, u, w):
        J[:, :] = 0.0
        J[0, 0], J[0, 1] = -1.0, -1.0
        J[1, 1] = -1.0
        J[1, 2] = -1.0
        J[0, 3], J[1, 4] = 1.0, 1.0
        if nonlinear:
            J[1, 0] = -3.0 * 0.1 * cos(x[0]) * u[0]
            J[1, 2] = -1.0 - 0.1 * sin(x[0])

    dt = api.Dynamics(f, fz, n, n, m)
    ot = lambda x, u, w: 0.1 * dot(x, x) + 0.1 * dot(u, u)
    oT = lambda x, u, w: 0.1 * dot(x, x)
    ct = api.Cost(ot, n, m, num_parameter=0)
    cT = api.Cost(oT, n, 0, num_parameter=0)
    x1 = np.array([0.0, 0.0])
    xT = np.array([1.0, 0.0])
    return dict(
        name="user_jacobian", T=T, n=n, m=m,
        dynamics=[dt] * (T - 1), objective=[ct] * (T - 1) + [cT],
        constraints=[api.Constraint() for _ in range(T)],
        bounds=[api.Bound(n, m, state_lower=x1, state_upper=x1)] + [api.Bound(n, m)] * (T - 2)
        + [api.Bound(n, 0, state_lower=xT, state_upper=xT)],
        general=None, evaluate_hessian=False, x1=x1, xT=xT,
    )


def build_piecewise(api, T=9, evaluate_hessian=True):
    """Not from the reference's examples: exercises `ifelse` in every element role (the reference imports
    IfElse, src/DirectTrajectoryOptimization.jl:5, but no model of it uses it) -- a pendulum whose torque
    saturates smoothly on one side and whose damping switches with the sign of the velocity, a cost with a
    one-sided penalty, and a stage constraint with a switched branch."""
    n, m = 2, 1
    h = 0.05

    def f(x, u, w):
        torque = ifelse(u[0] > 0.5, 0.5 + 0.25 * sin(2.0 * (u[0] - 0.5)), u[0])
        damp = ifelse(x[1] >= 0.0, 0.1 * x[1] + 0.05 * x[1] ** 2, 0.1 * x[1] - 0.05 * x[1] ** 2)
        return arr(x[1], 4.0 * torque - 19.62 * sin(x[0]) - 4.0 * damp)

    def dyn(y, x, u, w):
        return y - (x + h * f(0.5 * (x + y), u, w))

    dt = api.Dynamics(dyn, n, n, m, evaluate_hessian=evaluate_hessian)
    ot = lambda x, u, w: 0.1 * dot(x, x) + 0.1 * dot(u, u) + ifelse(x[0] > 1.0, 2.0 * (x[0] - 1.0) ** 3, 0.0 * x[0])
    oT = lambda x, u, w: 0.1 * dot(x, x)
    ct = api.Cost(ot, n, m, evaluate_hessian=evaluate_hessian)
    cT = api.Cost(oT, n, 0, evaluate_hessian=evaluate_hessian)
    x1 = np.array([0.0, 0.0])
    xT = np.array([math.pi, 0.0])
    con1 = api.Constraint(lambda x, u, w: x - x1, n, m, evaluate_hessian=evaluate_hessian)
    cont = api.Constraint(lambda x, u, w: arr(ifelse(x[1] < 0.0, x[1] ** 2 - 9.0, x[1] * u[0] - 9.0)), n, m,
                          indices_inequality=[1], evaluate_hessian=evaluate_hessian)
    conT = api.Constraint(lambda x, u, w: x - xT, n, 0, evaluate_hessian=evaluate_hessian)
    return dict(
        name="piecewise", T=T, n=n, m=m,
        dynamics=[dt] * (T - 1), objective=[ct] * (T - 1) + [cT],
        constraints=[con1] + [cont for _ in range(2, T)] + [conT],
        bounds=[api.Bound(n, m)] * (T - 1) + [api.Bound(n, 0)],
        general=None, evaluate_hessian=evaluate_hessian, x1=x1, xT=xT,
    )


BUILDERS = {
    "pendulum": build_pendulum,
    "cartpole": build_cartpole,
    "acrobot": build_acrobot,
    "car": build_car,
    "acrobot_hessian_test": build_acrobot_hessian_test,
    "linear_general": build_linear_general,
    "heterogeneous": build_heterogeneous,
    "user_jacobian": build_user_jacobian,
    "piecewise": build_piecewise,
}

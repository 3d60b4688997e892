"""Bound values per problem in the native solver (dto_sqp_solve_ex, bounds_stride = N_z) and in the torch-glued arm: a batch of
problems that share one bound pattern but not the values -- each its own pinned start state, its own actuator limits. Problems
are independent, so every problem must come out bit for bit as it does in a batch of problems that share its bounds."""
import ctypes as C

import numpy as np
import pytest

import dto_b200 as D
from dto_b200 import _lib, sqp
from examples import models as M

pytestmark = pytest.mark.gpu

STATS = 8          # the counter entries of stats[16] (the rest are host microseconds)


def _raw(nlp, z0, lo, up, stride, options=None, ex=True):
    """dto_sqp_solve (ex=False: the shared [N_z] pair) or dto_sqp_solve_ex through ctypes; returns every output"""
    L = _lib.lib()
    B, N_z, N_c = nlp.batch, nlp.num_variables, nlp.num_constraint
    co = _lib.SqpOptions()
    L.dto_sqp_default_options(C.byref(co))
    for k, v in (options or {}).items():
        setattr(co, k, v)
    out = dict(z=np.empty((B, N_z)), lam=np.empty((B, N_c)), iters=np.empty(B, np.int32), conv=np.empty(B, np.uint8), cv=np.empty(B),
               dr=np.empty(B), f=np.empty(B), stats=np.zeros(16, np.int64))
    z0, lo, up = (np.ascontiguousarray(v, dtype=np.float64) for v in (z0, lo, up))
    p = lambda a: a.ctypes.data  # noqa: E731
    tail = [p(out[k]) for k in ("z", "lam", "iters", "conv", "cv", "dr", "f", "stats")]
    if ex:
        st = L.dto_sqp_solve_ex(nlp.handle, C.byref(co), p(z0), None, p(lo), p(up), stride, *tail)
    else:
        st = L.dto_sqp_solve(nlp.handle, C.byref(co), p(z0), None, p(lo), p(up), *tail)
    return st, out


def _same(a, b, where=""):
    for k in ("z", "lam", "iters", "conv", "cv", "dr", "f"):
        assert np.array_equal(a[k], b[k]), (where, k)
    assert np.array_equal(a["stats"][:STATS], b["stats"][:STATS]), (where, "stats")


def _interp_guess(model, B, seed, scale=1.0, x1=None):
    T, n, m = model["T"], model["n"], model["m"]
    x1 = np.tile(model["x1"], (B, 1)) if x1 is None else x1
    rng = np.random.default_rng(seed)
    z = np.zeros((B, T * n + (T - 1) * m))
    for t in range(T):
        o = t * (n + m)
        z[:, o:o + n] = x1 + (model["xT"] - x1) * t / (T - 1)
        if t < T - 1:
            z[:, o + n:o + n + m] = scale * rng.normal(size=(B, m))
    return z


def _cartpole_guess(model, B, seed):
    T, n, m, x1 = model["T"], model["n"], model["m"], model["x1"]
    rng = np.random.default_rng(seed)
    z = np.zeros((B, T * n + (T - 1) * m))
    for b in range(B):
        u0 = np.array([0.01 * (1.0 + 0.2 * rng.normal())])
        xs = [x1.astype(float)]
        for _ in range(T - 1):
            xs.append(np.array(M.cartpole_rk3_explicit(xs[-1], u0, np.zeros(0)), dtype=float))
        for t in range(T):
            z[b, t * (n + m): t * (n + m) + n] = xs[t]
            if t < T - 1:
                z[b, t * (n + m) + n] = u0[0]
    return z


def _limits(n, m, T, u):
    return [D.Bound(n, m, action_lower=[-u] * m, action_upper=[u] * m)] * (T - 1) + [D.Bound(n, 0)]


def _pinned(n, m, T, x1, xT):
    return [D.Bound(n, m, state_lower=x1, state_upper=x1)] + [D.Bound(n, m)] * (T - 2) + [D.Bound(n, 0, state_lower=xT, state_upper=xT)]


def _car(n, m, T, x1, xT, u):
    al, au = [-u] * m, [u] * m
    return ([D.Bound(n, m, state_lower=x1, state_upper=x1, action_lower=al, action_upper=au)]
            + [D.Bound(n, m, action_lower=al, action_upper=au)] * (T - 2) + [D.Bound(n, 0, state_lower=xT, state_upper=xT)])


@pytest.mark.parametrize("case", ["pendulum_bounds", "cartpole_example", "acrobot_solve_jl"])
def test_identical_rows_give_the_bits_of_the_shared_bounds(case):
    """[B, N_z] rows that are all the same (bounds_stride = N_z) against the shared [N_z] pair of dto_sqp_solve: every output"""
    if case == "pendulum_bounds":
        model, B, o = M.build_pendulum(D, u_bnd=15.0), 4, dict(max_iter=60)
        z0 = _interp_guess(model, B, 5, 0.3)
    elif case == "cartpole_example":
        model, B, o = M.build_cartpole(D, T=101), 8, dict(max_iter=400)
        z0 = _cartpole_guess(model, B, 5)
    else:                        # test/solve.jl:1-138: acrobot T = 101, both end points pinned by bounds
        model, B, o = M.build_acrobot(D, T=101, stage_endpoint_constraints=False), 16, dict(max_iter=300)
        z0 = _interp_guess(model, B, 4)
    nlp = D.solver_from(model, batch=B).nlp
    if model.get("num_parameter"):
        nlp.set_parameters(np.tile(np.concatenate([model["x1"], model["xT"]]), (B, 1)))
    lo, up = nlp.variable_bounds
    st0, shared = _raw(nlp, z0, lo, up, 0, o, ex=False)
    st1, rows = _raw(nlp, z0, np.tile(lo, (B, 1)), np.tile(up, (B, 1)), nlp.num_variables, o)
    assert st0 == st1 == 0
    _same(shared, rows, case)
    assert shared["conv"].sum() >= B // 2 and shared["stats"][1] > 100
    nlp.close()


def _mixed_against_groups(model, groups, assign, z0, options, params=None):
    """groups: Bound lists; assign[b]: problem b's group. Solves the mixed batch (Solver.set_bounds per problem, native arm)
    and every group alone under its shared Bound list; each problem must carry its group solve's bits. Returns the mixed result."""
    B = len(assign)
    s = D.solver_from(model, batch=B)
    if params is not None:
        s.nlp.set_parameters(params)
    for b, g in enumerate(assign):
        s.set_bounds(groups[g], problem=b)
    assert s.nlp.batch_variable_bounds[0].shape == (B, s.nlp.num_variables)
    mixed = sqp.solve_native(s.nlp, z0, options=sqp.SQPOptions(**options))
    s.nlp.close()
    for g, bl in enumerate(groups):
        rows = np.nonzero(np.asarray(assign) == g)[0]
        sg = D.solver_from(dict(model, bounds=bl), batch=len(rows))
        if params is not None:
            sg.nlp.set_parameters(params[rows])
        assert sg.nlp.batch_variable_bounds[0].ndim == 1               # the shared-bounds path (bounds_stride = 0)
        ref = sqp.solve_native(sg.nlp, z0[rows], options=sqp.SQPOptions(**options))
        sg.nlp.close()
        for name in ("z", "lam", "iterations", "converged", "staged", "constraint_violation", "dual_residual", "objective"):
            assert np.array_equal(getattr(mixed, name)[rows], getattr(ref, name)), (g, name)
    return mixed


def test_acrobot_per_problem_start_states_equal_the_grouped_solves():
    model = M.build_acrobot(D, T=101, stage_endpoint_constraints=False)
    n, m, T, xT = model["n"], model["m"], model["T"], model["xT"]
    starts = [model["x1"] + np.array([a, -0.5 * a, 0.0, 0.0]) for a in (0.0, 0.3, -0.2, 0.6)]
    groups = [_pinned(n, m, T, x, xT) for x in starts]
    assign = [b % 4 for b in range(16)]
    z0 = _interp_guess(model, 16, 11, x1=np.stack([starts[g] for g in assign]))
    mixed = _mixed_against_groups(model, groups, assign, z0, dict(max_iter=300))
    assert mixed.converged.sum() >= 8
    for b, g in enumerate(assign):
        assert np.array_equal(mixed.z[b, :n], starts[g]) and np.array_equal(mixed.z[b, -n:], xT)


def _cartpole_mixed():
    model = M.build_cartpole(D, T=101)
    n, m, T = model["n"], model["m"], model["T"]
    limits = (3.0, 4.0, 6.0, 10.0)
    assign = [b % 4 for b in range(16)]
    params = np.tile(np.concatenate([model["x1"], model["xT"]]), (16, 1))
    return model, [_limits(n, m, T, u) for u in limits], limits, assign, params, _cartpole_guess(model, 16, 3)


def test_cartpole_per_problem_control_limits_equal_the_grouped_solves():
    model, groups, limits, assign, params, z0 = _cartpole_mixed()
    mixed = _mixed_against_groups(model, groups, assign, z0, dict(max_iter=600), params=params)
    assert mixed.converged.all()
    n, m, T = model["n"], model["m"], model["T"]
    U = np.stack([mixed.z[:, t * (n + m) + n] for t in range(T - 1)], axis=1)
    lim = np.array([limits[g] for g in assign])
    assert np.all(np.abs(U) < lim[:, None]) and np.any(np.abs(U[lim == 3.0]) > 3.0 - 1e-4)


def test_car_per_problem_control_limits_equal_the_grouped_solves_through_the_continuation():
    """the car example with its obstacle rows: per-group control limits; some problems converge only through the bound
    continuation (converged == 2), whose widening is then about every problem's own midpoints"""
    model = M.build_car(D, T=51, obstacle="stage")
    n, m, T, x1, xT = model["n"], model["m"], model["T"], model["x1"], model["xT"]
    groups = [_car(n, m, T, x1, xT, u) for u in (0.5, 0.4, 0.6, 0.8)]
    assign = [b % 4 for b in range(48)]
    z0 = _interp_guess(model, 48, 2, 0.001)
    mixed = _mixed_against_groups(model, groups, assign, z0, dict(max_iter=300))
    assert mixed.staged.any(), mixed.iterations
    assert mixed.converged.sum() >= 36


def test_sharded_solve_with_per_problem_bounds_equals_the_one_device_solve():
    """two shards (the device listed twice): every shard gets its slice of the rows"""
    import torch
    model, groups, _, assign, params, z0 = _cartpole_mixed()
    dev = [0, 1] if torch.cuda.device_count() > 1 else [0, 0]
    outs = []
    for devices in ([0], dev):
        s = D.solver_from(model, batch=len(assign), devices=devices)
        assert s.nlp.num_shards == len(devices)
        s.nlp.set_parameters(params)
        for b, g in enumerate(assign):
            s.set_bounds(groups[g], problem=b)
        s._initial[:] = z0
        res = s.solve(options=dict(max_iter=600))
        assert s.broker is None
        outs.append(res)
        s.nlp.close()
    for name in ("z", "lam", "iterations", "converged", "constraint_violation", "objective"):
        assert np.array_equal(getattr(outs[0], name), getattr(outs[1], name)), name
    assert outs[1].stats["devices"] == dev


def test_torch_glued_arm_agrees_with_the_native_arm_on_per_problem_limits():
    model, groups, _, assign, params, z0 = _cartpole_mixed()
    s = D.solver_from(model, batch=len(assign))
    s.nlp.set_parameters(params)
    for b, g in enumerate(assign):
        s.set_bounds(groups[g], problem=b)
    s._initial[:] = z0
    nat = s.solve(options=dict(max_iter=600), method="native")
    tor = s.solve(options=dict(max_iter=600), method="sqp")
    cn, ct = nat.converged, tor.converged.cpu().numpy()
    assert np.array_equal(cn, ct) and cn.sum() >= len(assign) - 1
    zn, zt = nat.z[cn], tor.z.cpu().numpy()[cn]
    assert np.max(np.abs(zn - zt) / np.maximum(1.0, np.abs(zt))) < 1e-5
    tor_staged = tor.staged.cpu().numpy() if hasattr(tor, "staged") else np.zeros(len(assign), bool)
    direct = cn & ~nat.staged & ~tor_staged
    assert np.max(np.abs(nat.iterations[direct] - tor.iterations.cpu().numpy()[direct])) <= 3
    s.nlp.close()


def test_refusals_name_the_problem_and_the_variable():
    model = M.build_cartpole(D, T=11)
    B = 3
    nlp = D.solver_from(model, batch=B).nlp
    nlp.set_parameters(np.tile(np.concatenate([model["x1"], model["xT"]]), (B, 1)))
    N_z = nlp.num_variables
    lo, up = (np.tile(v, (B, 1)) for v in nlp.variable_bounds)
    z0 = np.zeros((B, N_z))
    ui = 4                                   # the first control (0-based), |u| <= 3
    cases = []
    l2, u2 = lo.copy(), up.copy()
    l2[2, ui] = -np.inf                      # problem 2 has no lower bound where problem 0 has one
    cases.append((l2, u2, N_z, -7, ("problem 2", f"variable {ui + 1}")))
    l2, u2 = lo.copy(), up.copy()
    l2[1, ui], u2[1, ui] = 2.0, 1.0          # lower > upper
    cases.append((l2, u2, N_z, -1, ("problem 1", f"variable {ui + 1}")))
    l2, u2 = lo.copy(), up.copy()
    u2[2, ui] = np.nan
    cases.append((l2, u2, N_z, -1, ("problem 2", f"variable {ui + 1}")))
    cases.append((lo, up, N_z - 1, -1, ("bounds_stride",)))
    for l2, u2, stride, status, words in cases:
        st, _ = _raw(nlp, z0, l2, u2, stride, dict(max_iter=2))
        assert st == status, (st, words)
        msg = _lib.lib().dto_last_error().decode()
        assert all(w in msg for w in words), msg
    # the Python arms refuse a batch of two patterns before any solve
    s = D.solver_from(model, batch=B)
    s.nlp.set_parameters(np.tile(np.concatenate([model["x1"], model["xT"]]), (B, 1)))
    s.set_bounds(_limits(model["n"], model["m"], model["T"], 2.0), problem=1)
    bad = [D.Bound(model["n"], model["m"])] + _limits(model["n"], model["m"], model["T"], 2.0)[1:]
    s.set_bounds(bad, problem=2)
    with pytest.raises(_lib.DtoError) as e:
        s.solve(options=dict(max_iter=2), method="native")
    assert e.value.status == -7 and "problem 2" in str(e.value)
    with pytest.raises(ValueError, match="problem 2"):
        s.solve(options=dict(max_iter=2), method="sqp")
    s.nlp.close()
    nlp.close()

"""Bound values per problem, host side: Solver.set_bounds lays a problem's Bound list out as primal_bounds does, sqp.bound_arrays
on [B, N_z] rows gives every row what it gives that row alone (continuation scale included) and refuses rows of different
patterns, and the oracle-driven twin of the solver, run on a batch whose problems carry different bounds, gives every problem
exactly what a batch of problems sharing its bounds gives it (tests/test_sqp_bounds_gpu.py holds the device arms to the same)."""
import numpy as np
import pytest

import dto_b200 as D
from dto_b200 import kkt as PK
from dto_b200 import sqp
from examples import models as M
from oracle import api as O

from sqp_oracle import OracleBackend


def _guess(model, B, seed):
    T, n, m = model["T"], model["n"], model["m"]
    rng = np.random.default_rng(seed)
    z = np.zeros((B, T * n + (T - 1) * m))
    for t in range(T):
        o = t * (n + m)
        z[:, o:o + n] = model["x1"] + (model["xT"] - model["x1"]) * t / (T - 1)
        if t < T - 1:
            z[:, o + n:o + n + m] = rng.normal(size=(B, m))
    return z


def _with_bounds(be, lo, up, options=None):
    """the oracle twin's bounds replaced by lo, up ([N_z]: every problem, or [B, N_z]); the twin reads its own Bound objects"""
    clo, cup = be.o.constraint_bounds
    be._bound_args = (lo, up, options, clo, cup)
    be.fixed, be.bounds = sqp.bound_arrays(lo, up, options, clo, cup)
    be.free = (~be.fixed).astype(np.float64)
    be.pinned_value = np.where(be.fixed, lo, 0.0)
    return be


def _car_bounds(n, m, T, x1, xT, u):
    al, au = [-u] * m, [u] * m
    return ([D.Bound(n, m, state_lower=x1, state_upper=x1, action_lower=al, action_upper=au)]
            + [D.Bound(n, m, action_lower=al, action_upper=au)] * (T - 2) + [D.Bound(n, 0, state_lower=xT, state_upper=xT)])


def test_set_bounds_fills_a_problem_row_as_primal_bounds_would():
    model = M.build_car(D, T=51, obstacle="stage")
    n, m, T, x1, xT = model["n"], model["m"], model["T"], model["x1"], model["xT"]
    B = 4
    s = D.solver_from(model, batch=B)
    shared = [v.copy() for v in s.nlp.variable_bounds]
    assert s.nlp.batch_variable_bounds[0].shape == (s.nlp.num_variables,)          # nothing set: the shared pair
    lists = {1: _car_bounds(n, m, T, x1 + np.array([0.1, -0.2, 0.05]), xT, 0.7), 3: _car_bounds(n, m, T, x1, xT - 0.3, 0.25)}
    for b, bl in lists.items():
        s.set_bounds(bl, problem=b)
    lo, up = s.nlp.batch_variable_bounds
    assert lo.shape == up.shape == (B, s.nlp.num_variables)
    for b in range(B):
        if b in lists:         # the row a batch built with that Bound list has
            ref = D.solver_from(dict(model, bounds=lists[b]), batch=1).nlp.variable_bounds
        else:
            ref = shared
        assert np.array_equal(lo[b], ref[0]) and np.array_equal(up[b], ref[1]), b
    assert np.array_equal(s.nlp.variable_bounds[0], shared[0])      # variable_bounds keeps its meaning: the Bound objects
    s.set_bounds(lists[3])                                          # problem=None: every problem
    lo, up = s.nlp.batch_variable_bounds
    assert all(np.array_equal(lo[b], lo[3]) and np.array_equal(up[b], up[3]) for b in range(B))
    s.nlp.set_variable_bounds(None, None)
    assert np.array_equal(s.nlp.batch_variable_bounds[0], shared[0])
    with pytest.raises(ValueError):
        s.nlp.set_variable_bounds(np.zeros((B - 1, s.nlp.num_variables)), np.zeros((B - 1, s.nlp.num_variables)))


@pytest.mark.parametrize("scale", [1.0, 10.0])
def test_bound_arrays_on_rows_equal_the_row_by_row_results(scale):
    """car T = 51: pinned end states, two-sided control bounds, obstacle rows c(z) <= 0; per-problem end states and limits"""
    model = M.build_car(D, T=51, obstacle="stage")
    n, m, T, x1, xT = model["n"], model["m"], model["T"], model["x1"], model["xT"]
    nlp = D.solver_from(model, batch=1).nlp
    clo, cup = nlp.constraint_bounds
    rows = [nlp.primal_bounds(_car_bounds(n, m, T, x1 + 0.1 * k, xT - 0.05 * k, u)) for k, u in enumerate((0.5, 0.3, 2.0, 0.5))]
    lo, up = np.stack([r[0] for r in rows]), np.stack([r[1] for r in rows])
    o = sqp.SQPOptions()
    fixed, bnd = sqp.bound_arrays(lo, up, o, clo, cup, scale=scale)
    assert fixed.shape == bnd["hasL"].shape == bnd["hasU"].shape == (nlp.num_variables,)
    for b, (l1, u1) in enumerate(rows):
        f1, b1 = sqp.bound_arrays(l1, u1, o, clo, cup, scale=scale)
        assert np.array_equal(fixed, f1)
        for k in ("hasL", "hasU", "hasI"):
            assert np.array_equal(bnd[k], b1[k]), k
        for k in ("lo", "up", "pushL", "pushU"):
            assert np.array_equal(bnd[k][b], b1[k]), (k, b)
    # the widened bounds are about each problem's own midpoint
    u_idx = np.nonzero(bnd["hasL"] * bnd["hasU"])[0][0]
    mids = 0.5 * (bnd["lo"][:, u_idx] + bnd["up"][:, u_idx])
    assert np.allclose(mids, 0.5 * (lo[:, u_idx] + up[:, u_idx]))
    assert np.allclose(bnd["up"][:, u_idx] - bnd["lo"][:, u_idx], scale * (up[:, u_idx] - lo[:, u_idx]))


def test_bound_arrays_refuse_rows_of_another_pattern():
    lo = np.array([[0.0, -1.0, -np.inf], [0.5, -2.0, -np.inf]])
    up = np.array([[0.0, 1.0, np.inf], [0.5, 2.0, np.inf]])
    sqp.bound_arrays(lo, up)                                       # same pattern, different values
    for p, i, l, u, what in ((1, 0, 0.5, 0.6, "pinned"), (1, 2, -1.0, np.inf, "lower-bounded"), (1, 1, -np.inf, 2.0, "lower-bounded")):
        l2, u2 = lo.copy(), up.copy()
        l2[p, i], u2[p, i] = l, u
        with pytest.raises(ValueError, match=f"problem {p}, variable index {i}.*{what}"):
            sqp.bound_arrays(l2, u2)
    for l, u in ((3.0, 2.0), (np.nan, 2.0)):
        l2, u2 = lo.copy(), up.copy()
        l2[1, 1], u2[1, 1] = l, u
        with pytest.raises(ValueError, match="problem 1, variable index 1"):
            sqp.bound_arrays(l2, u2)


def _twin_mixed_against_groups(mo, mp, groups, assign, z0, opts):
    """groups: list of (lo, up) [N_z]; assign[b] = group of problem b. Every problem of the mixed solve must carry the bits of
    its group's solve (that group's problems alone, in order, with shared bounds)."""
    osolver = O.solver_from(mo)
    perm, bw = PK.analyze(D.solver_from(mp, batch=1).nlp)
    B = len(assign)
    twin = lambda n: OracleBackend(osolver, n, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band", options=opts)  # noqa: E731
    lo = np.stack([groups[g][0] for g in assign])
    up = np.stack([groups[g][1] for g in assign])
    mixed = sqp.solve(_with_bounds(twin(B), lo, up, opts), z0, options=opts)
    for g, (gl, gu) in enumerate(groups):
        rows = np.nonzero(np.asarray(assign) == g)[0]
        ref = sqp.solve(_with_bounds(twin(len(rows)), gl, gu, opts), z0[rows], options=opts)
        for name in ("z", "lam", "iterations", "converged", "constraint_violation", "dual_residual", "objective"):
            assert np.array_equal(getattr(mixed, name)[rows], getattr(ref, name)), (g, name)
    return mixed


def test_twin_with_per_problem_control_limits_equals_the_grouped_solves():
    """pendulum swing-up, |u| <= 14, 16 or 30 per problem, interleaved (the unconstrained optimum peaks at 18.6)"""
    mo, mp = M.build_pendulum(O, u_bnd=15.0), M.build_pendulum(D, u_bnd=15.0)
    n, m, T = mp["n"], mp["m"], mp["T"]
    nlp = D.solver_from(mp, batch=1).nlp
    groups = [nlp.primal_bounds([D.Bound(n, m, action_lower=[-u], action_upper=[u])] * (T - 1) + [D.Bound(n, 0)]) for u in (14.0, 16.0, 30.0)]
    assign = [0, 1, 2, 1, 0, 2]
    opts = sqp.SQPOptions(max_iter=60, dual_reg=1.0e-6)
    mixed = _twin_mixed_against_groups(mo, mp, groups, assign, _guess(mp, len(assign), 7), opts)
    assert mixed.converged.all()
    U = np.stack([mixed.z[:, t * (n + m) + n] for t in range(T - 1)], axis=1)
    lim = np.array([(14.0, 16.0, 30.0)[g] for g in assign])
    assert np.all(np.abs(U) < lim[:, None]) and np.any(np.abs(U[lim == 14.0]) > 14.0 - 1e-4)


def test_twin_with_per_problem_pinned_start_states_equals_the_grouped_solves():
    """test/solve.jl:227-296 set-up (x1 pinned by equal bounds, xT by a general constraint), a different x1 per group"""
    kw = dict(reference_exact=True)
    mo, mp = M.build_linear_general(O, **kw), M.build_linear_general(D, **kw)
    n, m, T = mp["n"], mp["m"], mp["T"]
    nlp = D.solver_from(mp, batch=1).nlp
    starts = [np.asarray(mp["x1"], float) + d for d in (0.0, 0.5, -0.3)]
    groups = [nlp.primal_bounds([D.Bound(n, m, state_lower=x, state_upper=x)] + [D.Bound(n, m)] * (T - 2) + [D.Bound(n, 0)]) for x in starts]
    assign = [2, 0, 1, 1, 2]
    opts = sqp.SQPOptions(max_iter=20, dual_reg=1.0e-6)
    mixed = _twin_mixed_against_groups(mo, mp, groups, assign, _guess(mp, len(assign), 21), opts)
    assert mixed.converged.all()
    for b, g in enumerate(assign):
        assert np.array_equal(mixed.z[b, :n], starts[g])                    # pinned: exactly the problem's own start state


def test_broker_hands_every_problem_its_own_bounds():
    """driver.solve_batch: the host solver of problem b gets row b (a stand-in task records what it was handed)"""
    from types import SimpleNamespace

    from dto_b200.driver import solve_batch
    mp = M.build_pendulum(D, u_bnd=15.0)
    n, m, T = mp["n"], mp["m"], mp["T"]
    B = 3
    s = D.solver_from(mp, batch=B)
    s.set_bounds([D.Bound(n, m, action_lower=[-7.0], action_upper=[7.0])] * (T - 1) + [D.Bound(n, 0)], problem=1)
    seen = {}

    def task(broker, b, z0, structures, bounds, options, record):
        seen[b] = bounds
        broker.finish(b)
        return SimpleNamespace(x=z0)

    solve_batch(s.nlp, np.zeros((B, s.nlp.num_variables)), task=task)
    lo, up = s.nlp.batch_variable_bounds
    for b in range(B):
        (zl, zu), (cl, cu) = seen[b]
        assert np.array_equal(zl, lo[b]) and np.array_equal(zu, up[b])
    fin = lambda v: v[np.isfinite(v)]  # noqa: E731
    assert np.all(fin(seen[1][0][1]) == 7.0) and np.all(fin(seen[0][0][1]) == 15.0) and np.all(fin(seen[2][0][1]) == 15.0)

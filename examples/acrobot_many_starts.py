"""Many acrobot swing-ups in one batch, each from its own start state -- the workload of MPC over a fleet or of generating a
dataset of trajectories.

    python examples/acrobot_many_starts.py [batch]

The problem is the reference's test/solve.jl:1-138 acrobot: T = 101, both end points pinned by bounds,
`Bound(state_lower = x1, state_upper = x1)` at the first knot and `Bound(state_lower = xT, state_upper = xT)` at the last.
Every problem gets its own start state x1 through `Solver.set_bounds(bounds, problem = b)`, the same list of T Bound objects
the Solver takes, and its own guess (states interpolated from its x1 to xT, random controls). The problems share the bound
pattern (which variables are pinned), so one native solve runs them all in lock step on the device (DESIGN section 10)."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import dto_b200 as D  # noqa: E402
from examples import models as M  # noqa: E402


def start_states(batch, seed=0):
    """measured start states: both links within 0.3 rad of hanging down, angular rates within 0.2 rad/s"""
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.uniform(-0.3, 0.3, (batch, 2)), rng.uniform(-0.2, 0.2, (batch, 2))], axis=1)


def build(batch=64, T=101, seed=0, per_problem=True):
    """the batch with its guesses; per_problem=False keeps the model's shared bounds (every problem pinned at x1 = 0) for
    the same guesses. Returns (solver, start states [batch, 4])."""
    model = M.build_acrobot(D, T=T, stage_endpoint_constraints=False)
    n, m, xT = model["n"], model["m"], model["xT"]
    solver = D.solver_from(model, batch=batch)
    starts = start_states(batch, seed)
    rng = np.random.default_rng(seed + 1)
    for b in range(batch):
        x1 = starts[b]
        if per_problem:
            solver.set_bounds([D.Bound(n, m, state_lower=x1, state_upper=x1)] + [D.Bound(n, m)] * (T - 2)
                              + [D.Bound(n, 0, state_lower=xT, state_upper=xT)], problem=b)
        solver.initialize_states(D.linear_interpolation(x1, xT, T), problem=b)
        solver.initialize_controls([rng.normal(size=m) for _ in range(T - 1)], problem=b)
    return solver, (starts if per_problem else np.tile(model["x1"], (batch, 1)))


def accepted(res, starts, xT):
    """test/solve.jl:134-137 for every problem, against its own start state"""
    n = starts.shape[1]
    Z = np.asarray(res.z)
    e1 = np.linalg.norm(Z[:, :n] - starts, axis=1)
    eT = np.linalg.norm(Z[:, -n:] - xT, axis=1)
    return (np.asarray(res.constraint_violation) < 1e-6) & (e1 < 1e-3) & (eT < 1e-3)


def main(batch=64, T=101):
    solver, starts = build(batch, T)
    xT = np.array([np.pi, 0.0, 0.0, 0.0])
    res = solver.solve(options=dict(max_iter=300))
    ok = accepted(res, starts, xT)
    print(f"{int(ok.sum())} of {batch} swing-ups solved, each from its own start state (||x_1 - x1_b||, ||x_T - xT|| < 1e-3, "
          f"||c||_inf < 1e-6); median iterations {float(np.median(res.iterations)):.0f}; kernels launched {solver.sqp_launches}")
    xs, _ = solver.get_trajectory(1)
    print("problem 1: x1 =", starts[1], " x_1 =", xs[0], " x_T =", xs[-1])
    solver.nlp.close()


if __name__ == "__main__":
    main(int(sys.argv[1]) if len(sys.argv) > 1 else 64)

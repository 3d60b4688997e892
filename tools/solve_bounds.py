"""Native solves with bound values per problem (dto_sqp_solve_ex), timed on the GPU:   python tools/solve_bounds.py [B] [out.jsonl]
  * examples/acrobot_many_starts.py at B problems, each pinned at its own start state, against the same B guesses under the
    model's shared bounds (every problem pinned at x1 = 0): accepted fraction (test/solve.jl:134-137 against the problem's own
    start state), median iterations, wall time;
  * the reference's cartpole example (T = 101, rollout guess) at B problems with |u| <= 3, 4, 6, 10 per problem (problem b
    takes limit b % 4), against the same guesses under the shared |u| <= 3.
Every batch is first solved for one untimed iteration, then three times timed (the median is `seconds`); a timed region runs
from the host guesses to the host results. One JSON line per run, on stdout and appended to out.jsonl; the first line names the card and its power limit."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import dto_b200 as D  # noqa: E402
from dto_b200 import sqp  # noqa: E402
from examples import acrobot_many_starts as AMS  # noqa: E402
from examples import models as M  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(device=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None)


def timed(nlp, z0, max_iter, repeats=3):
    """the result and the median wall time of `repeats` solves (all of them listed: the card may be shared)"""
    sqp.solve_native(nlp, z0, options=sqp.SQPOptions(max_iter=1))
    times = []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = sqp.solve_native(nlp, z0, options=sqp.SQPOptions(max_iter=max_iter))
        times.append(time.perf_counter() - t0)
    return res, float(np.median(times)), times


def acrobot(B, per_problem):
    solver, starts = AMS.build(B, 101, seed=0, per_problem=per_problem)
    res, dt, times = timed(solver.nlp, solver._initial, 300)
    ok = AMS.accepted(res, starts, np.array([np.pi, 0.0, 0.0, 0.0]))
    solver.nlp.close()
    return dict(workload=f"acrobot swing-up T=101 (test/solve.jl:1-138), {B} problems, "
                + ("each pinned at its own start state (bounds_stride = N_z)" if per_problem else "shared bounds, start pinned at x1 = 0 (bounds_stride = 0)"),
                B=B, seconds=dt, seconds_each=times, solves_per_s=B / dt, accepted_frac=float(ok.mean()), converged_frac=float(res.converged.mean()),
                iterations_median=float(np.median(res.iterations)), iterations_run=res.stats["iterations"], launches=res.stats["launches"])


def cartpole(B, limits):
    model = M.build_cartpole(D, T=101)
    n, m, T = model["n"], model["m"], model["T"]
    s = D.solver_from(model, batch=B)
    s.nlp.set_parameters(np.tile(np.concatenate([model["x1"], model["xT"]]), (B, 1)))
    for k, u in enumerate(limits):
        if len(limits) > 1:
            bl = [D.Bound(n, m, action_lower=[-u], action_upper=[u])] * (T - 1) + [D.Bound(n, 0)]
            for b in range(k, B, len(limits)):
                s.set_bounds(bl, problem=b)
    rng = np.random.default_rng(7)
    rolls = []
    for _ in range(64):         # the example's guess, 64 distinct ones (problem b takes guess b % 64)
        u0 = np.array([0.01 * (1.0 + 0.2 * rng.normal())])
        xs = [model["x1"].astype(float)]
        for _ in range(T - 1):
            xs.append(np.array(M.cartpole_rk3_explicit(xs[-1], u0, np.zeros(0)), dtype=float))
        rolls.append((u0, xs))
    for b in range(B):
        u0, xs = rolls[b % 64]
        s.initialize_states(xs, problem=b)
        s.initialize_controls([u0] * (T - 1), problem=b)
    res, dt, times = timed(s.nlp, s._initial, 600)
    lim = np.array([limits[b % len(limits)] for b in range(B)])
    U = np.stack([res.z[:, t * (n + m) + n] for t in range(T - 1)], axis=1)
    per = {str(u): dict(converged_frac=float(res.converged[lim == u].mean()), iterations_median=float(np.median(res.iterations[lim == u])),
                        at_bound=float((np.abs(U[lim == u]) > 0.997 * u).mean())) for u in limits}
    s.nlp.close()
    return dict(workload=f"cartpole example T=101, rollout guess, {B} problems, |u| <= " + ("/".join(f"{u:g}" for u in limits) + " per problem (bounds_stride = N_z)"
                if len(limits) > 1 else f"{limits[0]:g} shared (bounds_stride = 0)"),
                B=B, seconds=dt, seconds_each=times, solves_per_s=B / dt, converged_frac=float(res.converged.mean()), staged_frac=float(res.staged.mean()),
                iterations_median=float(np.median(res.iterations)), u_within_limits=bool(np.all(np.abs(U) < lim[:, None])), per_limit=per,
                iterations_run=res.stats["iterations"], launches=res.stats["launches"])


if __name__ == "__main__":
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
    out = sys.argv[2] if len(sys.argv) > 2 else None
    lines = [card()]
    for fn in (lambda: acrobot(B, True), lambda: acrobot(B, False), lambda: cartpole(B, (3.0, 4.0, 6.0, 10.0)), lambda: cartpole(B, (3.0,))):
        lines.append(fn())
        print(json.dumps(lines[-1]), flush=True)
    if out:
        with open(out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")

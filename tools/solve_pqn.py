"""Three Hessian arms of the native solver on the same seeded guesses: "exact" (models built with Hessians), "knot-bfgs" and
"partitioned-bfgs" (models built without them, the reference's default evaluate_hessian = false). Workloads:
  - the reference's test/solve.jl:1-138 set-up: acrobot swing-up, T = 101, both end points pinned by bounds, B seeded guesses
    (states interpolated from x1 to xT, controls ~ N(0, 1), as tools/solve_qn.py); acceptance ||c||_inf < 1e-6 and
    ||x_1 - x1||, ||x_T - xT|| < 1e-3 (test/solve.jl:134-137);
  - the reference's cartpole example: |u| <= 3, pinned end states, its rollout guess, 64 problems (interior-point mode);
    solved = converged with ||c||_inf < 1e-6.
    python tools/solve_pqn.py [B] [max_iter] [out.jsonl]
Prints (and appends to out.jsonl) one JSON line per (workload, arm) -- fractions accepted / converged, iterations, seconds,
the solver's stats counters (inertia-correction factorisations among them) and phase_ms -- then one line per quasi-Newton mode
with its kernels' share of the CUDA kernel time on the acrobot workload, from a torch.profiler run of its own."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import dto_b200 as D  # noqa: E402
from dto_b200 import sqp  # noqa: E402
from examples import models as M  # noqa: E402
from solve_config3 import initial_guess  # noqa: E402
from solve_qn import card  # noqa: E402

ARMS = ("exact", "knot-bfgs", "partitioned-bfgs")
KERNELS = {"knot-bfgs": ("k_qn_update",), "partitioned-bfgs": ("k_pqn_update", "k_pqn_assemble")}


def _summary(res, ok, dt):
    it = res.iterations
    st = dict(res.stats)
    return {"seconds": dt, "accepted_frac": float(ok.mean()), "converged_frac": float(np.asarray(res.converged, bool).mean()),
            "iterations": {"median": float(np.median(it)), "max": float(np.max(it)),
                           "median_converged": float(np.median(it[np.asarray(res.converged, bool)])) if np.any(res.converged) else None},
            "objective_median_accepted": float(np.median(res.objective[ok])) if ok.any() else None,
            "ms_per_iteration": 1e3 * dt / max(1, st["iterations"]), "phase_ms": st.pop("phase_ms"), "stats": st}


def acrobot(arm, B, max_iter, z0):
    model = M.build_acrobot(D, T=101, stage_endpoint_constraints=False, evaluate_hessian=(arm == "exact"))
    nlp = D.solver_from(model, batch=B).nlp
    sqp.solve_native(nlp, z0, options=sqp.SQPOptions(max_iter=1, hessian_approximation=arm))    # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = sqp.solve_native(nlp, z0, options=sqp.SQPOptions(max_iter=max_iter, hessian_approximation=arm))
    dt = time.perf_counter() - t0
    nlp.close()
    n = model["n"]
    ok = ((res.constraint_violation < 1e-6) & (np.linalg.norm(res.z[:, :n] - model["x1"], axis=1) < 1e-3)
          & (np.linalg.norm(res.z[:, -n:] - model["xT"], axis=1) < 1e-3))
    return dict({"workload": f"test/solve.jl:1-138 acrobot T=101, pinned end points, B={B}, native solver", "hessian_approximation": arm,
                 "B": B, "max_iter": max_iter}, **_summary(res, ok, dt))


def cartpole(arm, B, max_iter):
    T = 101
    model = M.build_cartpole(D, T=T, evaluate_hessian=(arm == "exact"))
    n, m, x1, xT = model["n"], model["m"], model["x1"], model["xT"]
    s = D.solver_from(model, batch=B)
    s.nlp.set_parameters(np.tile(np.concatenate([x1, xT]), (B, 1)))
    rng = np.random.default_rng(0)
    for b in range(B):
        u0 = np.array([0.01 * (1.0 + 0.2 * rng.normal())])
        xs = [x1.astype(float)]
        for _ in range(T - 1):
            xs.append(np.array(M.cartpole_rk3_explicit(xs[-1], u0, np.zeros(0)), dtype=float))
        s.initialize_states(xs, problem=b)
        s.initialize_controls([u0] * (T - 1), problem=b)
    s.solve(options=dict(max_iter=1, hessian_approximation=arm))       # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = s.solve(options=dict(max_iter=max_iter, hessian_approximation=arm))
    dt = time.perf_counter() - t0
    assert s.broker is None
    c = np.zeros((B, s.nlp.num_constraint))
    s.nlp.eval_constraint(c, res.z)
    ok = np.asarray(res.converged, bool) & (np.max(np.abs(c), axis=1) < 1e-6)
    s.nlp.close()
    return dict({"workload": f"cartpole example (|u| <= 3, pinned end states, rollout guess), T=101, B={B}, native solver",
                 "hessian_approximation": arm, "B": B, "max_iter": max_iter}, **_summary(res, ok, dt))


def kernel_share(arm, B, max_iter, z0):
    """the arm's quasi-Newton kernels' share of the CUDA kernel time of one acrobot solve (torch.profiler, a run of its own)"""
    from torch.profiler import ProfilerActivity, profile
    model = M.build_acrobot(D, T=101, stage_endpoint_constraints=False, evaluate_hessian=False)
    nlp = D.solver_from(model, batch=B).nlp
    sqp.solve_native(nlp, z0, options=sqp.SQPOptions(max_iter=1, hessian_approximation=arm))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sqp.solve_native(nlp, z0, options=sqp.SQPOptions(max_iter=max_iter, hessian_approximation=arm))
        torch.cuda.synchronize()
    nlp.close()
    tot, mine = 0.0, {k: [0.0, 0] for k in KERNELS[arm]}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if e.key.startswith("Memcpy") or e.key.startswith("Memset"):
            continue
        tot += t
        for k in mine:
            if k in e.key:
                mine[k][0] += t
                mine[k][1] += e.count
    out = {"hessian_approximation": arm, "kernel_us": tot}
    for k, (t, n) in mine.items():
        out.update({f"{k}_us": t, f"{k}_share": t / tot if tot else None, f"{k}_calls": n})
    return out


def main():
    a = sys.argv[1:]
    B = int(a[0]) if a else 4096
    max_iter = int(a[1]) if len(a) > 1 else 600
    out = a[2] if len(a) > 2 else None
    z0 = initial_guess(M.build_acrobot(D, T=101, stage_endpoint_constraints=False, evaluate_hessian=False), B)
    gpu = card()
    rows = [dict(acrobot(arm, B, max_iter, z0), gpu=gpu) for arm in ARMS]
    rows += [dict(cartpole(arm, 64, max_iter), gpu=gpu) for arm in ARMS]
    rows += [dict(kernel_share(arm, B, max_iter, z0), gpu=gpu, B=B, max_iter=max_iter, note="torch.profiler run of its own, acrobot")
             for arm in ("knot-bfgs", "partitioned-bfgs")]
    for r in rows:
        line = json.dumps(r)
        print(line, flush=True)
        if out:
            with open(out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()

"""BASELINE config 3: acrobot swing-up T=101, batch 4096, FULL SOLVES with device-resident callbacks
(/root/reference/examples/acrobot/acrobot.jl:94-133; acceptance of /root/reference/test/solve.jl:134-137:
||x_1 - x1|| < 1e-3 and ||x_T - xT|| < 1e-3). Every problem starts from the example's guess -- states
linearly interpolated from x1 to xT, controls ~ N(0, 1) (the example uses unseeded randn; here seeded per
problem) -- and is solved by the lock-step batched Newton-KKT solver (dto_b200/sqp.py). Ipopt is absent:
iterate parity with the reference's own solver is unverifiable and not claimed.
    python tools/solve_config3.py [B] [T] [max_iter] [model] [sqp|native]      -> one JSON line
`native` runs the same algorithm inside libdto.so (dto_sqp_solve: bookkeeping kernels instead of torch glue); its timed
region includes the host->device copy of the guesses and the device->host copy of the results."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import dto_b200 as D  # noqa: E402
from dto_b200 import sqp  # noqa: E402
from examples import models as M  # noqa: E402


def initial_guess(model, B, seed=20261017 + 3000):
    T, n, m = model["T"], model["n"], model["m"]
    x1, xT = model["x1"], model["xT"]
    rng = np.random.default_rng(seed)
    z = np.zeros((B, T * n + (T - 1) * m))
    for t in range(T):
        o = t * (n + m)
        z[:, o:o + n] = x1 + (xT - x1) * t / (T - 1)          # linear_interpolation (src/utils.jl:1-10)
        if t < T - 1:
            z[:, o + n:o + n + m] = rng.normal(size=(B, m))   # u_guess = randn (acrobot.jl:127)
    return z


def run_native(model, nlp, z0, o, name, B, T, max_iter):
    sqp.solve_native(nlp, z0[:], options=sqp.SQPOptions(max_iter=1))      # warm-up: lazy allocations, plan tables
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = sqp.solve_native(nlp, z0, options=o)
    dt = time.perf_counter() - t0
    n = model["n"]
    Z, cv, it = res.z, res.constraint_violation, res.iterations
    e1 = np.linalg.norm(Z[:, :n] - model["x1"], axis=1)
    eT = np.linalg.norm(Z[:, -n:] - model["xT"], axis=1)
    ok = (cv < 1e-6) & (e1 < 1e-3) & (eT < 1e-3)
    f = res.objective
    return {"workload": f"{name} swing-up T={T}, B={B}, full solves (native lock-step Newton-KKT SQP: dto_sqp_solve)", "method": "native",
            "B": B, "T": T, "max_iter": max_iter, "seconds": dt, "solves_per_s": B / dt, "knot_iterations_per_s": float(it.sum()) * T / dt,
            "accepted_frac": float(ok.mean()), "converged_frac": float(res.converged.mean()),
            "accept_rule": "||c||_inf < 1e-6 and ||x_1 - x1||, ||x_T - xT|| < 1e-3 (test/solve.jl:134-137)",
            "converge_rule": f"||c||_inf <= {o.tol_constraint} and ||g + J'lambda||_inf <= {o.tol_dual}",
            "iterations": {"median": float(np.median(it)), "p90": float(np.percentile(it, 90)), "max": float(it.max())},
            "objective": {"median": float(np.median(f)), "min": float(f.min()), "max": float(f.max())},
            "cv_max_accepted": float(cv[ok].max()) if ok.any() else None, "dual_residual_median": float(np.median(res.dual_residual)),
            "gpu_launches": res.stats["launches"], "factorisations": res.stats["factorisations"], "host_syncs": res.stats["syncs"],
            "refactorisations": res.stats["refactorisations"], "corrections": res.stats["corrections"], "search_rounds": res.stats["search_rounds"], "multi_trial_passes": res.stats["multi_trial_passes"], "phase_ms": res.stats["phase_ms"],
            "iterations_run": res.stats["iterations"], "ms_per_iteration": 1e3 * dt / max(1, res.stats["iterations"])}


def run(B=4096, T=101, max_iter=300, name="acrobot", options=None, method="sqp"):
    model = M.BUILDERS[name](D, T=T)
    solver = D.solver_from(model, batch=B)
    nlp = solver.nlp
    z0 = initial_guess(model, B)
    o = sqp.SQPOptions(max_iter=max_iter, **(options or {}))
    if method == "native":
        out = run_native(model, nlp, z0, o, name, B, T, max_iter)
        nlp.close()
        return out
    be = sqp.DeviceBackend(nlp, dual_reg=o.dual_reg)
    zt = torch.as_tensor(z0, device=be.xp.device)
    l0 = nlp.launch_count()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = sqp.solve(be, zt, options=o)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    launches = res.backend.total_launches()
    Z = res.z.cpu().numpy()
    n = model["n"]
    e1 = np.linalg.norm(Z[:, :n] - model["x1"], axis=1)
    eT = np.linalg.norm(Z[:, -n:] - model["xT"], axis=1)
    cv = res.constraint_violation.cpu().numpy()
    dr = res.dual_residual.cpu().numpy()
    it = res.iterations.cpu().numpy()
    conv = res.converged.cpu().numpy()
    ok = (cv < 1e-6) & (e1 < 1e-3) & (eT < 1e-3)
    f = res.objective.cpu().numpy()
    if res.backend is not be:
        res.backend.close()
    be.close()
    return {"workload": f"{name} swing-up T={T}, B={B}, full solves (lock-step Newton-KKT SQP, device-resident callbacks + KKT)",
            "B": B, "T": T, "max_iter": max_iter, "seconds": dt, "solves_per_s": B / dt, "knot_iterations_per_s": float(it.sum()) * T / dt,
            "accepted_frac": float(ok.mean()), "converged_frac": float(conv.mean()),
            "accept_rule": "||c||_inf < 1e-6 and ||x_1 - x1||, ||x_T - xT|| < 1e-3 (test/solve.jl:134-137)",
            "converge_rule": f"||c||_inf <= {o.tol_constraint} and ||g + J'lambda||_inf <= {o.tol_dual}",
            "iterations": {"median": float(np.median(it)), "p90": float(np.percentile(it, 90)), "max": float(it.max())},
            "objective": {"median": float(np.median(f)), "min": float(f.min()), "max": float(f.max())},
            "cv_max_accepted": float(cv[ok].max()) if ok.any() else None, "dual_residual_median": float(np.median(dr)),
            "gpu_launches": int(launches), "ms_per_iteration": 1e3 * dt / max(1.0, float(it.max()))}


if __name__ == "__main__":
    a = sys.argv[1:]
    opts = json.loads(os.environ.get("DTO_SQP_OPTIONS", "{}"))   # e.g. '{"max_backtrack": 12}'
    out = run(int(a[0]) if a else 4096, int(a[1]) if len(a) > 1 else 101, int(a[2]) if len(a) > 2 else 300, a[3] if len(a) > 3 else "acrobot",
              options=opts, method=a[4] if len(a) > 4 else "sqp")
    out["options"] = opts
    print(json.dumps(out))

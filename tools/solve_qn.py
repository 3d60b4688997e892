"""The reference's test/solve.jl:1-138 set-up WITHOUT Hessians (the reference's default evaluate_hessian = false): acrobot
swing-up, T = 101, both end points pinned by Bound(state_lower = state_upper), a batch of B seeded guesses (states
interpolated from x1 to xT, controls ~ N(0, 1), as tools/solve_config3.py) -- solved by the native solver's knot-block
damped BFGS mode (hessian_approximation = "knot-bfgs"), and the same guesses by the exact-Hessian native solver.
    python tools/solve_qn.py [B] [max_iter] [out.jsonl]
Prints (and appends to out.jsonl) one JSON line per arm, then one with k_qn_update's share of the kernel time from a
torch.profiler run of its own. Acceptance: ||c||_inf < 1e-6 and ||x_1 - x1||, ||x_T - xT|| < 1e-3 (test/solve.jl:134-137)."""
import json
import os
import subprocess
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


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name(0)


def solve(hessian, B, max_iter, z0):
    model = M.build_acrobot(D, T=101, stage_endpoint_constraints=False, evaluate_hessian=(hessian == "exact"))
    nlp = D.solver_from(model, batch=B).nlp
    o = sqp.SQPOptions(max_iter=max_iter, hessian_approximation=hessian)
    sqp.solve_native(nlp, z0, options=sqp.SQPOptions(max_iter=1, hessian_approximation=hessian))    # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = sqp.solve_native(nlp, z0, options=o)
    dt = time.perf_counter() - t0
    nlp.close()
    n = model["n"]
    e1 = np.linalg.norm(res.z[:, :n] - model["x1"], axis=1)
    eT = np.linalg.norm(res.z[:, -n:] - model["xT"], axis=1)
    ok = (res.constraint_violation < 1e-6) & (e1 < 1e-3) & (eT < 1e-3)
    it = res.iterations
    return {"workload": f"test/solve.jl:1-138 acrobot T=101, pinned end points, B={B}, native solver", "hessian_approximation": hessian,
            "B": B, "max_iter": max_iter, "seconds": dt, "accepted_frac": float(ok.mean()), "converged_frac": float(res.converged.mean()),
            "iterations": {"median": float(np.median(it)), "max": float(it.max()),
                           "median_converged": float(np.median(it[res.converged])) if res.converged.any() else None},
            "objective_median_accepted": float(np.median(res.objective[ok])) if ok.any() else None,
            "iterations_run": res.stats["iterations"], "ms_per_iteration": 1e3 * dt / max(1, res.stats["iterations"]),
            "launches": res.stats["launches"], "phase_ms": res.stats["phase_ms"]}


def kernel_share(B, max_iter, z0):
    """k_qn_update's share of the CUDA kernel time of one knot-bfgs solve (torch.profiler, a run of its own)"""
    from torch.profiler import ProfilerActivity, profile
    model = M.build_acrobot(D, T=101, stage_endpoint_constraints=False, evaluate_hessian=False)
    nlp = D.solver_from(model, batch=B).nlp
    o = sqp.SQPOptions(max_iter=max_iter, hessian_approximation="knot-bfgs")
    sqp.solve_native(nlp, z0, options=sqp.SQPOptions(max_iter=1, hessian_approximation="knot-bfgs"))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sqp.solve_native(nlp, z0, options=o)
        torch.cuda.synchronize()
    nlp.close()
    tot, qn, calls = 0.0, 0.0, 0
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if e.key.startswith("Memcpy") or e.key.startswith("Memset"):
            continue
        tot += t
        if "k_qn_update" in e.key:
            qn += t
            calls += e.count
    return {"k_qn_update_us": qn, "kernel_us": tot, "k_qn_update_share": qn / tot if tot else None, "k_qn_update_calls": calls}


def main():
    a = sys.argv[1:]
    B = int(a[0]) if a else 4096
    max_iter = int(a[1]) if len(a) > 1 else 600
    out = a[2] if len(a) > 2 else None
    z0 = initial_guess(M.build_acrobot(D, T=101, stage_endpoint_constraints=False, evaluate_hessian=False), B)
    gpu = card()
    rows = [dict(solve(h, B, max_iter, z0), gpu=gpu) for h in ("knot-bfgs", "exact")]
    rows.append(dict(kernel_share(B, max_iter, z0), gpu=gpu, B=B, max_iter=max_iter, note="torch.profiler run of its own, knot-bfgs"))
    for r in rows:
        line = json.dumps(r)
        print(line, flush=True)
        if out:
            with open(out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()

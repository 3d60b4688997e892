#!/usr/bin/env python
"""bench.py -- knot-point Jacobian+Hessian evaluations per second (FP64), BASELINE.json metric.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (config.workload): BASELINE configs[1] -- cartpole swing-up, T=101, B=4096 problems PER
GPU (weak scaling: each rank owns its own contiguous shard of the global batch, no collective on
the data path), callback evaluation only. One step = one fused Jacobian + Hessian-of-Lagrangian
pass over the rank's batch.

  value     evals/s with (z, lambda, sigma, w) resident in HBM; timed on the device with CUDA
            events on the launching stream, max over ranks, 3 rotating input/output sets
            (387 MB > 126 MB L2) so no step finds its data in L2.
  e2e       the same metric through the public host API (pinned host buffers -> set_x/set_duals ->
            eval_jacobian_hessian -> host J/H), copies inside the timed region.
  roofline  algorithmic bytes (8(N_z+N_c+N_w+nnz_J+nnz_H)+8 per problem) / kernel time vs the
            measured HBM copy bandwidth (MEASURED_PEAKS.json); plus an FP64-pipe estimate.
  cpu_baseline  the oracle's C twin (no-CSE, "what Symbolics 0.1.x emits") on the host cores.

--impl reference times that C twin itself (the reference needs Julia + Ipopt, absent here).

--dump-outputs DIR writes what the last timed step computed, as the host API would return it (J and H, float64), to
DIR/jacobian.npy and DIR/hessian.npy: rank 0's rows of a fixed, seeded sample of its problems (under 64 MB). The inputs
are seeded, so two builds run with the same arguments can be compared output for output.

The run writes nothing into the source tree: a model library it has to compile goes to a temporary directory.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # no __pycache__ in the source tree
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "knot-point Jac+Hessian evals/sec (FP64)"
UNIT = "knot-evals/s"
DUMP_BYTES = 60 * 10**6  # --dump-outputs: sampled problems x (J + H) rows, under 64 MB with the .npy headers


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def _ncu_headline():
    """Counters of the one committed `ncu --set full` capture of the shipped headline kernel
    (profiles/ncu_headline.json, written by tools/ncu_to_json.py): DRAM bytes per launch, executed FP64
    instructions per knot (SASS) and the FP64-pipe utilisation counter."""
    p = os.path.join(ROOT, "profiles", "ncu_headline.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


def _kkt_traffic():
    p = os.path.join(ROOT, "profiles", "traffic_kkt_r01.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


def _fp64_peak():
    p = os.path.join(ROOT, "profiles", "fp64_peak_r01.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["dfma_per_s"])
    return 16.7e12


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,utilization.gpu,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        sm, mx, reasons, pw = [], [], set(), []
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw),
                "window": "timed region + identical untimed continuation (>=1 s under load)"}


def host_threads() -> int:
    """All host cores this process may use (torchrun exports OMP_NUM_THREADS=1: do not trust it)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def bind_near_gpu(device: int):
    """Pin this process to the host cores NVML reports as local to `device` BEFORE any pinned host buffer is
    allocated (first touch puts the pages on that NUMA node): with one process per GPU the 8 ranks' D2H/H2D
    streams then land on the memory controllers next to their own PCIe root instead of all on node 0.
    Returns a short description for the JSON line; silently does nothing where NVML is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device)
        before = len(os.sched_getaffinity(0))
        pynvml.nvmlDeviceSetCpuAffinity(h)
        after = sorted(os.sched_getaffinity(0))
        node = None
        try:
            bus = pynvml.nvmlDeviceGetPciInfo(h).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            with open(f"/sys/bus/pci/devices/{bus[-12:].lower()}/numa_node") as f:
                node = int(f.read().strip())
        except Exception:  # noqa: BLE001
            pass
        return {"cpus": len(after), "of": before, "numa_node": node}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:80]}


def build_c_baseline(T: int, verbose=False):
    from examples import models as M
    from oracle import api as O, cgen
    mo = M.build_cartpole(O, T=T, evaluate_hessian=True, parameterized=True)
    osolver = O.solver_from(mo, parameters=[np.zeros(8) for _ in range(T)] + [np.zeros(0)])
    return cgen.build_c_oracle(osolver, f"cartpole{T}", shared_parameters=True, cse=False, verbose=verbose), mo


def time_cpu(co, z, lam, sigma, w, threads: int, budget_s: float = 10.0):
    """Jac+Hess on a bounded sample: up to the whole batch, repeated until ~budget_s of wall time
    has been spent; returns (evals/s, problems per pass, passes, seconds)."""
    T = co.T
    probe = min(z.shape[0], max(threads, 8))
    t = time.time()
    co.eval(8 | 16, z[:probe], lam[:probe], sigma[:probe], w[:probe], threads)
    dt = max(time.time() - t, 1e-6)
    Bs = int(min(z.shape[0], max(probe, probe * budget_s / dt)))
    zz, ll, ss, ww = z[:Bs], lam[:Bs], sigma[:Bs], w[:Bs]
    t = time.time()
    co.eval(8 | 16, zz, ll, ss, ww, threads)
    one = max(time.time() - t, 1e-6)
    reps = int(max(1, min(200, budget_s / one)))
    t = time.time()
    for _ in range(reps):
        co.eval(8 | 16, zz, ll, ss, ww, threads)
    dt = time.time() - t
    return Bs * T * reps / dt, Bs, reps, dt


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from util import make_inputs
    co, mo = build_c_baseline(args.T)
    threads = host_threads()
    Bs = args.ref_sample if args.ref_sample > 0 else args.batch
    z, lam, sigma, w = make_inputs("cartpole", mo, co.NZ, co.NC, co.NW, Bs, config=2, shard=0)
    what = 8 | 16
    for _ in range(args.warmup):
        co.eval(what, z, lam, sigma, w, threads)
    t0 = time.time()
    for _ in range(args.steps):
        co.eval(what, z, lam, sigma, w, threads)
    dt = time.time() - t0
    value = Bs * args.T * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"cartpole swing-up T={args.T}, B={args.batch} per GPU, fused Jacobian+Hessian callbacks",
                   "note": "the Julia reference cannot run here (no Julia/Ipopt); this arm times the oracle's C twin of the "
                           "reference callbacks (no-CSE element code, reference loop structure) on the host cores"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": f"{Bs} problems x T={args.T} per step (B={args.batch}), gcc -O2 -fopenmp, no-CSE element code"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))
    return 0


def bench_kkt(torch, n, stream, zp, lp, sp_, peak):
    """Secondary measurement (SURVEY 8f N3, not the headline): the device-resident consumer of J and H.
    One step = gradient + constraint + fused Jacobian/Hessian callbacks + KKT right-hand side + banded
    LDL' factorisation and solve for every problem of the batch (pendulum.jl:124-211 batched)."""
    from dto_b200 import kkt as PK
    B = n.batch
    k = PK.KKTSystem(n)
    steps = 30
    out = {}
    for name, cb in (("ms_kkt_kernels", False), ("ms_step", True)):
        for _ in range(3):
            k.launch(cb)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(steps):
                k.launch(cb)
            e1.record(stream)
        torch.cuda.synchronize()
        out[name] = e0.elapsed_time(e1) / steps
    solp = torch.empty((B, k.dim), dtype=torch.float64).pin_memory().numpy()
    for _ in range(2):
        k.solve(solp, variables=zp, scaling=sp_, duals=lp)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reps = 5
    for _ in range(reps):
        k.solve(solp, variables=zp, scaling=sp_, duals=lp)
    torch.cuda.synchronize()
    e2e_ms = 1e3 * (time.perf_counter() - t0) / reps
    alg = 8 * (n.num_jacobian + n.num_hessian + n.num_variables + 2 * n.num_constraint + 3 * k.dim) + 2 * k.factor_bytes_per_problem
    gbs = alg * B / (out["ms_kkt_kernels"] * 1e-3) / 1e9
    res = {"what": "device-resident KKT assembly + banded LDL' solve of all problems (consumer of J, H; SURVEY 8f N3)",
           "dim": k.dim, "half_bandwidth": k.bandwidth, "ms_kkt_kernels": out["ms_kkt_kernels"], "ms_step_callbacks_plus_kkt": out["ms_step"],
           "kkt_solves_per_s": B / (out["ms_kkt_kernels"] * 1e-3), "newton_steps_per_s": B / (out["ms_step"] * 1e-3),
           "e2e_ms_host_z_lambda_to_host_solution": e2e_ms, "e2e_d2h_bytes": 8 * B * k.dim,
           "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                        "algorithmic_bytes_per_problem": alg, "traffic": _kkt_traffic().get("dram_bytes_per_launch"),
                        "traffic_source": _kkt_traffic().get("source"),
                        "note": "read J,H,g,c,y once; write+read h; write+read the factor once; write the solution"}}
    k.close()
    return res


def sample_outputs(torch, nlp) -> dict:
    """Device copies of J and H of a fixed, seeded sample of the batch's problems (rows in ascending order), enqueued on
    the current stream: taken right behind the last timed step, before later work overwrites the arrays."""
    from dto_b200.evaluator import A_H, A_J
    from dto_b200.sqp import _CudaArray
    B = nlp.batch
    k = min(B, DUMP_BYTES // (8 * (nlp.num_jacobian + nlp.num_hessian)))
    dev = torch.device("cuda", nlp.shard_device(0))
    rows = torch.as_tensor(np.sort(np.random.default_rng(0).choice(B, size=k, replace=False)), device=dev)
    out = {}
    for name, arr, width in (("jacobian", A_J, nlp.num_jacobian), ("hessian", A_H, nlp.num_hessian)):
        view = torch.as_tensor(_CudaArray(nlp.device_pointer(arr, 0), (B, width)), device=dev)
        out[name] = view.index_select(0, rows)
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    binding = None if args.no_bind else bind_near_gpu(local)
    if world > 1:
        # NCCL prints its version banner on stdout when the first communicator is created: keep stdout
        # for the one JSON line by pointing fd 1 at stderr until the communicator exists
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    import dto_b200 as D
    from dto_b200.evaluator import A_H, A_J, A_LAMBDA, A_SIGMA, A_W, A_Z, K_JAC_HESS
    from examples import models as M
    from util import make_inputs

    T = args.T
    strong = args.scaling == "strong"
    if strong:  # the global batch is fixed: contiguous shards of ceil(B/N) problems (sharding.partition)
        from dto_b200 import sharding
        B = sharding.partition(args.batch, world)[rank][1]
        B_total = args.batch
    else:
        B = args.batch
        B_total = args.batch * world
    model = M.build_cartpole(D, T=T, evaluate_hessian=True, parameterized=True)
    solver = D.solver_from(model, batch=B, devices=[local])
    nlp0 = solver.nlp
    R = 3  # rotating input/output sets: 3 x 129 MB > 126 MB L2
    nlps = [nlp0] + [nlp0.new_batch() for _ in range(R - 1)]
    stream = torch.cuda.Stream()
    host = []
    for i, n in enumerate(nlps):
        z, lam, sigma, w = make_inputs("cartpole", model, n.num_variables, n.num_constraint, n.num_parameter, B, config=2,
                                       shard=rank * R + i)
        n.set_parameters(w)
        n.set_x(z)
        n.set_duals(sigma, lam)
        n.set_stream(stream.cuda_stream)
        host.append((z, lam, sigma, w))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    with torch.cuda.stream(stream):
        for i in range(max(args.warmup, 3)):
            nlps[i % R].launch(K_JAC_HESS)
        barrier()
        n0 = sum(n.launch_count() for n in nlps)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_start = time.time()
        e0.record(stream)
        for i in range(args.steps):
            nlps[i % R].launch(K_JAC_HESS)
        e1.record(stream)
        dumped = sample_outputs(torch, nlps[(args.steps - 1) % R]) if args.dump_outputs and rank == 0 else None
        barrier()
        ms = e0.elapsed_time(e1)
        n1 = sum(n.launch_count() for n in nlps)
        # identical untimed continuation so the clock sampler sees >= 1 s under the same load
        t_busy = time.time()
        while time.time() - t_busy < 1.0:
            for i in range(50):
                nlps[i % R].launch(K_JAC_HESS)
            torch.cuda.synchronize()
        t_end = time.time()
    clocks = sampler.stop(t_start, t_end) if sampler else None

    tms = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms.item())
    ms_per_step = ms / args.steps
    value = B_total * T / (ms_per_step * 1e-3)

    # ---- end to end through the public host API, pinned host buffers
    n = nlps[0]
    z, lam, sigma, w = host[0]
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    zp, lp, sp_ = pin(z), pin(lam), pin(sigma)
    Jp = torch.empty((B, n.num_jacobian), dtype=torch.float64).pin_memory().numpy()
    Hp = torch.empty((B, n.num_hessian), dtype=torch.float64).pin_memory().numpy()
    e2e_steps = max(3, min(args.steps, 20))
    for _ in range(2):
        n.eval_jacobian_hessian(Jp, Hp, zp, sp_, lp)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        n.eval_jacobian_hessian(Jp, Hp, zp, sp_, lp)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tdt = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
    dt = float(tdt.item())
    e2e_value = B_total * T * e2e_steps / dt
    h2d = 8 * B * (n.num_variables + n.num_constraint + 1)
    d2h = 8 * B * (n.num_jacobian + n.num_hessian)

    # ---- secondary: device-resident KKT consumer (30 MB instead of 99 MB back over PCIe), at every N
    kkt = None
    if not args.no_kkt:
        peak, _ = _peaks()
        kkt = bench_kkt(torch, n, stream, zp, lp, sp_, peak)
        tk = torch.tensor([kkt["ms_kkt_kernels"], kkt["ms_step_callbacks_plus_kkt"], kkt["e2e_ms_host_z_lambda_to_host_solution"]],
                          dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tk, op=dist.ReduceOp.MAX)
        kkt["ms_kkt_kernels"], kkt["ms_step_callbacks_plus_kkt"], kkt["e2e_ms_host_z_lambda_to_host_solution"] = [float(x) for x in tk.tolist()]
        kkt["kkt_solves_per_s"] = B_total / (kkt["ms_kkt_kernels"] * 1e-3)
        kkt["newton_steps_per_s"] = B_total / (kkt["ms_step_callbacks_plus_kkt"] * 1e-3)
        kkt["e2e_newton_steps_per_s"] = B_total / (kkt["e2e_ms_host_z_lambda_to_host_solution"] * 1e-3)
        kkt["e2e_knot_evals_per_s"] = B_total * T / (kkt["e2e_ms_host_z_lambda_to_host_solution"] * 1e-3)
        kkt["n_gpus"] = world
        kkt["timing"] = "max over ranks"

    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.cpu().numpy())

    line = None
    if rank == 0:
        peak, peak_src = _peaks()
        bytes_per_launch = n.algorithmic_bytes_per_problem() * B
        achieved = bytes_per_launch / (ms_per_step * 1e-3) / 1e9
        ncu = _ncu_headline()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": (f"cartpole swing-up T={T}, B={args.batch} per GPU, fused Jacobian+Hessian callbacks" if not strong else
                                    f"cartpole swing-up T={T}, B={args.batch} in total over {world} GPUs, fused Jacobian+Hessian callbacks"),
                       "l2": f"{R} rotating input/output sets ({R * bytes_per_launch / 1e6:.0f} MB) > 126 MB L2",
                       "parallelism": f"{world} independent shards, no collective",
                       "host_binding": binding},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": 1e3 * dt / e2e_steps,
                    "pcie_gbs_per_gpu": (h2d + d2h) / (dt / e2e_steps) / 1e9},
            "gpu_launches": int(n1 - n0),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (ncu.get("traffic") or {}).get("dram_bytes_per_launch"), "peak_source": peak_src,
                         "traffic_source": (ncu.get("traffic") or {}).get("source"),
                         "algorithmic_bytes_per_launch": bytes_per_launch},
        }
        f64 = ncu.get("fp64")
        if f64:
            # FP64 pipe: executed DFMA/DMUL/DADD per knot from the committed ncu capture of the shipped kernel x the
            # knots of this run / the live kernel time, against the measured DFMA issue peak; next to it the
            # pipe-utilisation counter ncu itself reported for that capture
            fp = _fp64_peak()
            rate = f64["sass_fp64_thread_instructions_per_knot"] * B * T / (ms_per_step * 1e-3)
            line["fp64"] = {"sass_fp64_per_knot": f64["sass_fp64_thread_instructions_per_knot"], "mix_per_knot": f64["mix_per_knot"],
                            "achieved_ginst": rate / 1e9, "peak_ginst": fp / 1e9, "frac_of_fp64_issue_peak": rate / fp,
                            "ncu_pipe_fp64_pct": f64["ncu_pipe_fp64_pct"], "source": f64["source"]}
        if kkt is not None:
            line["kkt"] = kkt
        if world == 1 and not args.no_solve:
            # secondary (BASELINE config 3): acrobot T=101 x 4096 FULL SOLVES on the device (lock-step Newton-KKT
            # solver over the same callbacks + KKT kernels); Ipopt is absent, so this is this repository's solver
            try:
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import solve_config3
                for n_ in nlps:
                    n_.close()
                # the shipped solver is the native arm (dto_sqp_solve; host z0 in, host results out inside its timed
                # region); the torch-glued arm of the same algorithm (sqp.py) is reported beside it
                line["solve"] = solve_config3.run(B=4096, T=101, max_iter=300, method="native")
                t_arm = solve_config3.run(B=4096, T=101, max_iter=300, method="sqp")
                line["solve"]["torch_glue_arm"] = {k: t_arm[k] for k in ("seconds", "solves_per_s", "accepted_frac", "gpu_launches")}
                # the reference's cartpole example (BASELINE config 2's model, |u| <= 3 as bounds, its rollout guess): interior-point
                # mode of the torch-glued arm, 4096 problems (64 distinct guesses)
                import ip_cartpole
                cp = ip_cartpole.run(3.0, 4096, 600, guess="rollout", distinct=64)
                line["solve"]["cartpole_example_with_bounds"] = {k: cp[k] for k in ("seconds", "solves_per_s", "converged", "it_median", "it_max", "cv_max",
                                                                                        "u_max", "at_bound", "end_error_max")}
            except Exception as e:  # noqa: BLE001
                line["solve"] = {"error": str(e)[:200]}
        if world == 1 and not args.no_cpu:
            co, mo = build_c_baseline(T)
            try:
                os.sched_setaffinity(0, range(os.cpu_count() or 1))  # the CPU baseline uses every host core again
            except OSError:
                pass
            threads = host_threads()
            v, Bs, reps, dtc = time_cpu(co, z, lam, sigma, w, threads)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": f"{Bs} of {B} problems x T={T}, {reps} passes, {dtc:.1f} s, oracle C twin (no-CSE "
                                              "element code, reference loop structure), gcc -O2 -fopenmp"}
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if line is not None:
        print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 200; 5 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed steps before them (default 10; 1 with --impl reference)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=4096)
    ap.add_argument("--T", type=int, default=101)
    ap.add_argument("--ref-sample", type=int, default=0, dest="ref_sample", help="problems per step of the reference arm (0 = the whole batch)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="weak: --batch problems per GPU; strong: --batch problems in total, split over the GPUs")
    ap.add_argument("--no-bind", action="store_true", dest="no_bind", help="do not bind the process to the GPU-local host cores")
    ap.add_argument("--no-cpu", action="store_true", dest="no_cpu")
    ap.add_argument("--no-kkt", action="store_true", dest="no_kkt")
    ap.add_argument("--no-solve", action="store_true", dest="no_solve")
    ap.add_argument("--dump-outputs", default=None, dest="dump_outputs", metavar="DIR",
                    help="write J and H of the last timed step (sampled problems) as DIR/<name>.npy")
    args = ap.parse_args()
    reference = args.impl == "reference"
    if args.steps is None:
        args.steps = 5 if reference else 200
    if args.warmup is None:
        args.warmup = 1 if reference else 10
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if reference and args.dump_outputs:
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl ours")
    with tempfile.TemporaryDirectory(prefix="dto_bench_") as cache:
        os.environ.setdefault("DTO_CACHE_DIR", cache)
        return run_reference(args) if reference else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())

"""Device-timed fused Jacobian+Hessian pass over a list of (model, T, B): config-5 style size sweep, one JSON
line per case.   python tools/size_sweep.py cartpole:T=101:4096 cartpole:T=101:65536 ...

    python tools/size_sweep.py --rounds cartpole:T=101

splits the launch time into a fixed cost per launch and a cost per round of tiles. It times the batches that give
k = 2 ... 16 full rounds of 32-item tiles over all compute warps, B = floor(SMs * 8 * 32 * k / T), plus B = 4096.
Each batch is timed back to back (as above) and isolated (one launch between two device synchronisations, median
of 60), and `t = a + b * k` is fitted to both columns: `a` is the fixed cost per launch, `b` the time per round.
The difference of the two intercepts is what overlapping consecutive launches hides. The isolated start event is
recorded before the host enqueues the kernel, so its intercept includes the launch call's host latency. The k axis
assumes 32-item tiles, the tile of models without a Hessian halo (cartpole); a model with a halo has 31-item tiles,
so its rounds are ragged. The first line of this mode names the card, its power limit and its maximum SM clock."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import dto_b200 as D  # noqa: E402
from dto_b200.evaluator import K_JAC_HESS  # noqa: E402
from examples import models as M  # noqa: E402
from util import make_inputs  # noqa: E402

COMPUTE_WARPS = 8  # must equal DTO_WS_COMPUTE (csrc/dto_kernel_ws.cuh): compute warps per CTA, one CTA per SM
ISOLATED = 60


def parse(spec: str):
    parts = spec.split(":")
    name, kw = parts[0], {}
    for kv in parts[1].split(","):
        if kv:
            k, v = kv.split("=")
            kw[k] = int(v) if v.isdigit() else v
    return name, kw, [int(b) for b in parts[2:]]


def batches(name, kw, B):
    """R rotating batches of seeded inputs on one stream (3 while they fit: no launch finds its inputs in L2)."""
    model = M.BUILDERS[name](D, **kw)
    n0 = D.solver_from(model, batch=B).nlp
    byt = n0.algorithmic_bytes_per_problem() * B
    R = 3 if byt < 4e9 else 1
    nl = [n0] + [n0.new_batch() for _ in range(R - 1)]
    st = torch.cuda.Stream()
    for i, n in enumerate(nl):
        z, lam, sig, w = make_inputs(name, model, n.num_variables, n.num_constraint, n.num_parameter, B, 2, i)
        if n.num_parameter:
            n.set_parameters(w)
        n.set_x(z)
        n.set_duals(sig, lam)
        n.set_stream(st.cuda_stream)
    return nl, st, byt


def back_to_back(nl, st, steps):
    """ms per launch over `steps` launches enqueued back to back on one stream"""
    R = len(nl)
    with torch.cuda.stream(st):
        for i in range(5):
            nl[i % R].launch(K_JAC_HESS)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for i in range(steps):
            nl[i % R].launch(K_JAC_HESS)
        e1.record(st)
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def isolated(nl, st, reps=ISOLATED):
    """median ms of one launch with nothing before or after it on the device"""
    R = len(nl)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    with torch.cuda.stream(st):
        for i, (e0, e1) in enumerate(ev):
            torch.cuda.synchronize()
            e0.record(st)
            nl[i % R].launch(K_JAC_HESS)
            e1.record(st)
            torch.cuda.synchronize()
    return float(np.median([e0.elapsed_time(e1) for e0, e1 in ev]))


def fit(k, t):
    """least-squares t = a + b k: (a, b, standard error of a, standard error of b)"""
    (b, a), cov = np.polyfit(np.asarray(k, float), np.asarray(t, float), 1, cov=True)
    return float(a), float(b), float(np.sqrt(cov[1, 1])), float(np.sqrt(cov[0, 0]))


def gpu_line():
    dev = torch.cuda.current_device()
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"nvidia-smi unavailable: {e}"
    return {"gpu": q, "torch_name": torch.cuda.get_device_name(dev), "sms": torch.cuda.get_device_properties(dev).multi_processor_count}


def rounds(spec):
    name, kw, _ = parse(spec)
    T = kw["T"]
    sms = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    per_round = sms * COMPUTE_WARPS * 32  # knots per round of tiles
    rows = []
    for B in sorted({per_round * k // T for k in range(2, 17)} | {4096}):
        nl, st, byt = batches(name, kw, B)
        steps = max(200, min(2000, int(1e11 / byt)))
        row = {"model": name, **kw, "B": B, "k": B * T / per_round, "ms_back_to_back": back_to_back(nl, st, steps),
               "ms_isolated": isolated(nl, st), "steps": steps, "isolated_reps": ISOLATED}
        print(json.dumps(row), flush=True)
        rows.append(row)
        for n in nl:
            n.close()
    k = [r["k"] for r in rows]
    out = {"model": name, **kw, "fit": "t_us = a + b * k over k = 2..16 and B = 4096",
           "note": "isolated times include the host latency of the launch call"}
    for col in ("back_to_back", "isolated"):
        a, b, sa, sb = fit(k, [1e3 * r["ms_" + col] for r in rows])
        out[col] = {"a_us": a, "b_us": b, "a_err_us": sa, "b_err_us": sb}
    out["hidden_by_overlap_us"] = out["isolated"]["a_us"] - out["back_to_back"]["a_us"]
    print(json.dumps(out), flush=True)


def sizes(spec):
    name, kw, Bs = parse(spec)
    for B in Bs:
        nl, st, byt = batches(name, kw, B)
        steps = max(5, min(200, int(2e11 / byt)))
        ms = back_to_back(nl, st, steps)
        print(json.dumps({"model": name, **kw, "B": B, "ms": ms, "GBs": byt / ms / 1e6, "frac_hbm": byt / ms / 1e6 / 6549.4,
                          "evals_per_s": B * nl[0].T / ms * 1e3, "steps": steps}), flush=True)
        for n in nl:
            n.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("specs", nargs="*", help="model:kw=v,...:B[:B...] (with --rounds: model:T=..,...)")
    ap.add_argument("--rounds", action="store_true", help="fixed cost and cost per round of tiles, back to back and isolated")
    args = ap.parse_args()
    if args.rounds:
        print(json.dumps(gpu_line()), flush=True)
    for spec in args.specs:
        (rounds if args.rounds else sizes)(spec)


if __name__ == "__main__":
    main()

"""GPU tuning sweep for the fused Jacobian+Hessian kernel (cartpole T=101, B=4096).
Builds one model library per DTO_TUNE setting (run once on the CPU box with --build-only so the
.so files ship with gpurun) and times each on the device with rotating buffers."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TUNES = ["", "ws=0,persist=0", "ws=0", "ws_all=1", "ws_plan=0", "bf=0,emit=0", "ws_helpers=4"]   # codegen.TUNE_VALUES

CHILD = r"""
import sys, os, json, time
sys.path.insert(0, %r); sys.path.insert(0, os.path.join(%r, 'tests'))
import numpy as np
import dto_b200 as D
from dto_b200.evaluator import K_JAC_HESS
from examples import models as M
from util import make_inputs
build_only = %r
KID = %d
model = M.BUILDERS[%r](D, **%r)
s = D.solver_from(model, batch=%d, verbose=build_only)
if build_only: sys.exit(0)
import torch
n0 = s.nlp
nl = [n0, n0.new_batch(), n0.new_batch()]
st = torch.cuda.Stream()
for i, n in enumerate(nl):
    z, lam, sig, w = make_inputs(%r, model, n.num_variables, n.num_constraint, n.num_parameter, n.batch, 2, i)
    if n.num_parameter: n.set_parameters(w)
    n.set_x(z); n.set_duals(sig, lam); n.set_stream(st.cuda_stream)
with torch.cuda.stream(st):
    for i in range(10): nl[i %% 3].launch(KID)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for i in range(200): nl[i %% 3].launch(KID)
    e1.record(st); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / 200
byt = n0.algorithmic_bytes_per_problem() * n0.batch
print(json.dumps({"tune": os.environ.get("DTO_TUNE", ""), "deriv": os.environ.get("DTO_DERIV", ""), "kernel": KID, "model": %r, "ms": ms, "GBs": byt / ms / 1e6,
                  "evals_per_s": n0.batch * n0.T / ms * 1e3, "smem": n0.kernel_smem_bytes(KID)}))
"""


def main():
    build_only = "--build-only" in sys.argv
    model, kw, B = "cartpole", dict(T=101), 4096
    for a in sys.argv[1:]:
        if a.startswith("--model="):  # e.g. --model=car:T=201,obstacle=general:16384
            parts = a.split("=", 1)[1].split(":")
            model = parts[0]
            kw = {}
            if len(parts) > 1 and parts[1]:
                for kv in parts[1].split(","):
                    k, v = kv.split("=")
                    kw[k] = int(v) if v.isdigit() else v
            if len(parts) > 2:
                B = int(parts[2])
    tunes = TUNES
    kid = 5
    for a in sys.argv[1:]:
        if a.startswith("--kernel="):
            kid = int(a.split("=", 1)[1])
    for a in sys.argv[1:]:
        if a.startswith("--tunes="):
            tunes = a.split("=", 1)[1].split(";")
    for t in tunes:
        # "DERIV=dag|bf=1,emit=2": derivative mode (DTO_DERIV) in front of the DTO_TUNE string
        env = dict(os.environ)
        if "|" in t:
            pre, t = t.split("|", 1)
            for kv in pre.split(","):
                k, v = kv.split("=")
                env["DTO_" + k] = v
        env["DTO_TUNE"] = t
        code = CHILD % (ROOT, ROOT, build_only, kid, model, kw, B, model, model + repr(kw))
        r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True)
        out = (r.stdout.strip().splitlines() or [""])[-1]
        print(out if r.returncode == 0 else f"FAILED {t}: {r.stderr[-500:]}", flush=True)


if __name__ == "__main__":
    main()

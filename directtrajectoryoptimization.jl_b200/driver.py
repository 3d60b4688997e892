"""Lock-step batched solve driver (SURVEY 8f row N1): B independent NLP solvers, one per problem of a
batch, whose MOI callbacks rendezvous into ONE batched GPU call per callback kind.

Reference wiring being replaced: /root/reference/src/data.jl:222-255 (`SolverData`: one
`Ipopt.Optimizer` owning one `NLPData` evaluator) and /root/reference/src/solver.jl:45-47 (`solve!`).
There every callback of the one optimizer runs the per-knot CPU closures; here B optimizers run as
cooperative tasks, each task's callback parks its `(z, sigma, lambda)` in row b of the batch arrays and
blocks, and when every live task is parked the last one to arrive flushes: one `eval_*` of the batched
evaluator per callback kind that is waiting, then everybody resumes with its own row of the result.

Ipopt (libipopt / Ipopt.jl) is NOT available in this image, so the per-problem solver that plays the
caller is SciPy's interior-point / SQP `trust-constr` -- same callback set (objective, gradient,
constraint residuals, sparse Jacobian, sparse Hessian of the Lagrangian with the reference's fixed
sparsity structures, variable and constraint bounds). The broker does not know which solver sits above
it: an Ipopt task calls the same five entry points. Iterates are therefore comparable between two
*evaluators* under the same solver (tests: CPU oracle vs GPU), not against Ipopt's.

Nothing here evaluates model numerics: every number comes from the evaluator handed in (the product
passes `BatchedNLPData`, i.e. libdto.so's CUDA kernels).
"""
from __future__ import annotations

import threading
from typing import Callable, List, Optional

import numpy as np

KINDS = ("f", "g", "c", "J", "H")


class CallbackBroker:
    """Rendezvous of per-problem callbacks into batched evaluations.

    `nlp` needs: batch, num_variables, num_constraint, num_jacobian, num_hessian, and the batched
    eval_objective(Z) -> f[B], eval_objective_gradient(G, Z), eval_constraint(C, Z),
    eval_constraint_jacobian(J, Z), eval_hessian_lagrangian(H, Z, sigma[B], lam[B, N_c])."""

    def __init__(self, nlp, z0: np.ndarray):
        self.nlp = nlp
        B = nlp.batch
        self.Z = np.ascontiguousarray(z0, dtype=np.float64).reshape(B, nlp.num_variables).copy()
        self.SIG = np.ones(B)
        self.LAM = np.zeros((B, nlp.num_constraint))
        self.out = {"f": np.zeros(B), "g": np.zeros((B, nlp.num_variables)), "c": np.zeros((B, nlp.num_constraint)),
                    "J": np.zeros((B, nlp.num_jacobian)), "H": np.zeros((B, nlp.num_hessian))}
        self.cv = threading.Condition()
        self.live = set(range(B))
        self.waiting = {}            # problem -> kind
        self.generation = 0
        self.flushes = 0
        self.batched_calls = {k: 0 for k in KINDS}
        self.requests = {k: 0 for k in KINDS}
        self.error: Optional[BaseException] = None

    # ---- called by the last task to park (holds the lock)
    def _flush(self) -> None:
        kinds = sorted(set(self.waiting.values()), key=KINDS.index)
        try:
            for k in kinds:
                if k == "f":
                    self.out["f"][:] = self.nlp.eval_objective(self.Z)
                elif k == "g":
                    self.nlp.eval_objective_gradient(self.out["g"], self.Z)
                elif k == "c":
                    self.nlp.eval_constraint(self.out["c"], self.Z)
                elif k == "J":
                    self.nlp.eval_constraint_jacobian(self.out["J"], self.Z)
                else:
                    self.nlp.eval_hessian_lagrangian(self.out["H"], self.Z, self.SIG, self.LAM)
                self.batched_calls[k] += 1
        except BaseException as e:  # noqa: BLE001 -- propagate to every task
            self.error = e
        self.flushes += 1
        self.waiting.clear()
        self.generation += 1
        self.cv.notify_all()

    def request(self, b: int, kind: str, z, sigma: float = 1.0, lam=None) -> np.ndarray:
        """Callback of problem b: parks (z, sigma, lam), returns problem b's row of the batched result."""
        with self.cv:
            if self.error is not None:
                raise RuntimeError("batched evaluation failed") from self.error
            self.Z[b] = z
            if kind == "H":
                self.SIG[b] = sigma
                self.LAM[b] = 0.0 if lam is None else lam
            self.waiting[b] = kind
            self.requests[kind] += 1
            gen = self.generation
            if len(self.waiting) == len(self.live):
                self._flush()
            else:
                while self.generation == gen:
                    self.cv.wait()
            if self.error is not None:
                raise RuntimeError("batched evaluation failed") from self.error
            r = self.out[kind][b]
            return float(r) if kind == "f" else np.array(r, copy=True)

    def finish(self, b: int) -> None:
        """Problem b's solver has terminated: the others stop waiting for it."""
        with self.cv:
            self.live.discard(b)
            if self.live and len(self.waiting) == len(self.live):
                self._flush()


def _scipy_task(broker: CallbackBroker, b: int, z0, structures, bounds, options, record: Optional[list]):
    """One problem under SciPy's trust-constr (the stand-in for one Ipopt.Optimizer, src/data.jl:237-251)."""
    import scipy.sparse as sp
    from scipy.optimize import Bounds, NonlinearConstraint, minimize

    (jr, jc), (hr, hc), nz, nc, use_hessian = structures
    (zl, zu), (cl, cu) = bounds
    if not use_hessian:
        # features_available without :Hess (src/moi.jl:122): the reference lets Ipopt fall back to its
        # limited-memory quasi-Newton approximation; the stand-in solver does the same with BFGS updates
        from scipy.optimize import BFGS

    def fun(z):
        return broker.request(b, "f", z)

    def grad(z):
        return broker.request(b, "g", z)

    def hess_obj(z):  # sigma * Hessian of the objective: the Lagrangian callback with lambda = 0
        v = broker.request(b, "H", z, 1.0, None)
        return sp.csr_matrix((v, (hr, hc)), shape=(nz, nz))

    cons = []
    if nc:
        def con(z):
            return broker.request(b, "c", z)

        def jac(z):
            return sp.csr_matrix((broker.request(b, "J", z), (jr, jc)), shape=(nc, nz))

        def hess_con(z, v):  # sum_i v_i Hessian(c_i): the Lagrangian callback with sigma = 0
            return sp.csr_matrix((broker.request(b, "H", z, 0.0, v), (hr, hc)), shape=(nz, nz))

        cons = [NonlinearConstraint(con, cl, cu, jac=jac, hess=hess_con if use_hessian else BFGS())]
    kw = {}
    if np.isfinite(zl).any() or np.isfinite(zu).any():
        kw["bounds"] = Bounds(zl, zu)
    cb = None
    if record is not None:
        def cb(xk, state=None):  # noqa: ANN001
            record.append(np.array(xk, copy=True))
            return False
    try:
        return minimize(fun, z0, jac=grad, hess=hess_obj if use_hessian else BFGS(), constraints=cons, method="trust-constr", options=options,
                        callback=cb, **kw)
    finally:
        broker.finish(b)


def solve_batch(nlp, z0: np.ndarray, options: Optional[dict] = None, record_iterates: bool = False,
                task: Callable = _scipy_task):
    """solve! for every problem of the batch: B solver tasks in lock step over one batched evaluator.
    Returns (Z[B, N_z] final iterates, list of per-problem solver results, broker, iterates or None)."""
    B = nlp.batch
    jr, jc = nlp.jacobian_structure_arrays()
    use_hessian = bool(getattr(nlp, "hessian_lagrangian", True))
    if use_hessian:
        hr, hc = nlp.hessian_lagrangian_structure_arrays()
    else:
        hr = hc = np.ones(0, dtype=np.int64)
    structures = ((jr - 1, jc - 1), (hr - 1, hc - 1), nlp.num_variables, nlp.num_constraint, use_hessian)
    # every problem's own variable bounds: [B, N_z] rows when the batch has per-problem values, else the shared pair
    lo, up = (np.asarray(v, dtype=np.float64) for v in getattr(nlp, "batch_variable_bounds", nlp.variable_bounds))
    cbounds = nlp.constraint_bounds
    bounds_of = (lambda b: ((lo[b], up[b]), cbounds)) if lo.ndim == 2 else (lambda b: ((lo, up), cbounds))
    opts = {"gtol": 1e-8, "xtol": 1e-10, "maxiter": 1000, "verbose": 0}
    opts.update(options or {})
    z0 = np.asarray(z0, dtype=np.float64).reshape(B, nlp.num_variables)
    broker = CallbackBroker(nlp, z0)
    results: List = [None] * B
    errors: List = [None] * B
    iterates = [[] for _ in range(B)] if record_iterates else None

    def run(b):
        try:
            results[b] = task(broker, b, z0[b].copy(), structures, bounds_of(b), opts, iterates[b] if iterates is not None else None)
        except BaseException as e:  # noqa: BLE001
            errors[b] = e

    threads = [threading.Thread(target=run, args=(b,), daemon=True) for b in range(B)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for e in errors:
        if e is not None:
            raise e
    Z = np.stack([np.asarray(r.x, dtype=np.float64) for r in results])
    return Z, results, broker, iterates

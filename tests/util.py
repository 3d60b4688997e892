"""Shared test helpers: seeded inputs (SURVEY 8d), oracle batch evaluation, comparisons."""
from __future__ import annotations

import math

import numpy as np

from examples import models as M
from oracle import api as O

RTOL, ATOL = 1e-12, 1e-14   # BASELINE.json north_star: 1e-12 relative or 1e-14 absolute

# DTO_TUNE kernel-selection variants the GPU tests compare against the default build (test_gpu_properties.py); build()
# compiles their model libraries ahead of the tests
KERNEL_VARIANTS = ["ws=0,persist=0", "ws=0", "ws_all=1", "ws_plan=0", "bf=0,emit=0", "ws_helpers=4"]


def rng_for(config: int, shard: int = 0):
    return np.random.default_rng(20261017 + 1000 * config + shard)


def make_inputs(name: str, model: dict, nz: int, nc: int, nw: int, B: int, config: int = 0, shard: int = 0):
    """z, lambda, sigma, w per SURVEY 8(d)."""
    r = rng_for(config, shard)
    T, n, m = model["T"], model["n"], model["m"]
    z = np.empty((B, nz))
    if name == "cartpole":
        X = np.concatenate([r.uniform(-math.pi, math.pi, (B, T, 2)), r.normal(0, 1, (B, T, 2))], axis=2)
        U = r.uniform(-3, 3, (B, T, m))
    elif name == "acrobot":
        X = np.concatenate([r.uniform(-math.pi, math.pi, (B, T, 2)), r.normal(0, 1, (B, T, 2))], axis=2)
        U = r.uniform(-3, 3, (B, T, m))
    elif name == "car":
        X = np.concatenate([r.uniform(0, 1, (B, T, 2)), r.uniform(-math.pi, math.pi, (B, T, 1))], axis=2)
        U = r.uniform(-0.5, 0.5, (B, T, m))
    elif name == "piecewise":  # both branches of every ifelse get exercised
        X = r.uniform(-1.5, 1.5, (B, T, n))
        U = r.uniform(-1.5, 1.5, (B, T, m))
    else:
        X = r.uniform(0, 1, (B, T, n))
        U = r.uniform(0, 1, (B, T, m))
    for t in range(T):
        o = t * (n + m)
        z[:, o:o + n] = X[:, t]
        if t < T - 1:
            z[:, o + n:o + n + m] = U[:, t]
    lam = r.normal(0, 1, (B, nc)) if name in ("cartpole", "acrobot", "car") else r.uniform(0, 1, (B, nc))
    sigma = np.ones(B)
    if B > 1:
        sigma[1::2] = 0.37
    w = np.zeros((B, nw))
    if nw == 8:  # cartpole: w = [x1; xT]
        w[:, 0:4] = r.normal(0, 0.1, (B, 4))
        w[:, 4:8] = np.array([0.0, math.pi, 0.0, 0.0]) + r.normal(0, 0.1, (B, 4))
    elif nw > 0:
        w[:] = r.normal(0, 1, (B, nw))
    return z, lam, sigma, w


def oracle_parameters(model: dict, w_row: np.ndarray):
    """Per-knot parameter list for ONE problem from its flat row (reference: T+1 vectors, Q10)."""
    T = model["T"]
    if model.get("shared_parameters"):
        return [w_row.copy() for _ in range(T)] + [np.zeros(0)]
    return None


def oracle_eval_all(osolver, model, z, lam, sigma, w, hessian=True):
    """Run the five callbacks of the CPU oracle problem by problem."""
    nlp = osolver.nlp
    B = z.shape[0]
    out = dict(f=np.zeros(B), g=np.zeros((B, nlp.num_variables)), c=np.zeros((B, nlp.num_constraint)),
               J=np.zeros((B, nlp.num_jacobian)), H=np.zeros((B, len(nlp.hessian_lagrangian_sparsity))))
    for b in range(B):
        p = oracle_parameters(model, w[b])
        if p is not None:
            osolver.set_parameters(p)
        out["f"][b] = nlp.eval_objective(z[b])
        nlp.eval_objective_gradient(out["g"][b], z[b])
        nlp.eval_constraint(out["c"][b], z[b])
        nlp.eval_constraint_jacobian(out["J"][b], z[b])
        if hessian:
            nlp.eval_hessian_lagrangian(out["H"][b], z[b], float(sigma[b]), lam[b])
    return out


def assert_close(name, got, ref, rtol=RTOL, atol=ATOL):
    got, ref = np.asarray(got), np.asarray(ref)
    assert got.shape == ref.shape, f"{name}: shape {got.shape} vs {ref.shape}"
    err = np.abs(got - ref)
    ok = (err <= atol) | (err <= rtol * np.abs(ref))
    if not ok.all():
        idx = np.argwhere(~ok)
        i = tuple(idx[0])
        worst = np.nanmax(np.where(np.abs(ref) > 0, err / np.maximum(np.abs(ref), 1e-300), 0))
        raise AssertionError(f"{name}: {len(idx)} of {got.size} values differ beyond rtol={rtol}/atol={atol}; "
                             f"first at {i}: got {got[i]!r} ref {ref[i]!r}; worst rel {worst:.3e}")


class OracleBatch:
    """The CPU oracle behind the batched evaluator interface (B problems evaluated one by one): the
    reference arm for driver tests -- same solver above, oracle callbacks below."""

    def __init__(self, osolver, batch: int):
        self.o = osolver.nlp
        self.batch = batch
        self.num_variables = self.o.num_variables
        self.num_constraint = self.o.num_constraint
        self.num_jacobian = self.o.num_jacobian
        self.num_hessian = len(self.o.hessian_lagrangian_sparsity)
        self.variable_bounds = self.o.variable_bounds
        self.constraint_bounds = self.o.constraint_bounds
        self.hessian_lagrangian = bool(getattr(self.o, "hessian_lagrangian", True))

    def jacobian_structure_arrays(self):
        s = self.o.jacobian_structure()
        return np.array([i for i, _ in s], dtype=np.int64), np.array([j for _, j in s], dtype=np.int64)

    def hessian_lagrangian_structure_arrays(self):
        s = self.o.hessian_lagrangian_structure()
        return np.array([i for i, _ in s], dtype=np.int64), np.array([j for _, j in s], dtype=np.int64)

    def eval_objective(self, Z):
        return np.array([self.o.eval_objective(Z[b]) for b in range(self.batch)])

    def eval_objective_gradient(self, G, Z):
        for b in range(self.batch):
            self.o.eval_objective_gradient(G[b], Z[b])

    def eval_constraint(self, Cv, Z):
        for b in range(self.batch):
            self.o.eval_constraint(Cv[b], Z[b])

    def eval_constraint_jacobian(self, J, Z):
        for b in range(self.batch):
            self.o.eval_constraint_jacobian(J[b], Z[b])

    def eval_hessian_lagrangian(self, H, Z, sigma, lam):
        for b in range(self.batch):
            self.o.eval_hessian_lagrangian(H[b], Z[b], float(sigma[b]), lam[b])

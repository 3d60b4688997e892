"""Batched MOI evaluator + Solver: the host-side mirror of the reference's NLPData / Solver
(/root/reference/src/data.jl:106-121,150-220, src/moi.jl:1-125, src/solver.jl:1-47) on top of
the C ABI of libdto.so. Method names, argument order and in-place output conventions follow
the reference's MOI methods; the only addition is the leading batch dimension.

    solver = Solver(dynamics, objective, constraints, bounds; evaluate_hessian, general_constraint,
                    parameters, batch=B, devices=[0..])
    nlp = solver.nlp
    nlp.eval_objective(z)                         -> f[B]
    nlp.eval_objective_gradient(g, z)             g[B, N_z]   in place
    nlp.eval_constraint(c, z)                     c[B, N_c]
    nlp.eval_constraint_jacobian(J, z)            J[B, nnz_J]
    nlp.eval_hessian_lagrangian(H, z, sigma, lam) H[B, nnz_H]
    nlp.jacobian_structure() / nlp.hessian_lagrangian_structure()

x, lambda, sigma, parameters stay device-resident between calls; pass z=None to reuse the
resident iterate (MOI has no new_x flag). All numerics run in the CUDA model library; this
module raises if the native pieces or a GPU are missing.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import _lib
from .codegen import ModelSpec, build_model
from .elements import Bound, Constraint, Cost, Dynamics, GeneralConstraint

K_OBJECTIVE, K_GRADIENT, K_CONSTRAINT, K_JACOBIAN, K_HESSIAN, K_JAC_HESS = range(6)
A_Z, A_LAMBDA, A_SIGMA, A_W, A_F, A_G, A_C, A_J, A_H = range(9)


def _i32(a) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(a, dtype=np.int32))


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _f64(a, shape, name) -> np.ndarray:
    a = np.asarray(a)
    if a.dtype != np.float64 or not a.flags.c_contiguous:
        a = np.ascontiguousarray(a, dtype=np.float64)
    if a.size != int(np.prod(shape)):
        raise ValueError(f"{name}: expected {shape} ({int(np.prod(shape))} values), got shape {a.shape}")
    return a


def _out(a, shape, name) -> np.ndarray:
    if not isinstance(a, np.ndarray) or a.dtype != np.float64 or not a.flags.c_contiguous:
        raise TypeError(f"{name} must be a C-contiguous float64 numpy array (it is written in place)")
    if a.size != int(np.prod(shape)):
        raise ValueError(f"{name}: expected {shape} ({int(np.prod(shape))} values), got shape {a.shape}")
    return a


class Model:
    """A compiled + loaded model library."""

    def __init__(self, spec: ModelSpec, verbose: bool = False):
        self.spec = spec
        self.path = build_model(spec, verbose=verbose)
        L = _lib.lib()
        h = C.c_void_p()
        _lib.check(L.dto_model_load(self.path.encode(), C.byref(h)))
        self.handle = h

    @property
    def name(self) -> str:
        return _lib.lib().dto_model_name(self.handle).decode()


class BatchedNLPData:
    """NLPData for B problems of one shape. Host-only queries (sizes, structures, bounds) work
    without a GPU; evaluation creates the device batch on first use."""

    def __init__(self, model: Model, T: int, dynamics_kind, cost_kind, stage_kind, use_general: bool,
                 parameter_dim, parameter_offset, num_parameter: int, evaluate_hessian: bool, bounds, batch: int,
                 devices: Optional[Sequence[int]]):
        L = _lib.lib()
        self.model = model
        self.T = T
        self.batch = int(batch)
        self.devices = list(devices) if devices is not None else None
        self.hessian_lagrangian = bool(evaluate_hessian)
        self.use_general = bool(use_general)
        self._keep = [_i32(dynamics_kind), _i32(cost_kind), _i32(stage_kind), _i32(parameter_dim),
                      _i32(parameter_offset) if parameter_offset is not None else None]
        ip = C.POINTER(C.c_int32)
        desc = _lib.ShapeDesc(
            T=T,
            dynamics_kind=self._keep[0].ctypes.data_as(ip),
            cost_kind=self._keep[1].ctypes.data_as(ip),
            stage_kind=self._keep[2].ctypes.data_as(ip),
            use_general=int(use_general),
            parameter_dim=self._keep[3].ctypes.data_as(ip),
            parameter_offset=self._keep[4].ctypes.data_as(ip) if self._keep[4] is not None else None,
            num_parameter=int(num_parameter),
        )
        h = C.c_void_p()
        _lib.check(L.dto_shape_create(model.handle, C.byref(desc), C.byref(h)))
        self.shape = h
        self.num_variables = int(L.dto_num_variables(h))
        self.num_constraint = int(L.dto_num_constraint(h))
        self.num_jacobian = int(L.dto_num_jacobian(h))
        self.num_hessian = int(L.dto_num_hessian(h))
        self.num_hessian_lagrangian = int(L.dto_num_hessian_nonunique(h))  # reference field (Q4)
        self.num_parameter = int(L.dto_num_parameter(h))
        self._batch = None
        self._bounds = bounds
        self._bounds_host = None        # [lower, upper] of set_variable_bounds, [B, N_z] each

    # ---- structure (host only)
    def jacobian_structure_arrays(self):
        r = np.empty(self.num_jacobian, dtype=np.int64)
        c = np.empty(self.num_jacobian, dtype=np.int64)
        _lib.check(_lib.lib().dto_jacobian_structure(self.shape, r.ctypes.data_as(C.POINTER(C.c_int64)),
                                                     c.ctypes.data_as(C.POINTER(C.c_int64))))
        return r, c

    def hessian_lagrangian_structure_arrays(self):
        r = np.empty(self.num_hessian, dtype=np.int64)
        c = np.empty(self.num_hessian, dtype=np.int64)
        _lib.check(_lib.lib().dto_hessian_lagrangian_structure(self.shape, r.ctypes.data_as(C.POINTER(C.c_int64)),
                                                               c.ctypes.data_as(C.POINTER(C.c_int64))))
        return r, c

    def hessian_block_structure(self):
        """(rows, cols), 1-based, sorted: every entry of one dense block per knot over that knot's variables [x_t; u_t]
        (the last knot: x_T). The H of a KKT system in knot-blocks mode, e.g. the solver's BFGS approximation."""
        n = int(_lib.lib().dto_hessian_block_count(self.shape))
        r = np.empty(n, dtype=np.int64)
        c = np.empty(n, dtype=np.int64)
        _lib.check(_lib.lib().dto_hessian_block_structure(self.shape, r.ctypes.data_as(C.POINTER(C.c_int64)),
                                                          c.ctypes.data_as(C.POINTER(C.c_int64))))
        return r, c

    def hessian_chain_structure(self):
        """(rows, cols), 1-based, sorted: row block t of the knot chain, rows [x_t; u_t] against columns [x_t; u_t; x_{t+1}]
        (the last knot: x_T against x_T), dense row-major. The H of a KKT system in knot-chain mode, e.g. the solver's
        partitioned BFGS approximation (sqp.py `PARTITIONED_BFGS`)."""
        n = int(_lib.lib().dto_hessian_chain_count(self.shape))
        r = np.empty(n, dtype=np.int64)
        c = np.empty(n, dtype=np.int64)
        _lib.check(_lib.lib().dto_hessian_chain_structure(self.shape, r.ctypes.data_as(C.POINTER(C.c_int64)),
                                                          c.ctypes.data_as(C.POINTER(C.c_int64))))
        return r, c

    def jacobian_structure(self):
        """MOI.jacobian_structure (src/moi.jl:124): list of 1-based (row, col)."""
        r, c = self.jacobian_structure_arrays()
        return list(zip(r.tolist(), c.tolist()))

    def hessian_lagrangian_structure(self):
        """MOI.hessian_lagrangian_structure (src/moi.jl:125)."""
        r, c = self.hessian_lagrangian_structure_arrays()
        return list(zip(r.tolist(), c.tolist()))

    def features_available(self):
        """src/moi.jl:122"""
        return ["Grad", "Jac", "Hess"] if self.hessian_lagrangian else ["Grad", "Jac"]

    def initialize(self, features=None):
        """src/moi.jl:123"""
        return None

    @property
    def constraint_bounds(self):
        lo = np.empty(self.num_constraint)
        hi = np.empty(self.num_constraint)
        dp = C.POINTER(C.c_double)
        _lib.check(_lib.lib().dto_constraint_bounds(self.shape, lo.ctypes.data_as(dp), hi.ctypes.data_as(dp)))
        return [lo, hi]

    def knot_layout(self):
        xs, us = np.empty(self.T, np.int64), np.empty(self.T, np.int64)
        nx, nu = np.empty(self.T, np.int32), np.empty(self.T, np.int32)
        _lib.check(_lib.lib().dto_knot_layout(self.shape, xs.ctypes.data_as(C.POINTER(C.c_int64)),
                                              nx.ctypes.data_as(C.POINTER(C.c_int32)),
                                              us.ctypes.data_as(C.POINTER(C.c_int64)),
                                              nu.ctypes.data_as(C.POINTER(C.c_int32))))
        return xs, nx, us, nu

    @property
    def variable_bounds(self):
        """primal_bounds (src/data.jl:123-133) of the Bound objects the batch was built with."""
        return self.primal_bounds(self._bounds)

    def primal_bounds(self, bounds):
        """[lower, upper] ([N_z] each) of a list of T Bound objects, laid out as primal_bounds (src/data.jl:123-133)."""
        lo = np.full(self.num_variables, -np.inf)
        hi = np.full(self.num_variables, np.inf)
        xs, nx, us, nu = self.knot_layout()
        for t, b in enumerate(bounds or []):
            if len(b.state_lower) > 0:
                lo[xs[t] - 1: xs[t] - 1 + nx[t]] = b.state_lower
            if len(b.state_upper) > 0:
                hi[xs[t] - 1: xs[t] - 1 + nx[t]] = b.state_upper
            if len(b.action_lower) > 0:
                lo[us[t] - 1: us[t] - 1 + nu[t]] = b.action_lower
            if len(b.action_upper) > 0:
                hi[us[t] - 1: us[t] - 1 + nu[t]] = b.action_upper
        return [lo, hi]

    def set_variable_bounds(self, lower, upper):
        """Bound values per problem: lower, upper [B, N_z] (row b = problem b's primal_bounds), or None for both to return to
        the Bound objects. The solvers take one bound pattern per batch -- which variables are pinned (lower == upper), which
        have a finite lower and which a finite upper bound -- and every problem's own values; a batch whose rows differ in
        pattern is refused when it is solved. Kept on the host (a solve over several devices hands every shard its rows)."""
        if lower is None and upper is None:
            self._bounds_host = None
            return
        if lower is None or upper is None:
            raise ValueError("set_variable_bounds: lower and upper come together (or both None)")
        shape = (self.batch, self.num_variables)
        lo = np.array(_f64(lower, shape, "lower"), dtype=np.float64, copy=True).reshape(shape)
        up = np.array(_f64(upper, shape, "upper"), dtype=np.float64, copy=True).reshape(shape)
        self._bounds_host = [lo, up]

    @property
    def batch_variable_bounds(self):
        """[lower, upper] as the solvers take them: the [B, N_z] rows of set_variable_bounds, or else the shared [N_z] pair
        of `variable_bounds`."""
        if self._bounds_host is not None:
            return [self._bounds_host[0], self._bounds_host[1]]
        return self.variable_bounds

    # ---- device batch
    @property
    def handle(self):
        if self._batch is None:
            L = _lib.lib()
            h = C.c_void_p()
            if self.devices is None:
                _lib.check(L.dto_batch_create(self.shape, self.batch, None, 0, C.byref(h)))
            else:
                dv = (C.c_int * len(self.devices))(*self.devices)
                _lib.check(L.dto_batch_create(self.shape, self.batch, dv, len(self.devices), C.byref(h)))
            self._batch = h
        return self._batch

    def close(self):
        if self._batch is not None:
            _lib.lib().dto_batch_destroy(self._batch)
            self._batch = None

    def set_parameters(self, w):
        w = _f64(w, (self.batch, self.num_parameter), "parameters")
        _lib.check(_lib.lib().dto_set_parameters(self.handle, _p(w)))
        self._w_host = w.copy()         # (a solve over several devices re-creates one batch per device: it needs them again)

    def set_x(self, z):
        z = _f64(z, (self.batch, self.num_variables), "variables")
        _lib.check(_lib.lib().dto_set_x(self.handle, _p(z)))

    def set_duals(self, scaling, duals):
        s = np.ascontiguousarray(np.broadcast_to(np.asarray(scaling, dtype=np.float64), (self.batch,)))
        lam = _f64(duals, (self.batch, self.num_constraint), "duals")
        _lib.check(_lib.lib().dto_set_duals(self.handle, _p(s), _p(lam)))

    # ---- the five callbacks (src/moi.jl)
    def eval_objective(self, variables=None):
        if variables is not None:
            self.set_x(variables)
        f = np.empty(self.batch)
        _lib.check(_lib.lib().dto_eval_objective(self.handle, _p(f)))
        return f

    def eval_objective_gradient(self, gradient, variables=None):
        g = _out(gradient, (self.batch, self.num_variables), "gradient")
        if variables is not None:
            self.set_x(variables)
        _lib.check(_lib.lib().dto_eval_objective_gradient(self.handle, _p(g)))

    def eval_constraint(self, violations, variables=None):
        c = _out(violations, (self.batch, self.num_constraint), "violations")
        if variables is not None:
            self.set_x(variables)
        _lib.check(_lib.lib().dto_eval_constraint(self.handle, _p(c)))

    def eval_constraint_jacobian(self, jacobian, variables=None):
        J = _out(jacobian, (self.batch, self.num_jacobian), "jacobian")
        if variables is not None:
            self.set_x(variables)
        _lib.check(_lib.lib().dto_eval_constraint_jacobian(self.handle, _p(J)))

    def eval_hessian_lagrangian(self, hessian, variables=None, scaling=None, duals=None):
        H = _out(hessian, (self.batch, self.num_hessian), "hessian")
        if variables is not None:
            self.set_x(variables)
        if duals is not None:
            self.set_duals(1.0 if scaling is None else scaling, duals)
        elif scaling is not None:
            # MOI's signature always carries sigma together with lambda (src/moi.jl:72): a lone sigma would silently
            # keep the multipliers of some earlier call
            raise ValueError("eval_hessian_lagrangian: scaling given without duals; pass both (MOI.eval_hessian_lagrangian(H, z, sigma, lambda))")
        _lib.check(_lib.lib().dto_eval_hessian_lagrangian(self.handle, _p(H)))

    def eval_jacobian_hessian(self, jacobian, hessian, variables=None, scaling=None, duals=None, chunks: int = 0):
        """Fused Jacobian + Hessian-of-Lagrangian pass (one kernel over the knots)."""
        J = _out(jacobian, (self.batch, self.num_jacobian), "jacobian")
        H = _out(hessian, (self.batch, self.num_hessian), "hessian")
        if variables is not None and duals is not None:
            # one pipelined host call: chunked copy-in / kernel / copy-out over several streams
            z = _f64(variables, (self.batch, self.num_variables), "variables")
            s = np.ascontiguousarray(np.broadcast_to(np.asarray(1.0 if scaling is None else scaling, dtype=np.float64),
                                                     (self.batch,)))
            lam = _f64(duals, (self.batch, self.num_constraint), "duals")
            _lib.check(_lib.lib().dto_eval_jacobian_hessian_host(self.handle, _p(z), _p(s), _p(lam), _p(J), _p(H), chunks))
            return
        if variables is not None:
            self.set_x(variables)
        if duals is not None:
            self.set_duals(1.0 if scaling is None else scaling, duals)
        elif scaling is not None:
            raise ValueError("eval_jacobian_hessian: scaling given without duals; pass both")
        _lib.check(_lib.lib().dto_eval_jacobian_hessian(self.handle, _p(J), _p(H)))

    # ---- device-resident interface (no host copies)
    def new_batch(self, batch: Optional[int] = None, devices: Optional[Sequence[int]] = None) -> "BatchedNLPData":
        """Another batch of the same shape (shares the model library and static tables)."""
        other = object.__new__(BatchedNLPData)
        other.__dict__.update(self.__dict__)
        other._batch = None
        other.batch = int(batch) if batch is not None else self.batch
        if other.batch != self.batch:       # per-problem rows belong to this batch's problems: the caller hands over a slice
            other._bounds_host = None
        other.devices = list(devices) if devices is not None else self.devices
        return other

    def launch(self, kernel_id: int) -> None:
        """Enqueue one callback on the batch's stream(s) without synchronising."""
        _lib.check(_lib.lib().dto_launch(self.handle, kernel_id))

    def sync(self) -> None:
        _lib.check(_lib.lib().dto_sync(self.handle))

    def set_stream(self, cuda_stream: int, shard: int = 0) -> None:
        _lib.check(_lib.lib().dto_set_stream(self.handle, shard, C.c_void_p(cuda_stream)))

    def launch_count(self) -> int:
        return int(_lib.lib().dto_launch_count(self.handle))

    @property
    def num_shards(self) -> int:
        return int(_lib.lib().dto_batch_num_shards(self.handle))

    def shard_device(self, shard: int = 0) -> int:
        return int(_lib.lib().dto_shard_device(self.handle, shard))

    def shard_range(self, shard: int = 0):
        L = _lib.lib()
        return int(L.dto_shard_begin(self.handle, shard)), int(L.dto_shard_size(self.handle, shard))

    def stream_pointer(self, shard: int = 0) -> int:
        return int(_lib.lib().dto_get_stream(self.handle, shard) or 0)

    def device_pointer(self, array: int, shard: int = 0) -> int:
        p = _lib.lib().dto_device_pointer(self.handle, array, shard)
        if not p:
            raise _lib.DtoError(-1, _lib.lib().dto_last_error().decode(errors="replace"))
        return int(p)

    def algorithmic_bytes_per_problem(self) -> int:
        return int(_lib.lib().dto_algorithmic_bytes_per_problem(self.shape))

    def compiled_gather(self) -> bool:
        return bool(_lib.lib().dto_shape_compiled_gather(self.shape))

    def kernel_smem_bytes(self, kernel_id: int) -> int:
        return int(_lib.lib().dto_kernel_smem_bytes(self.shape, kernel_id))

    def last_x(self, problem: int = 0) -> np.ndarray:
        z = np.empty(self.num_variables)
        _lib.check(_lib.lib().dto_get_last_x(self.handle, problem, _p(z)))
        return z


class Solver:
    """Solver(dynamics, objective, constraints, bounds; evaluate_hessian, general_constraint, options,
    parameters) (src/solver.jl:6-21) + batch=B, devices=[...], shared_parameters, name.

    `parameters`: the reference's per-knot list (broadcast to every problem) -- or call
    `solver.nlp.set_parameters(W)` with W[B, num_parameter] for per-problem data.
    `shared_parameters=True` lets every knot see the same small per-problem vector
    (w_t = w for all t) instead of the reference's vcat(parameters...) layout."""

    def __init__(self, dynamics: List[Dynamics], objective: List[Cost], constraints: List[Constraint],
                 bounds: List[Bound], evaluate_hessian: bool = False,
                 general_constraint: Optional[GeneralConstraint] = None, options=None, parameters=None,
                 batch: int = 1, devices: Optional[Sequence[int]] = None, shared_parameters: bool = False,
                 name: str = "model", verbose: bool = False):
        T = len(objective)
        if len(dynamics) != T - 1 or len(constraints) != T:
            raise ValueError(f"need T-1 dynamics and T constraints for T={T} costs (got {len(dynamics)}, {len(constraints)})")
        self.options = options

        def kinds(elems, allow_empty=False):
            uniq, ids, out = [], {}, []
            for e in elems:
                if allow_empty and e.spec is None:
                    out.append(-1)
                    continue
                if id(e) not in ids:
                    ids[id(e)] = len(uniq)
                    uniq.append(e)
                out.append(ids[id(e)])
            return uniq, out

        dyn_u, dyn_k = kinds(dynamics)
        cost_u, cost_k = kinds(objective)
        stage_u, stage_k = kinds(constraints, allow_empty=True)
        general = general_constraint if (general_constraint is not None and general_constraint.spec is not None) else None
        spec = ModelSpec(name=name, dyn=[e.spec for e in dyn_u], cost=[e.spec for e in cost_u],
                         stage=[e.spec for e in stage_u], general=general.spec if general else None)
        # compiled Hessian gather: the distinct per-knot recipes of THIS shape (a handful for any horizon)
        from .recipes import classes_of, knot_meta, knot_recipes
        rec = knot_recipes(T, dyn_k, cost_k, stage_k, spec.dyn, spec.cost, spec.stage, spec.general)
        import os
        if rec is not None and os.environ.get("DTO_TABLE_GATHER", "0") != "1":
            classes, metas, _ = classes_of(rec, knot_meta(T, dyn_k, cost_k, stage_k, spec.dyn, spec.cost, spec.stage))
            if len(classes) <= 16 and max(len(c) for c in classes) <= 128:
                spec.hg_classes = classes
                spec.hg_meta = metas
        self.model = Model(spec, verbose=verbose)

        pdim = []
        for t in range(T):
            els = [objective[t], constraints[t]] + ([dynamics[t]] if t < T - 1 else [])
            pdim.append(max(e.num_parameter for e in els))
        if shared_parameters:
            poff, nparam = [0] * T, max(pdim) if pdim else 0
        else:
            poff, nparam = None, sum(pdim)
        self.parameter_dim = pdim
        self.nlp = BatchedNLPData(self.model, T, dyn_k, cost_k, stage_k, general is not None, pdim, poff, nparam,
                                  evaluate_hessian, bounds, batch, devices)
        self._initial = np.zeros((batch, self.nlp.num_variables))
        if parameters is not None and self.nlp.num_parameter > 0:
            flat = np.concatenate([np.asarray(p, float).reshape(-1) for p in parameters]) if not shared_parameters \
                else np.asarray(parameters, float).reshape(-1)
            self.nlp.set_parameters(np.tile(flat, (batch, 1)))

    # warm start (src/solver.jl:23-39): stored host-side until a solver consumes it
    def initialize_states(self, states, problem: Optional[int] = None):
        xs, nx, _, _ = self.nlp.knot_layout()
        rows = slice(None) if problem is None else problem
        for t, xt in enumerate(states):
            self._initial[rows, xs[t] - 1: xs[t] - 1 + len(xt)] = np.asarray(xt, float)

    def set_bounds(self, bounds: List[Bound], problem: Optional[int] = None):
        """The variable bounds of one problem (or, with problem=None, of every problem): a list of T Bound objects laid out
        exactly as the `bounds` argument (primal_bounds, src/data.jl:123-133). Problems of one batch may differ in bound
        values -- start and end states pinned by Bound(state_lower = x1, state_upper = x1), actuator limits -- but not in
        pattern (which variables are pinned, lower-bounded, upper-bounded): see BatchedNLPData.set_variable_bounds."""
        lo, up = self.nlp.primal_bounds(bounds)
        if self.nlp._bounds_host is None:       # the first per-problem row: every problem starts from the Bound objects
            self.nlp.set_variable_bounds(*(np.tile(v, (self.nlp.batch, 1)) for v in self.nlp.variable_bounds))
        sel = slice(None) if problem is None else problem
        self.nlp._bounds_host[0][sel] = lo      # (in place: a batch of thousands is filled one problem at a time)
        self.nlp._bounds_host[1][sel] = up

    def initialize_controls(self, actions, problem: Optional[int] = None):
        _, _, us, _ = self.nlp.knot_layout()
        rows = slice(None) if problem is None else problem
        for t, ut in enumerate(actions):
            self._initial[rows, us[t] - 1: us[t] - 1 + len(ut)] = np.asarray(ut, float)

    def get_trajectory(self, problem: int = 0):
        """src/solver.jl:41-43: per-knot views of the last z any callback saw."""
        z = self.nlp.last_x(problem)
        xs, nx, us, nu = self.nlp.knot_layout()
        states = [z[xs[t] - 1: xs[t] - 1 + nx[t]].copy() for t in range(self.nlp.T)]
        actions = [z[us[t] - 1: us[t] - 1 + nu[t]].copy() for t in range(self.nlp.T - 1)]
        return states, actions

    def solve(self, options: Optional[dict] = None, record_iterates: bool = False, method: str = "auto"):
        """solve!(solver) (src/solver.jl:45-47) for every problem of the batch. The reference's caller is
        Ipopt, which is not available in this image. These drivers stand in for it:
          * "native" (default where it applies: exact Hessians; equality rows and rows c(z) <= 0; variables free, pinned
            by equal bounds, or bounded): the lock-step batched Newton-KKT solver inside libdto.so (dto_sqp_solve) --
            callbacks, KKT assembly, factorisation, line-search evaluations and all bookkeeping on the device, no
            per-problem host solver; inequalities by a primal-dual interior point on the same kernels (no restoration
            phase: scope note in sqp.py). A batch over several devices is solved one device per host thread;
          * "sqp": the same algorithm with torch doing the bookkeeping (sqp.py `solve` / `solve_bounded`; the statement of
            the algorithm and the arm the oracle-driven twin mirrors; the only one that records iterates; one device);
          * "broker": B per-problem host NLP solvers (SciPy trust-constr) running in lock step whose
            callbacks rendezvous into batched GPU calls (driver.py, SURVEY 8f N1): the protocol an Ipopt-
            per-task driver would use.
        `get_trajectory(problem)` afterwards returns the final iterate."""
        if method == "auto":
            lo, up = self.nlp.variable_bounds
            clo, cup = self.nlp.constraint_bounds
            pinned = np.isfinite(lo) & (lo == up)
            rows_ok = bool(np.all((clo == cup) | (np.isneginf(clo) & (cup == 0.0))))      # equalities and c(z) <= 0 rows
            # a problem without Hessians reaches the native solver when one of its quasi-Newton modes is asked for
            qn = (options or {}).get("hessian_approximation", "exact") in ("knot-bfgs", "partitioned-bfgs")
            ok = (self.nlp.hessian_lagrangian or qn) and rows_ok        # (several devices: one native solve per device, side by side)
            # (bounds on variables (Bound(action_lower = ..., ...)) and inequality rows (Constraint(...; indices_inequality)): the
            # interior-point mode, in both arms)
            method = ("sqp" if record_iterates else "native") if ok else "broker"
        if method in ("sqp", "native"):
            from . import sqp
            o = sqp.SQPOptions()
            ref_opts = self.options if isinstance(self.options, dict) else {}
            if "max_iter" in ref_opts:
                o.max_iter = int(ref_opts["max_iter"])       # Options.max_iter (src/options.jl:9)
            for k_, v in (options or {}).items():
                setattr(o, k_, v)
        if method == "native":
            if record_iterates:
                raise ValueError("solve: record_iterates needs method='sqp' (the native solver keeps no history)")
            res = sqp.solve_native(self.nlp, self._initial, options=o) if self.nlp.num_shards == 1 else \
                sqp.solve_native_sharded(self.nlp, self._initial, options=o)
            self.sqp_launches = res.stats["launches"]
            self.results, self.iterates, self.broker = res, [], None
            return res
        if method == "sqp":
            be = sqp.DeviceBackend(self.nlp, dual_reg=o.dual_reg, options=o)
            res = None
            try:
                z0 = be.torch.as_tensor(self._initial, device=be.xp.device)
                res = sqp.solve_bounded(be, z0, options=o, record=record_iterates)    # = sqp.solve when no bound is an inequality
                Z = res.z.cpu().numpy()
                self.sqp_launches = res.backend.total_launches()
            finally:
                if res is not None and res.backend is not be:
                    res.backend.close()
                be.close()
            self.nlp.set_x(Z)
            self.results, self.iterates, self.broker = res, res.history, None
            return res
        from .driver import solve_batch
        opts = dict(options or {})
        opts.pop("hessian_approximation", None)         # (SciPy's trust-constr keeps its own quasi-Newton approximation)
        ref_opts = self.options if isinstance(self.options, dict) else {}
        if "tol" in ref_opts and "gtol" not in opts:        # Options.tol (src/options.jl:7)
            opts["gtol"] = float(ref_opts["tol"])
        if "max_iter" in ref_opts and "maxiter" not in opts:  # Options.max_iter (src/options.jl:9)
            opts["maxiter"] = int(ref_opts["max_iter"])
        Z, results, broker, iterates = solve_batch(self.nlp, self._initial, options=opts, record_iterates=record_iterates)
        self.nlp.set_x(Z)   # get_trajectory returns the evaluator's last z (src/solver.jl:41-43)
        self.results, self.broker, self.iterates = results, broker, iterates
        return results


def initialize_states(solver: Solver, states):
    solver.initialize_states(states)


def initialize_controls(solver: Solver, actions):
    solver.initialize_controls(actions)


def get_trajectory(solver: Solver):
    return solver.get_trajectory()


def solve(solver: Solver):
    return solver.solve()


def linear_interpolation(initial_state, final_state, horizon):
    """src/utils.jl:1-10"""
    x0, x1 = np.asarray(initial_state, float), np.asarray(final_state, float)
    return [(x1 - x0) / (horizon - 1) * t + x0 for t in range(horizon)]


def solver_from(model: dict, batch: int = 1, devices=None, parameters=None, verbose: bool = False) -> Solver:
    """Assemble a Solver from an examples.models builder dict."""
    return Solver(model["dynamics"], model["objective"], model["constraints"], model["bounds"],
                  evaluate_hessian=model.get("evaluate_hessian", False), general_constraint=model.get("general"),
                  parameters=parameters, batch=batch, devices=devices,
                  shared_parameters=bool(model.get("shared_parameters", False)), name=model.get("name", "model"),
                  verbose=verbose)

"""Device-resident KKT systems of a batch: host mirror of the `dto_kkt_*` entry points of
include/dto.h (SURVEY 8f row N3).

The reference sketches this consumer of the callbacks in
/root/reference/examples/pendulum/pendulum.jl:138-211: from g, c, J, H build

    K = [H + primal_reg I, J'; J, -dual_reg I],   h = [g + J'y; c],   F = qdldl(K),   sol = F \\ h

Here that happens for every problem of the batch on the GPU, from the arrays the callback kernels
left in HBM; only `sol` comes back. All numerics are in libdto.so's CUDA kernels -- this module only
marshals pointers and raises if the native pieces or a GPU are missing.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .evaluator import BatchedNLPData, _out, _p


HESSIAN = {"exact": 0, "knot-blocks": 1}   # DTO_KKT_HESSIAN_EXACT, DTO_KKT_HESSIAN_KNOT_BLOCKS


def _hessian_mode(hessian: str) -> int:
    if hessian not in HESSIAN:
        raise ValueError(f"hessian={hessian!r}: expected one of {sorted(HESSIAN)}")
    return HESSIAN[hessian]


def analyze(nlp: BatchedNLPData, hessian: str = "exact"):
    """Host-only symbolic phase: (perm, bandwidth). perm[p] is the 1-based index (variables first,
    then constraint rows) placed at position p of the banded ordering. hessian="knot-blocks": the H block
    of K is one dense block per knot (nlp.hessian_block_structure()) instead of the Hessian's structure."""
    n = nlp.num_variables + nlp.num_constraint
    perm = np.empty(n, dtype=np.int64)
    bw = C.c_int64()
    _lib.check(_lib.lib().dto_kkt_analyze_ex(nlp.shape, _hessian_mode(hessian), perm.ctypes.data_as(C.POINTER(C.c_int64)), C.byref(bw)))
    return perm, int(bw.value)


class KKTSystem:
    """K sol = h for all problems of `nlp` (pendulum.jl:138-211 batched).

    hessian="knot-blocks": H is not the callbacks' Hessian but one dense symmetric block per knot owned by this
    object (the identity at first; set_hessian_blocks / hessian_blocks, shape [B, nnz_blk] in the order of
    nlp.hessian_block_structure()); the callbacks then run without a Hessian pass, so a problem built without
    evaluate_hessian works."""

    def __init__(self, nlp: BatchedNLPData, primal_reg: float = 1.0e-5, dual_reg: float = 1.0e-5, hessian: str = "exact"):
        L = _lib.lib()
        self.nlp = nlp
        self.hessian = hessian
        h = C.c_void_p()
        _lib.check(L.dto_kkt_create_ex(nlp.handle, float(primal_reg), float(dual_reg), _hessian_mode(hessian), C.byref(h)))
        self._h = h
        self.num_blocks = int(L.dto_hessian_block_count(nlp.shape)) if hessian == "knot-blocks" else 0
        self.dim = int(L.dto_kkt_dim(h))
        self.bandwidth = int(L.dto_kkt_bandwidth(h))
        self.row_width = int(L.dto_kkt_row_width(h))
        self.factor_bytes_per_problem = int(L.dto_kkt_factor_bytes_per_problem(h))

    def close(self):
        if self._h is not None:
            _lib.lib().dto_kkt_destroy(self._h)
            self._h = None

    def permutation(self) -> np.ndarray:
        perm = np.empty(self.dim, dtype=np.int64)
        _lib.check(_lib.lib().dto_kkt_permutation(self._h, perm.ctypes.data_as(C.POINTER(C.c_int64))))
        return perm

    def solve(self, solution=None, variables=None, scaling=None, duals=None, chunks: int = 0):
        """Callbacks at (z, sigma, y) + assembly + LDL' + solve; `solution` [B, dim] is written in
        place (None: results stay on the device). With host `variables`, `duals` and `solution` all
        given, the call is one chunk-pipelined host call (copies overlap the kernels)."""
        if variables is not None and duals is not None and solution is not None:
            from .evaluator import _f64
            nlp = self.nlp
            z = _f64(variables, (nlp.batch, nlp.num_variables), "variables")
            lam = _f64(duals, (nlp.batch, nlp.num_constraint), "duals")
            sg = None
            if scaling is not None:
                sg = np.ascontiguousarray(np.broadcast_to(np.asarray(scaling, dtype=np.float64), (nlp.batch,)))
            sol = _out(solution, (nlp.batch, self.dim), "solution")
            _lib.check(_lib.lib().dto_kkt_solve_host(self._h, _p(z), _p(sg) if sg is not None else None, _p(lam), _p(sol), int(chunks)))
            return solution
        if variables is not None:
            self.nlp.set_x(variables)
        if duals is not None:
            self.nlp.set_duals(1.0 if scaling is None else scaling, duals)
        if solution is not None:
            solution = _out(solution, (self.nlp.batch, self.dim), "solution")
        _lib.check(_lib.lib().dto_kkt_solve(self._h, _p(solution) if solution is not None else None))
        return solution

    def launch(self, with_callbacks=True) -> None:
        """with_callbacks: True/1 callbacks + right-hand side + factor/solve; False/0 linear algebra only on the
        g, c, J, H resident on the device; 2 callbacks only."""
        _lib.check(_lib.lib().dto_kkt_launch(self._h, int(with_callbacks)))

    def launch_subset(self, idx_device_ptr: int, count: int) -> None:
        """Linear algebra only (as launch(0)) for `count` problems whose int32 numbers sit at a DEVICE address."""
        _lib.check(_lib.lib().dto_kkt_launch_subset(self._h, C.c_void_p(int(idx_device_ptr)), int(count)))

    def resolve(self, idx_device_ptr: int = 0, count: int = 0) -> None:
        """New right-hand side, solve with the factor already on the device (no factorisation): all problems, or `count`
        problems listed at a DEVICE address. Bit-identical to launch(0) while K is unchanged."""
        _lib.check(_lib.lib().dto_kkt_resolve(self._h, C.c_void_p(int(idx_device_ptr)) if idx_device_ptr else None, int(count)))

    def set_fixed(self, fixed=None) -> None:
        """Pinned variables (equal lower/upper bounds): boolean mask [num_variables]; their step is exactly zero."""
        if fixed is None:
            _lib.check(_lib.lib().dto_kkt_set_fixed(self._h, None))
            return
        m = np.ascontiguousarray(np.asarray(fixed).astype(np.uint8))
        if m.shape != (self.nlp.num_variables,):
            raise ValueError(f"fixed: expected shape ({self.nlp.num_variables},)")
        _lib.check(_lib.lib().dto_kkt_set_fixed(self._h, m.ctypes.data_as(C.c_void_p)))

    def set_primal_reg(self, reg=None) -> None:
        """Per-problem primal regularisation [B] (inertia control); None: back to the scalar of the constructor."""
        if reg is None:
            _lib.check(_lib.lib().dto_kkt_set_primal_reg(self._h, None))
            return
        from .evaluator import _f64
        r = _f64(reg, (self.nlp.batch,), "reg")
        _lib.check(_lib.lib().dto_kkt_set_primal_reg(self._h, _p(r)))

    def inertia(self) -> np.ndarray:
        """Negative pivots of D per problem for the last factorisation (== num_constraint when K is quasi-definite)."""
        out = np.empty(self.nlp.batch, dtype=np.int32)
        _lib.check(_lib.lib().dto_kkt_inertia(self._h, out.ctypes.data_as(C.c_void_p)))
        return out

    def rhs(self) -> np.ndarray:
        out = np.empty((self.nlp.batch, self.dim))
        _lib.check(_lib.lib().dto_kkt_get(self._h, 0, _p(out)))
        return out

    def solution(self) -> np.ndarray:
        out = np.empty((self.nlp.batch, self.dim))
        _lib.check(_lib.lib().dto_kkt_get(self._h, 1, _p(out)))
        return out

    def matrix(self, problem: int = 0) -> np.ndarray:
        out = np.empty((self.dim, self.dim))
        _lib.check(_lib.lib().dto_kkt_matrix(self._h, int(problem), _p(out)))
        return out

    def factor(self, problem: int = 0):
        """(L, D) of P K P' = L D L' as dense arrays, P = permutation()."""
        W = self.row_width
        band = np.empty((self.dim, W))
        D = np.empty(self.dim)
        _lib.check(_lib.lib().dto_kkt_factor(self._h, int(problem), _p(band), _p(D)))
        Lm = np.eye(self.dim)
        for q in range(1, W):
            idx = np.arange(q, self.dim)
            Lm[idx, idx - q] = band[q:, q]
        return Lm, D

    def set_hessian_blocks(self, blocks) -> None:
        """knot-blocks mode: the blocks of every problem, [B, nnz_blk] (host -> device)."""
        from .evaluator import _f64
        v = _f64(blocks, (self.nlp.batch, self.num_blocks), "blocks")
        _lib.check(_lib.lib().dto_kkt_set_hessian_blocks(self._h, _p(v)))

    def hessian_blocks(self) -> np.ndarray:
        """knot-blocks mode: the blocks of every problem, [B, nnz_blk] (device -> host)."""
        out = np.empty((self.nlp.batch, self.num_blocks))
        _lib.check(_lib.lib().dto_kkt_get_hessian_blocks(self._h, _p(out)))
        return out

    def device_pointer(self, which: int, shard: int = 0) -> int:
        p = _lib.lib().dto_kkt_device_pointer(self._h, int(which), int(shard))
        if not p:
            raise _lib.DtoError(-1, _lib.lib().dto_last_error().decode(errors="replace"))
        return int(p)

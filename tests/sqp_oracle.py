"""TEST INFRASTRUCTURE: the oracle-driven twin of the batched SQP solver (dto_b200/sqp.py). Same algorithm
(the very function sqp.solve), numpy arrays, callbacks from the CPU oracle (python restatement or its C twin),
KKT solves problem by problem with the oracle's restatement of the pendulum script + QDLDL (oracle/kkt.py), the banded LDL'
of the product's ordering (problem by problem, or vectorised over the batch for shipped sizes) or a dense factorisation. Used
by the parity tests of the solver and to prototype on the CPU."""
from __future__ import annotations

import numpy as np

from dto_b200.sqp import _XP
from oracle import kkt as OK


def band_ldl_solve(K, h, perm, bw):
    """P K P' = L D L' without pivoting on the band (the factorisation the GPU kernel computes, and QDLDL for
    that ordering), solve, and the number of negative pivots."""
    n = K.shape[0]
    A = K[np.ix_(perm, perm)].copy()
    x = np.asarray(h, dtype=np.float64)[perm].copy()
    D = np.empty(n)
    Ls = []
    for j in range(n):
        hi = min(n, j + bw + 1)
        d = A[j, j]
        D[j] = d
        col = A[j + 1:hi, j].copy()
        l = col / d
        A[j + 1:hi, j + 1:hi] -= np.outer(l, col)
        x[j + 1:hi] -= l * x[j]
        Ls.append(l)
    x = x / D
    for j in range(n - 1, -1, -1):
        hi = min(n, j + bw + 1)
        x[j] -= Ls[j] @ x[j + 1:hi]
    out = np.empty(n)
    out[perm] = x
    return out, int((D < 0).sum())


def band_ldl_solve_batched(K, h, perm, bw):
    """`band_ldl_solve` of a batch, K [B, n, n] and h [B, n]: the same column order and the same operations, each applied to
    every problem at once (the back substitution's dot products through a stacked matmul, which takes the same dot as `@`).
    Gives the bits of `band_ldl_solve` problem by problem. Returns the solutions [B, n] and negative pivots [B]."""
    B, n = K.shape[0], K.shape[1]
    A = K[:, perm][:, :, perm]
    x = np.asarray(h, dtype=np.float64)[:, perm].copy()
    D = np.empty((B, n))
    Ls = []
    for j in range(n):
        hi = min(n, j + bw + 1)
        d = A[:, j, j].copy()
        D[:, j] = d
        col = A[:, j + 1:hi, j].copy()
        l = col / d[:, None]
        A[:, j + 1:hi, j + 1:hi] -= l[:, :, None] * col[:, None, :]
        x[:, j + 1:hi] -= l * x[:, j:j + 1]
        Ls.append(l)
    x = x / D
    for j in range(n - 1, -1, -1):
        hi = min(n, j + bw + 1)
        if hi > j + 1:
            x[:, j] -= np.matmul(Ls[j][:, None, :], x[:, j + 1:hi, None])[:, 0, 0]
    out = np.empty((B, n))
    out[:, perm] = x
    return out, (D < 0).sum(axis=1)


class OracleBackend:
    """`linear`: "qdldl" (the oracle's QDLDL, problem by problem), "band" (`band_ldl_solve` problem by problem), "band-batched"
    (`band_ldl_solve_batched`: the same bits, the whole batch at once; for the shipped sizes) or "dense". `w` [B, N_w]: each
    problem's parameters for the C twin `c_twin` (built with shared_parameters=True); without a C twin the oracle's own
    parameters (osolver.set_parameters) are shared by the whole batch. `retries` lists, for every inertia-correction pass,
    how many problems it factorised again."""

    def __init__(self, osolver, B, dual_reg=1.0e-9, c_twin=None, perm=None, linear="qdldl", bw=None, options=None, w=None):
        self.bw = bw
        self.gauss_newton = False
        self.o = osolver.nlp
        self.B, self.N_z, self.N_c = B, self.o.num_variables, self.o.num_constraint
        self.xp = _XP(np)
        lo, up = self.o.variable_bounds
        lo, up = np.asarray(lo, float), np.asarray(up, float)
        from dto_b200.sqp import bound_arrays
        clo, cup = self.o.constraint_bounds
        self._bound_args = (lo, up, options, clo, cup)
        self.fixed, self.bounds = bound_arrays(lo, up, options, clo, cup)
        self.free = (~self.fixed).astype(np.float64)
        self.pinned_value = np.where(self.fixed, lo, 0.0)
        self.diag = None
        self.dual_reg = dual_reg
        self.co = c_twin
        self.perm = perm
        self.linear = linear
        self.w = None if w is None else np.ascontiguousarray(w, dtype=np.float64)
        if self.w is not None and (c_twin is None or self.w.shape[0] != B):
            raise ValueError("per-problem parameters need the C twin and one row per problem")
        self.retries = []
        self.js, self.hs = self.o.jacobian_structure(), self.o.hessian_lagrangian_structure()
        jr = np.array([r for r, _ in self.js]) - 1
        jc = np.array([c for _, c in self.js]) - 1
        hr = np.array([r for r, _ in self.hs]) - 1
        hc = np.array([c for _, c in self.hs]) - 1
        self._idx = (jr, jc, hr, hc)

    def set_bound_scale(self, scale):
        if self.bounds is not None:
            from dto_b200.sqp import bound_arrays
            _, self.bounds = bound_arrays(*self._bound_args, scale=scale)

    def pin(self, z):
        return z * self.free + self.pinned_value

    def shrink(self, keep):
        import copy
        other = copy.copy(self)
        other.B = int(np.count_nonzero(keep))
        if self.w is not None:
            other.w = self.w[np.asarray(keep, dtype=bool)]
        return other

    def _eval(self, z, lam, what):
        B = z.shape[0]
        if self.co is not None:
            return self.co.eval(what, z, lam, np.ones(B), np.zeros((B, 0)) if self.w is None else self.w)
        out = dict(f=np.zeros(B), g=np.zeros((B, self.N_z)), c=np.zeros((B, self.N_c)), J=np.zeros((B, len(self.js))),
                   H=np.zeros((B, len(self.hs))))
        for b in range(B):
            out["f"][b] = self.o.eval_objective(z[b])
            if what & 2:
                self.o.eval_objective_gradient(out["g"][b], z[b])
            if what & 4:
                self.o.eval_constraint(out["c"][b], z[b])
            if what & 8:
                self.o.eval_constraint_jacobian(out["J"][b], z[b])
            if what & 16:
                self.o.eval_hessian_lagrangian(out["H"][b], z[b], 1.0, lam[b])
        return out

    def callbacks(self, z, lam, lam_hess, delta=None, diag=None, gshift=None, cshift=None):
        self.cur = self._eval(z, lam_hess, 31)
        self.lam = lam.copy()
        self.diag = None if diag is None else np.array(diag, copy=True)     # interior point: diagonal added to K,
        if gshift is not None:                                              # barrier gradient in g,
            self.cur["g"] = self.cur["g"] + gshift
        c_raw = self.cur["c"].copy()
        if cshift is not None:                                              # c + mu / lam on inequality rows (right-hand side)
            self.cur["c"] = self.cur["c"] + cshift
        return self.cur["f"].copy(), self.cur["g"].copy(), c_raw

    def _assemble(self, b, delta):
        jr, jc, hr, hc = self._idx
        n, m = self.N_z, self.N_c
        K = np.zeros((n + m, n + m))
        K[hr, hc] = self.cur["H"][b]
        K[n + jr, jc] = self.cur["J"][b]
        K[jc, n + jr] = self.cur["J"][b]
        K[np.arange(n), np.arange(n)] += delta
        if self.diag is not None:
            w = self.diag.shape[1]
            K[np.arange(w), np.arange(w)] += self.diag[b]
        K[n + np.arange(m), n + np.arange(m)] -= self.dual_reg
        Jd = np.zeros((m, n))
        Jd[jr, jc] = self.cur["J"][b]
        h = np.concatenate([self.cur["g"][b] + Jd.T @ self.lam[b], self.cur["c"][b]])
        if self.fixed.any():          # pinned variables: identity rows / columns, zero right-hand side
            fx = np.nonzero(self.fixed)[0]
            K[fx, :] = 0.0
            K[:, fx] = 0.0
            K[fx, fx] = 1.0
            h[fx] = 0.0
        return K, h

    def newton_soc(self, c_soc, delta, mask=None):
        saved = self.cur["c"]
        self.cur["c"] = np.asarray(c_soc)
        try:
            return self.newton(delta)[0]
        finally:
            self.cur["c"] = saved

    def _assemble_batch(self, delta):
        """`_assemble` of every problem at once: K [B, dim, dim], h [B, dim] (the same entries; J'lam by the same matvec)"""
        jr, jc, hr, hc = self._idx
        B, n, m = self.B, self.N_z, self.N_c
        K = np.zeros((B, n + m, n + m))
        K[:, hr, hc] = self.cur["H"]
        K[:, n + jr, jc] = self.cur["J"]
        K[:, jc, n + jr] = self.cur["J"]
        K[:, np.arange(n), np.arange(n)] += np.asarray(delta, dtype=np.float64)[:, None]
        if self.diag is not None:
            w = self.diag.shape[1]
            K[:, np.arange(w), np.arange(w)] += self.diag
        K[:, n + np.arange(m), n + np.arange(m)] -= self.dual_reg
        h = np.empty((B, n + m))
        Jd = np.zeros((m, n))
        for b in range(B):
            Jd[jr, jc] = self.cur["J"][b]
            h[b, :n] = self.cur["g"][b] + Jd.T @ self.lam[b]
        h[:, n:] = self.cur["c"]
        if self.fixed.any():
            fx = np.nonzero(self.fixed)[0]
            K[:, fx, :] = 0.0
            K[:, :, fx] = 0.0
            K[:, fx, fx] = 1.0
            h[:, fx] = 0.0
        return K, h

    def newton(self, delta, mask=None):
        n, m = self.N_z, self.N_c
        if mask is not None:
            self.retries.append(int(np.count_nonzero(mask)))
        if self.linear == "band-batched":
            K, h = self._assemble_batch(delta)
            sol, nneg = band_ldl_solve_batched(K, h, self.perm, self.bw)
            return sol, nneg.astype(np.float64), h[:, :n].copy()
        sol = np.zeros((self.B, n + m))
        nneg = np.zeros(self.B)
        rz = np.zeros((self.B, n))
        for b in range(self.B):
            K, h = self._assemble(b, float(delta[b]))
            rz[b] = h[:n]
            if self.linear == "qdldl":
                try:
                    Lm, D, Dinv, pos = OK.qdldl_factor(K, self.perm)
                    sol[b] = OK.qdldl_solve(Lm, Dinv, h, self.perm)
                    nneg[b] = (n + m) - pos
                except ZeroDivisionError:
                    sol[b] = np.nan
            elif self.linear == "band":
                sol[b], nneg[b] = band_ldl_solve(K, h, self.perm, self.bw)
            else:
                ev = np.linalg.eigvalsh(K)
                nneg[b] = int((ev < 0).sum())
                sol[b] = np.linalg.solve(K, h)
        return sol, nneg, rz

    def objective_constraint(self, z):
        out = self._eval(z, np.zeros((z.shape[0], self.N_c)), 1 | 4)
        return out["f"].copy(), out["c"].copy()

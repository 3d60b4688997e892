"""CPU tests of the knot-block damped BFGS mode of the native solver (hessian_approximation = "knot-bfgs"): the block Hessian
structure and the KKT ordering it gives (host-only queries of libdto.so), the update rule `sqp.knot_bfgs_update` on random
data, and the oracle-driven twin of the mode -- the very `sqp.solve` with H taken from knot blocks that the twin updates with
`knot_bfgs_update` -- which the GPU tests hold the native solver to."""
import numpy as np
import pytest

import dto_b200 as D
from dto_b200 import _lib
from dto_b200 import kkt as PK
from dto_b200 import sqp
from examples import models as M
from oracle import api as O

from sqp_oracle import OracleBackend

XP = sqp._XP(np)


class QNOracleBackend(OracleBackend):
    """OracleBackend whose H is the knot blocks (nlp.hessian_block_structure()), updated in `callbacks` -- after the
    callbacks, before the right-hand side, with the multipliers as they stand and g before any barrier term: where the
    native solver's k_qn_update runs. No Hessian is evaluated."""

    def __init__(self, osolver, pnlp, B, **kw):
        super().__init__(osolver, B, **kw)
        r, c = pnlp.hessian_block_structure()
        self.hs = list(zip(r.tolist(), c.tolist()))
        jr, jc, _, _ = self._idx
        self._idx = (jr, jc, r - 1, c - 1)
        xs, nx, _, nu = pnlp.knot_layout()
        self.knots = [(int(xs[t]) - 1, int(nx[t] + nu[t])) for t in range(pnlp.T)]
        self.blocks = [np.tile(np.eye(n), (B, 1, 1)) for _, n in self.knots]
        self.first = [np.ones(B, dtype=bool) for _ in self.knots]
        self.prev = None

    def _jtl(self, J, lam):
        jr, jc, _, _ = self._idx
        Jd = np.zeros((J.shape[0], self.N_c, self.N_z))
        Jd[:, jr, jc] = J
        return np.einsum("bij,bi->bj", Jd, lam)

    def callbacks(self, z, lam, lam_hess, delta=None, diag=None, gshift=None, cshift=None):
        cur = self._eval(z, lam, 1 | 2 | 4 | 8)
        g, J = cur["g"], cur["J"]
        if self.prev is not None:
            zp, gp, Jp = self.prev
            s = z - zp
            y = (g + self._jtl(J, lam)) - (gp + self._jtl(Jp, lam))
            for k, (o, n) in enumerate(self.knots):
                self.blocks[k], self.first[k] = sqp.knot_bfgs_update(XP, self.blocks[k], s[:, o:o + n], y[:, o:o + n], self.free[o:o + n],
                                                                     self.first[k])
        self.prev = (z.copy(), g.copy(), J.copy())
        cur["H"] = np.concatenate([b.reshape(self.B, -1) for b in self.blocks], axis=1)
        self.cur = cur
        self.lam = lam.copy()
        self.diag = None if diag is None else np.array(diag, copy=True)
        if gshift is not None:
            self.cur["g"] = self.cur["g"] + gshift
        c_raw = self.cur["c"].copy()
        if cshift is not None:
            self.cur["c"] = self.cur["c"] + cshift
        return self.cur["f"].copy(), self.cur["g"].copy(), c_raw


def qn_twin(name, kw, B, opts, lower=None):
    """(oracle solver, product nlp, twin backend) of model `name` built without Hessians"""
    mo, mp = M.BUILDERS[name](O, evaluate_hessian=False, **kw), M.BUILDERS[name](D, evaluate_hessian=False, **kw)
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    perm, bw = PK.analyze(pn, hessian="knot-blocks")
    be = QNOracleBackend(osolver, pn, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band", options=opts)
    return mp, pn, be


BLOCK_SHAPES = [("pendulum", dict()), ("cartpole", dict(T=11)), ("acrobot", dict(T=9)), ("car", dict(T=12, obstacle="general")),
                ("heterogeneous", dict())]


@pytest.mark.parametrize("name,kw", BLOCK_SHAPES)
def test_block_structure_is_one_dense_block_per_knot(name, kw):
    pn = D.solver_from(M.BUILDERS[name](D, evaluate_hessian=False, **kw), batch=1).nlp
    r, c = pn.hessian_block_structure()
    xs, nx, _, nu = pn.knot_layout()
    want = []
    for t in range(pn.T):
        o, n = int(xs[t]), int(nx[t] + nu[t])
        want += [(o + i, o + j) for i in range(n) for j in range(n)]
    assert list(zip(r.tolist(), c.tolist())) == want == sorted(want)
    assert len(r) == sum(int(nx[t] + nu[t]) ** 2 for t in range(pn.T))


@pytest.mark.parametrize("name,kw", [("pendulum", dict()), ("cartpole", dict(T=101)), ("acrobot", dict(T=101)),
                                     ("car", dict(T=51, obstacle="general"))])
def test_block_mode_ordering_fits_the_banded_factorisation(name, kw):
    pq = D.solver_from(M.BUILDERS[name](D, evaluate_hessian=False, **kw), batch=1).nlp
    pe = D.solver_from(M.BUILDERS[name](D, **kw), batch=1).nlp
    perm, bw = PK.analyze(pq, hessian="knot-blocks")
    _, bw_exact = PK.analyze(pe)
    print(f"{name} {kw}: half bandwidth knot-blocks {bw}, exact {bw_exact}")
    assert bw <= 31
    assert sorted(perm.tolist()) == list(range(1, pq.num_variables + pq.num_constraint + 1))
    with pytest.raises(ValueError):
        PK.analyze(pq, hessian="lbfgs")


def test_block_of_more_than_32_variables_is_unsupported():
    n, m = 32, 1                                  # a knot block of 33 variables
    x1 = np.zeros(n)
    dt = D.Dynamics(lambda y, x, u, w: y - (x + 0.1 * u[0]), n, n, m)
    ct = D.Cost(lambda x, u, w: sum(x[i] * x[i] for i in range(n)) + u[0] * u[0], n, m)
    cT = D.Cost(lambda x, u, w: sum(x[i] * x[i] for i in range(n)), n, 0)
    s = D.Solver([dt] * 2, [ct, ct, cT], [D.Constraint(lambda x, u, w: x - x1, n, m), D.Constraint(), D.Constraint()],
                 [D.Bound(n, m), D.Bound(n, m), D.Bound(n, 0)], name="wide33")
    with pytest.raises(_lib.DtoError) as e:
        PK.analyze(s.nlp, hessian="knot-blocks")
    assert e.value.status == -7
    PK.analyze(s.nlp)                             # the exact mode's analysis is not affected


def _spd(rng, M_, n):
    A = rng.normal(size=(M_, n, n))
    return A @ A.transpose(0, 2, 1) + n * np.eye(n)


def test_knot_bfgs_update_secant_condition_and_symmetry():
    rng = np.random.default_rng(1)
    Bk, s, y = _spd(rng, 6, 5), rng.normal(size=(6, 5)), rng.normal(size=(6, 5))
    y = np.where((s * y).sum(1, keepdims=True) > 0, y, -y)        # s'y > 0 everywhere
    out, first = sqp.knot_bfgs_update(XP, Bk, s, y, np.ones(5), np.zeros(6, dtype=bool))
    sBs, sy = np.einsum("mi,mij,mj->m", s, Bk, s), (s * y).sum(1)
    theta = np.where(sy >= 0.2 * sBs, 1.0, 0.8 * sBs / (sBs - sy))
    r = theta[:, None] * y + (1 - theta)[:, None] * np.einsum("mij,mj->mi", Bk, s)
    assert np.allclose(np.einsum("mij,mj->mi", out, s), r, rtol=1e-12, atol=1e-12)      # B+ s = r
    assert np.array_equal(out, out.transpose(0, 2, 1))
    assert not first.any()


def test_knot_bfgs_update_stays_positive_definite_after_negative_curvature():
    rng = np.random.default_rng(2)
    Bk, s = _spd(rng, 8, 6), rng.normal(size=(8, 6))
    y = -s * rng.uniform(0.5, 2.0, size=(8, 1))                     # s'y < 0: damping (theta < 1)
    out, first = sqp.knot_bfgs_update(XP, Bk, s, y, np.ones(6), np.zeros(8, dtype=bool))
    assert np.all(np.linalg.eigvalsh(out) > 0) and not first.any()
    assert not np.allclose(out, Bk)
    # sr = 0.2 s'Bs exactly when damped
    r = np.einsum("mij,mj->mi", out, s)
    assert np.allclose((s * r).sum(1), 0.2 * np.einsum("mi,mij,mj->m", s, Bk, s), rtol=1e-10)


def test_knot_bfgs_update_skips_steps_that_did_not_move_and_masks_pinned_variables():
    rng = np.random.default_rng(3)
    Bk = _spd(rng, 4, 3)
    y = rng.normal(size=(4, 3))
    out, first = sqp.knot_bfgs_update(XP, Bk, np.zeros((4, 3)), y, np.ones(3), np.ones(4, dtype=bool))
    assert np.array_equal(out, Bk) and first.all()
    s = rng.normal(size=(4, 3))
    out, first = sqp.knot_bfgs_update(XP, Bk, s, y, np.zeros(3), np.ones(4, dtype=bool))      # everything pinned
    assert np.array_equal(out, Bk) and first.all()
    s[0, 0] = np.nan                                                                       # non-finite: skipped
    out, _ = sqp.knot_bfgs_update(XP, Bk, s, y, np.ones(3), np.zeros(4, dtype=bool))
    assert np.array_equal(out[0], Bk[0])


def test_knot_bfgs_first_update_is_scaled():
    rng = np.random.default_rng(4)
    n = 4
    s, y = rng.normal(size=(3, n)), rng.normal(size=(3, n))
    y = np.where((s * y).sum(1, keepdims=True) > 0, y, -y)
    eye = np.tile(np.eye(n), (3, 1, 1))
    out, first = sqp.knot_bfgs_update(XP, eye, s, y, np.ones(n), np.ones(3, dtype=bool))
    sc = (y * y).sum(1) / (s * y).sum(1)
    ref, _ = sqp.knot_bfgs_update(XP, sc[:, None, None] * eye, s, y, np.ones(n), np.zeros(3, dtype=bool))
    assert np.array_equal(out, ref) and not first.any()
    unscaled, _ = sqp.knot_bfgs_update(XP, eye, s, y, np.ones(n), np.zeros(3, dtype=bool))
    assert not np.allclose(out, unscaled)


def test_oracle_twin_converges_on_pendulum_without_hessians():
    opts = sqp.SQPOptions(max_iter=150, dual_reg=1.0e-6)
    mp, pn, be = qn_twin("pendulum", dict(), 3, opts)
    rng = np.random.default_rng(5)
    T, n, m = mp["T"], mp["n"], mp["m"]
    z0 = np.zeros((3, T * n + (T - 1) * m))
    for t in range(T):
        z0[:, t * (n + m):t * (n + m) + n] = mp["x1"] + (mp["xT"] - mp["x1"]) * t / (T - 1)
        if t < T - 1:
            z0[:, t * (n + m) + n] = rng.normal(size=3)
    res = sqp.solve(be, z0, options=opts)
    assert res.converged.all(), res.iterations
    assert np.all(res.constraint_violation <= 1e-8)
    assert not any(f.any() for f in be.first)       # every block took at least one update

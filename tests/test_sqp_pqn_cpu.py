"""CPU tests of the partitioned damped BFGS mode of the native solver (hessian_approximation = "partitioned-bfgs"): the knot
chain (host-only queries of libdto.so) against a numpy construction, the KKT orderings it gives, its refusals, the partition of
the Lagrangian's gradient into knot elements (`sqp.knot_elements`), the chain assembly, and the oracle-driven twin of the mode
-- `sqp.solve` with H assembled from element blocks that the twin updates with `sqp.knot_bfgs_update` -- which the GPU tests
hold the native solver to."""
import numpy as np
import pytest

import dto_b200 as D
from dto_b200 import _lib
from dto_b200 import kkt as PK
from dto_b200 import sqp
from examples import models as M
from oracle import api as O

from band_models import band_kwargs, build_band
from sqp_oracle import OracleBackend

XP = sqp._XP(np)

# a chain KKT matrix of half bandwidth 31 whose elements have 22 variables (k_pqn_update with 32 lanes)
PQN_BAND = (10, 2, 9, False)


class PQNOracleBackend(OracleBackend):
    """OracleBackend whose H is the knot chain (nlp.hessian_chain_structure()) assembled from element blocks that are updated
    in `callbacks` -- after the callbacks, before the right-hand side, with the multipliers as they stand and g before any
    barrier term: where the native solver's k_pqn_update runs. No Hessian is evaluated."""

    def __init__(self, osolver, pnlp, B, **kw):
        super().__init__(osolver, B, **kw)
        r, c = (v - 1 for v in pnlp.hessian_chain_structure())
        up = r < c                                          # the coupling part lists only its upper copy: mirror it for K
        self._mirror = up
        jr, jc, _, _ = self._idx
        self._idx = (jr, jc, np.concatenate([r, c[up]]), np.concatenate([c, r[up]]))
        self.elements = sqp.knot_elements(pnlp)
        self.blocks = [np.tile(np.eye(m), (B, 1, 1)) for _, _, m, _ in self.elements]
        self.first = [np.ones(B, dtype=bool) for _ in self.elements]
        self.prev = None

    def _dense(self, J):
        jr, jc, _, _ = self._idx
        Jd = np.zeros((J.shape[0], self.N_c, self.N_z))
        Jd[:, jr, jc] = J
        return Jd

    def callbacks(self, z, lam, lam_hess, delta=None, diag=None, gshift=None, cshift=None):
        cur = self._eval(z, lam, 1 | 2 | 4 | 8)
        g, J = cur["g"], cur["J"]
        if self.prev is not None:
            zp, gp, Jp = self.prev
            now = sqp.element_gradients(self.elements, g, self._dense(J), lam)
            before = sqp.element_gradients(self.elements, gp, self._dense(Jp), lam)
            for k, (v0, _, m, _) in enumerate(self.elements):
                self.blocks[k], self.first[k] = sqp.knot_bfgs_update(XP, self.blocks[k], z[:, v0:v0 + m] - zp[:, v0:v0 + m], now[k] - before[k],
                                                                     self.free[v0:v0 + m], self.first[k])
        self.prev = (z.copy(), g.copy(), J.copy())
        H = sqp.chain_from_elements(self.elements, self.blocks)
        cur["H"] = np.concatenate([H, H[:, self._mirror]], axis=1)
        self.cur = cur
        self.lam = lam.copy()
        self.diag = None if diag is None else np.array(diag, copy=True)
        if gshift is not None:
            self.cur["g"] = self.cur["g"] + gshift
        c_raw = self.cur["c"].copy()
        if cshift is not None:
            self.cur["c"] = self.cur["c"] + cshift
        return self.cur["f"].copy(), self.cur["g"].copy(), c_raw


def _build(name, kw):
    if name == "band":
        return build_band(O, **kw), build_band(D, **kw)
    return M.BUILDERS[name](O, evaluate_hessian=False, **kw), M.BUILDERS[name](D, evaluate_hessian=False, **kw)


def pqn_twin(name, kw, B, opts):
    """(product model, product nlp, twin backend) of model `name` built without Hessians"""
    mo, mp = _build(name, kw)
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    perm, bw = PK.analyze(pn, hessian="knot-chain")
    be = PQNOracleBackend(osolver, pn, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band", options=opts)
    return mp, pn, be


def guess(model, B, seed):
    T, n, m = model["T"], model["n"], model["m"]
    rng = np.random.default_rng(seed)
    z = np.zeros((B, T * n + (T - 1) * m))
    for t in range(T):
        o = t * (n + m)
        z[:, o:o + n] = model["x1"] + (model["xT"] - model["x1"]) * t / (T - 1)
        if t < T - 1:
            z[:, o + n:o + n + m] = rng.normal(size=(B, m))
    return z


CHAIN_SHAPES = [("pendulum", dict()), ("cartpole", dict(T=11)), ("acrobot", dict(T=9)), ("car", dict(T=12, obstacle="general")),
                ("car", dict(T=7, obstacle="stage")), ("heterogeneous", dict())]
EXAMPLES = [("pendulum", dict()), ("cartpole", dict(T=11, parameterized=False)), ("acrobot", dict(T=9)), ("car", dict(T=7, obstacle="stage"))]


@pytest.mark.parametrize("name,kw", CHAIN_SHAPES)
def test_chain_structure_is_one_row_block_per_knot(name, kw):
    pn = D.solver_from(M.BUILDERS[name](D, evaluate_hessian=False, **kw), batch=1).nlp
    r, c = pn.hessian_chain_structure()
    xs, nx, _, nu = pn.knot_layout()
    want = []
    for t in range(pn.T):
        o, n = int(xs[t]), int(nx[t] + nu[t])
        m = n + (int(nx[t + 1]) if t + 1 < pn.T else 0)
        want += [(o + i, o + j) for i in range(n) for j in range(m)]
    assert list(zip(r.tolist(), c.tolist())) == want == sorted(want)
    assert int(_lib.lib().dto_hessian_chain_count(pn.shape)) == len(want)
    # the diagonal part lists both triangles, the coupling part (columns x_{t+1}) its upper copy only
    pairs = set(want)
    assert all((j, i) in pairs for i, j in want if i > j)
    coupling = [(i, j) for t in range(pn.T - 1) for i, j in want if i < int(xs[t + 1]) <= j and i >= int(xs[t])]
    assert coupling and not any((j, i) in pairs for i, j in coupling)


@pytest.mark.parametrize("name,kw", [("pendulum", dict()), ("cartpole", dict(T=101)), ("acrobot", dict(T=101)),
                                     ("car", dict(T=51, obstacle="general")), ("car", dict(T=51, obstacle="stage"))])
def test_chain_mode_ordering_fits_the_banded_factorisation(name, kw):
    pn = D.solver_from(M.BUILDERS[name](D, evaluate_hessian=False, **kw), batch=1).nlp
    perm, bw = PK.analyze(pn, hessian="knot-chain")
    _, bw_blocks = PK.analyze(pn, hessian="knot-blocks")
    print(f"{name} {kw}: half bandwidth knot-chain {bw}, knot-blocks {bw_blocks}")
    assert bw_blocks <= bw <= 15                     # 16-lane rows of the factor kernel, as in the other modes
    assert sorted(perm.tolist()) == list(range(1, pn.num_variables + pn.num_constraint + 1))


def test_element_of_more_than_32_variables_is_unsupported():
    n, m = 16, 1                                  # elements of 16 + 1 + 16 = 33 variables
    x1 = np.zeros(n)
    dt = D.Dynamics(lambda y, x, u, w: y - (x + 0.1 * u[0]), n, n, m)
    ct = D.Cost(lambda x, u, w: sum(x[i] * x[i] for i in range(n)) + u[0] * u[0], n, m)
    cT = D.Cost(lambda x, u, w: sum(x[i] * x[i] for i in range(n)), n, 0)
    s = D.Solver([dt] * 2, [ct, ct, cT], [D.Constraint(lambda x, u, w: x - x1, n, m), D.Constraint(), D.Constraint()],
                 [D.Bound(n, m), D.Bound(n, m), D.Bound(n, 0)], name="wide33")
    with pytest.raises(_lib.DtoError) as e:
        PK.analyze(s.nlp, hessian="knot-chain")
    assert e.value.status == -7 and "at most 32" in str(e.value)
    PK.analyze(s.nlp)                             # the exact mode's analysis is not affected


def test_chain_bandwidth_over_31_is_unsupported():
    pn = D.solver_from(build_band(D, **band_kwargs((11, 2, 4, True)), evaluate_hessian=False), batch=1).nlp
    assert max(m for _, _, m, _ in sqp.knot_elements(pn)) == 24      # elements fit in 32 lanes ...
    with pytest.raises(_lib.DtoError) as e:
        PK.analyze(pn, hessian="knot-chain")                           # ... the ordered band does not
    assert e.value.status == -7 and "31" in str(e.value)
    _, bw = PK.analyze(pn)
    assert bw == 31


def test_general_constraint_has_no_knot_elements():
    pn = D.solver_from(M.build_car(D, T=12, obstacle="general", evaluate_hessian=False), batch=2).nlp
    with pytest.raises(ValueError, match="general constraint"):
        sqp.knot_elements(pn)
    perm, bw = PK.analyze(pn, hessian="knot-chain")     # the KKT layer takes the shape; the solver refuses it (GPU tests)
    assert bw <= 31


def _oracle_point(osolver, z):
    o = osolver.nlp
    B = z.shape[0]
    g = np.zeros((B, o.num_variables))
    J = np.zeros((B, len(o.jacobian_structure())))
    for b in range(B):
        o.eval_objective_gradient(g[b], z[b])
        o.eval_constraint_jacobian(J[b], z[b])
    return g, J


@pytest.mark.parametrize("name,kw", EXAMPLES)
def test_element_secant_pairs_partition_the_lagrangian_gradient_change(name, kw):
    """scattering every element's y_t back by P_t' and summing gives the knot-bfgs mode's (g + J'lam) difference"""
    mo, mp = _build(name, kw)
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=1).nlp
    jr, jc = (v - 1 for v in pn.jacobian_structure_arrays())
    assert [(r + 1, c + 1) for r, c in zip(jr.tolist(), jc.tolist())] == list(osolver.nlp.jacobian_structure())
    el = sqp.knot_elements(pn)
    rows = np.concatenate([r for *_, r in el])
    assert sorted(rows.tolist()) == sorted(set(jr.tolist()))            # every row with a Jacobian entry has one owner
    assert el[0][0] == 0 and all(el[t + 1][0] == el[t][0] + el[t][1] for t in range(len(el) - 1))
    rng = np.random.default_rng(11)
    B, N_z, N_c = 3, pn.num_variables, pn.num_constraint
    z, zp = guess(mp, B, 1) + 0.1 * rng.normal(size=(B, N_z)), guess(mp, B, 2)
    lam = rng.normal(size=(B, N_c))
    (g, J), (gp, Jp) = _oracle_point(osolver, z), _oracle_point(osolver, zp)
    Jd, Jpd = np.zeros((B, N_c, N_z)), np.zeros((B, N_c, N_z))
    Jd[:, jr, jc], Jpd[:, jr, jc] = J, Jp
    full = (g + np.einsum("bij,bi->bj", Jd, lam)) - (gp + np.einsum("bij,bi->bj", Jpd, lam))
    y = [a - b for a, b in zip(sqp.element_gradients(el, g, Jd, lam), sqp.element_gradients(el, gp, Jpd, lam))]
    summed = np.zeros((B, N_z))
    for (v0, _, m, _), yt in zip(el, y):
        summed[:, v0:v0 + m] += yt
    assert np.allclose(summed, full, rtol=1e-12, atol=1e-12 * max(1.0, np.abs(full).max()))


@pytest.mark.parametrize("name,kw", EXAMPLES)
def test_chain_assembly_is_the_sum_of_the_element_blocks(name, kw):
    pn = D.solver_from(M.BUILDERS[name](D, evaluate_hessian=False, **kw), batch=1).nlp
    el = sqp.knot_elements(pn)
    rng = np.random.default_rng(3)
    B, N_z = 2, pn.num_variables
    blocks = []
    for _, _, m, _ in el:
        A = rng.normal(size=(B, m, m))
        blocks.append(A @ A.transpose(0, 2, 1) + m * np.eye(m))
    H = np.zeros((B, N_z, N_z))
    for (v0, _, m, _), Bt in zip(el, blocks):
        H[:, v0:v0 + m, v0:v0 + m] += Bt
    chain = sqp.chain_from_elements(el, blocks)
    r, c = (v - 1 for v in pn.hessian_chain_structure())
    assert chain.shape == (B, len(r))
    K = np.zeros((B, N_z, N_z))
    K[:, r, c] = chain
    K[:, c, r] = chain
    assert np.array_equal(K, H)


def _twin_solve(name, kw, B, iters, **okw):
    opts = sqp.SQPOptions(max_iter=iters, dual_reg=1.0e-6, **okw)
    mp, pn, be = pqn_twin(name, kw, B, opts)
    res = sqp.solve(be, guess(mp, B, 5), options=opts)
    return mp, be, res


def test_oracle_twin_converges_on_pendulum_without_hessians():
    mp, be, res = _twin_solve("pendulum", dict(), 3, 150)
    print("pendulum twin iterations", res.iterations)
    assert res.converged.all(), res.iterations
    assert np.all(res.constraint_violation <= 1e-8)
    assert not any(f.any() for f in be.first)       # every element block took at least one update


def test_oracle_twin_on_acrobot_without_hessians():
    """runs (whether it converges is measured on the device: DESIGN 10(c)); every element block takes updates"""
    mp, be, res = _twin_solve("acrobot", dict(T=9), 3, 60)
    print("acrobot T=9 twin iterations", res.iterations, "converged", res.converged)
    assert np.all(np.isfinite(res.z)) and np.all(res.constraint_violation < 1.0)
    assert not any(f.any() for f in be.first)


def test_oracle_twin_interior_point_on_bounded_pendulum():
    mp, be, res = _twin_solve("pendulum", dict(u_bnd=15.0), 3, 150)
    print("bounded pendulum twin iterations", res.iterations, "converged", res.converged)
    n, m, T = mp["n"], mp["m"], mp["T"]
    U = np.stack([res.z[:, t * (n + m) + n] for t in range(T - 1)], axis=1)
    assert np.all(np.abs(U) < 15.0) and res.converged.any()

"""GPU parity of the device-resident KKT consumer (SURVEY 8f N3), through the C ABI (dto_kkt_*):

  * assembled K and h: BIT-EXACT against the oracle's assembly (pendulum.jl:138-199 restated) fed
    with the very g, c, J, H the GPU callbacks produced (pure copies, one add per diagonal entry, and
    the script's ascending-row sum for C'y), and within 1e-12 of the all-oracle K, h;
  * factor: P K P' = L D L' to 1e-12 relative (normwise), pivots' inertia (N_z positive, N_c
    negative where K is quasi-definite; always the oracle's pivot signs), and L, D against the oracle's QDLDL restatement in the same ordering;
  * solution: normwise backward error <= 1e-13, and forward error against the oracle's solve within
    cond(K)-scaled rounding (the systems are regularised with 1e-5, cond ~ 1e6..1e9, so a fixed
    1e-12 on the solution would not be meaningful; with regularisation 1e-2 the test uses 1e-9).
"""
import numpy as np
import pytest

import dto_b200 as D
from dto_b200 import kkt as PK
from examples import models as M
from oracle import api as O
from oracle import kkt as OK

from util import assert_close, make_inputs, oracle_parameters

pytestmark = pytest.mark.gpu

CASES = [
    ("pendulum", dict(), 5, 1),
    ("cartpole", dict(T=11), 37, 2),
    ("acrobot", dict(T=9), 6, 3),
    ("car", dict(T=12, obstacle="general"), 4, 4),
    ("car", dict(T=7, obstacle="stage"), 3, 4),
    ("acrobot_hessian_test", dict(), 5, 6),   # half bandwidth 19 -> 32-wide rows
    ("linear_general", dict(), 3, 7),
]


def _setup(name, kw, B, config):
    mo = M.BUILDERS[name](O, **kw)
    mp = M.BUILDERS[name](D, **kw)
    osolver = O.solver_from(mo)
    pn = D.solver_from(mp, batch=B).nlp
    z, lam, sigma, w = make_inputs(name, mp, pn.num_variables, pn.num_constraint, pn.num_parameter, B, config)
    sigma = np.ones(B)  # the script evaluates the Hessian with sigma = 1.0 (pendulum.jl:136)
    if pn.num_parameter:
        pn.set_parameters(w)
    return mo, osolver, pn, z, lam, sigma, w


@pytest.mark.parametrize("name,kw,B,config", CASES, ids=[f"{c[0]}-{i}" for i, c in enumerate(CASES)])
@pytest.mark.parametrize("reg", [1.0e-5, 1.0e-2])
def test_kkt_matches_oracle(name, kw, B, config, reg):
    mo, osolver, pn, z, lam, sigma, w = _setup(name, kw, B, config)
    on = osolver.nlp
    nz, ny = pn.num_variables, pn.num_constraint
    n = nz + ny
    kkt = PK.KKTSystem(pn, primal_reg=reg, dual_reg=reg)
    assert kkt.dim == n and kkt.bandwidth < kkt.row_width
    perm = kkt.permutation() - 1
    assert sorted(perm.tolist()) == list(range(n))
    sol = np.full((B, n), np.nan)
    kkt.solve(sol, variables=z, scaling=sigma, duals=lam)
    h = kkt.rhs()
    assert np.array_equal(kkt.solution(), sol)
    # the callback outputs the solve consumed
    g = np.empty((B, nz)); c = np.empty((B, ny)); J = np.empty((B, pn.num_jacobian)); H = np.empty((B, pn.num_hessian))
    pn.eval_objective_gradient(g); pn.eval_constraint(c); pn.eval_jacobian_hessian(J, H)
    js, hs = pn.jacobian_structure(), pn.hessian_lagrangian_structure()
    for b in range(B):
        Kg, hg = OK.assemble(nz, ny, js, hs, g[b], c[b], J[b], H[b], lam[b], reg, reg)
        Kd = kkt.matrix(b)
        assert np.array_equal(Kd, Kg), f"problem {b}: assembled K differs from the oracle assembly of the same J, H"
        assert np.array_equal(h[b], hg), f"problem {b}: right-hand side differs (max {np.max(np.abs(h[b] - hg)):.3e})"
        # all-oracle reference
        p = oracle_parameters(mo, w[b])
        if p is not None:
            osolver.set_parameters(p)
        ref = OK.kkt_solve(on, z[b], lam[b], reg, reg, perm)
        assert_close(f"K[{b}]", Kd, ref["K"])
        assert_close(f"h[{b}]", h[b], ref["h"], rtol=1e-12, atol=1e-13)
        # factor
        Lm, Dv = kkt.factor(b)
        Kp = Kd[np.ix_(perm, perm)]
        scale = np.max(np.abs(Kp))
        growth = max(1.0, np.max(np.abs(Lm)) ** 2 * np.max(np.abs(Dv)) / scale)
        assert np.max(np.abs(Lm @ np.diag(Dv) @ Lm.T - Kp)) <= 1e-13 * scale * growth * kkt.row_width
        # inertia (Sylvester): the pivots' signs match the oracle factor's and the eigenvalues' signs. K is
        # quasi-definite (nz positive, ny negative pivots) only where H + primal_reg I is positive definite,
        # which random multipliers do not guarantee -- the reference script has the same caveat
        assert np.array_equal(Dv > 0, ref["D"] > 0)
        ev = np.linalg.eigvalsh(Kd)
        assert int((Dv > 0).sum()) == int((ev > 0).sum())
        cond = np.linalg.cond(Kd)
        tol = 50 * cond * np.finfo(float).eps
        assert np.max(np.abs(Dv - ref["D"]) / np.abs(ref["D"])) <= tol
        assert np.max(np.abs(Lm - ref["L"])) <= tol * max(1.0, np.max(np.abs(ref["L"])))
        # solution: backward error, then forward error vs the oracle solve
        x = sol[b]
        resid = np.max(np.abs(Kd @ x - h[b]))
        assert resid <= 1e-13 * growth * (np.linalg.norm(Kd, np.inf) * np.max(np.abs(x)) + np.max(np.abs(h[b])))
        assert np.max(np.abs(x - ref["sol"])) <= tol * max(1.0, np.max(np.abs(ref["sol"])))
        if reg == 1.0e-2 and cond < 1e6:
            assert np.max(np.abs(x - ref["sol"])) <= 1e-9 * max(1.0, np.max(np.abs(ref["sol"])))
    kkt.close()
    pn.close()


def test_kkt_matches_golden_fixtures():
    """Product vs the committed fixtures tests/golden/kkt_*.npz (oracle outputs frozen by
    make_golden_kkt.py): K and h to 1e-12, solution within cond-scaled rounding of the fixture's pivoted-LU reference."""
    import os
    from golden.make_golden import tag
    from golden.make_golden_kkt import KKT_GOLDEN, REG
    here = os.path.join(os.path.dirname(__file__), "golden")
    for name, kw, _ in KKT_GOLDEN:
        fx = np.load(os.path.join(here, tag(name, kw) + ".npz"))
        gk = np.load(os.path.join(here, "kkt_" + tag(name, kw) + ".npz"))
        B = fx["z"].shape[0]
        pn = D.solver_from(M.BUILDERS[name](D, **kw), batch=B).nlp
        if pn.num_parameter:
            pn.set_parameters(fx["w"])
        kkt = PK.KKTSystem(pn, REG, REG)
        sol = np.empty((B, kkt.dim))
        kkt.solve(sol, variables=fx["z"], scaling=np.ones(B), duals=fx["lam"])
        h = kkt.rhs()
        for b in range(B):
            assert_close(f"{name} K[{b}]", kkt.matrix(b), gk["K"][b])
            assert_close(f"{name} h[{b}]", h[b], gk["h"][b], rtol=1e-12, atol=1e-13)
            # solution: against the fixture's pivoted-LU + refinement solution (`sol_lu`; the fixture's own
            # natural-ordering QDLDL solution `sol` is off by up to 5e-7 on the acrobot systems, which are
            # not quasi-definite for random multipliers), scaled by cond(K); and by backward error
            Kf, hf, xf = gk["K"][b], gk["h"][b], gk["sol_lu"][b]
            be = np.max(np.abs(Kf @ sol[b] - hf)) / (np.linalg.norm(Kf, np.inf) * np.max(np.abs(sol[b])) + np.max(np.abs(hf)))
            assert be <= 1e-11, f"{name}[{b}]: backward error {be:.3e}"
            cond = np.linalg.cond(Kf)
            fe = np.max(np.abs(sol[b] - xf)) / max(1.0, np.max(np.abs(xf)))
            assert fe <= 1e3 * cond * np.finfo(float).eps, f"{name}[{b}]: forward error {fe:.3e}, cond {cond:.3e}"
        kkt.close()
        pn.close()


def test_kkt_full_size_properties():
    """cartpole T=101, B=512: every problem's solution satisfies K x = h to rounding (K rebuilt on the
    host from the GPU's J, H), results do not depend on sharding, a second solve is bit-identical, and a
    solve enqueues two KKT kernels (right-hand side, factor) on top of the callbacks."""
    import scipy.sparse as sp

    name, kw, B = "cartpole", dict(T=101), 512
    mo, osolver, pn, z, lam, sigma, w = _setup(name, kw, B, 2)
    nz, ny = pn.num_variables, pn.num_constraint
    n = nz + ny
    kkt = PK.KKTSystem(pn)
    sol = np.empty((B, n))
    kkt.solve(sol, variables=z, scaling=sigma, duals=lam)
    h = kkt.rhs()
    J = np.empty((B, pn.num_jacobian)); H = np.empty((B, pn.num_hessian)); g = np.empty((B, nz)); c = np.empty((B, ny))
    pn.eval_jacobian_hessian(J, H); pn.eval_objective_gradient(g); pn.eval_constraint(c)
    jr, jc = pn.jacobian_structure_arrays()
    hr, hc = pn.hessian_lagrangian_structure_arrays()
    rows = np.concatenate([hr - 1, nz + jr - 1, jc - 1, np.arange(n)])
    cols = np.concatenate([hc - 1, jc - 1, nz + jr - 1, np.arange(n)])
    diag = np.concatenate([np.full(nz, 1e-5), np.full(ny, -1e-5)])
    worst = 0.0
    for b in range(0, B, 7):
        K = sp.csr_matrix((np.concatenate([H[b], J[b], J[b], diag]), (rows, cols)), shape=(n, n))
        Jm = sp.csr_matrix((J[b], (jr - 1, jc - 1)), shape=(ny, nz))
        hb = np.concatenate([g[b] + Jm.T @ lam[b], c[b]])
        assert np.allclose(h[b], hb, rtol=1e-13, atol=1e-13)
        x = sol[b]
        be = np.max(np.abs(K @ x - h[b])) / (abs(K).sum(axis=1).max() * np.max(np.abs(x)) + np.max(np.abs(h[b])))
        worst = max(worst, be)
    assert worst <= 1e-12, f"normwise backward error {worst:.3e}"
    sol2 = np.empty((B, n))
    l0 = pn.launch_count()
    kkt.solve(sol2)
    solve_launches = pn.launch_count() - l0
    assert np.array_equal(sol, sol2)
    l0 = pn.launch_count()
    kkt.launch(2)                                   # the same callbacks alone
    pn.sync()
    assert solve_launches - (pn.launch_count() - l0) == 2
    kkt.close()
    pn.close()
    # two logical shards on the one device: same bits
    pn2 = D.solver_from(M.BUILDERS[name](D, **kw), batch=B, devices=[0, 0]).nlp
    pn2.set_parameters(w)
    k2 = PK.KKTSystem(pn2)
    sol3 = np.empty((B, n))
    k2.solve(sol3, variables=z, scaling=sigma, duals=lam)
    assert np.array_equal(sol, sol3)
    k2.close()
    pn2.close()


def test_kkt_heterogeneous_shape():
    """Per-knot dims / element kinds / parameter lengths differ and a nonlinear GeneralConstraint couples
    distant knots (half bandwidth 17 -> the 32-lane kernel): K and h bit-exact against the oracle
    assembly of the GPU's own g, c, J, H; factor and solution by backward error."""
    mp = M.build_heterogeneous(D)
    B = 9
    r = np.random.default_rng(5)
    pn = D.Solver(mp["dynamics"], mp["objective"], mp["constraints"], mp["bounds"], evaluate_hessian=True,
                  general_constraint=mp["general"], batch=B, name="heterogeneous").nlp
    nz, ny = pn.num_variables, pn.num_constraint
    n = nz + ny
    z = r.uniform(-1, 1, (B, nz)); lam = r.normal(size=(B, ny)); w = r.uniform(-1, 1, (B, pn.num_parameter))
    pn.set_parameters(w)
    kkt = PK.KKTSystem(pn, 1e-3, 1e-3)
    assert kkt.row_width == 32 and 15 < kkt.bandwidth < 32
    sol = np.empty((B, n))
    kkt.solve(sol, variables=z, scaling=np.ones(B), duals=lam)
    h = kkt.rhs()
    g = np.empty((B, nz)); c = np.empty((B, ny)); J = np.empty((B, pn.num_jacobian)); H = np.empty((B, pn.num_hessian))
    pn.eval_objective_gradient(g); pn.eval_constraint(c); pn.eval_jacobian_hessian(J, H)
    perm = kkt.permutation() - 1
    for b in range(B):
        Kg, hg = OK.assemble(nz, ny, pn.jacobian_structure(), pn.hessian_lagrangian_structure(), g[b], c[b], J[b], H[b], lam[b], 1e-3, 1e-3)
        Kd = kkt.matrix(b)
        assert np.array_equal(Kd, Kg) and np.array_equal(h[b], hg)
        Lm, Dv = kkt.factor(b)
        Kp = Kd[np.ix_(perm, perm)]
        growth = max(1.0, np.max(np.abs(Lm)) ** 2 * np.max(np.abs(Dv)) / np.max(np.abs(Kp)))
        assert np.max(np.abs(Lm @ np.diag(Dv) @ Lm.T - Kp)) <= 1e-13 * np.max(np.abs(Kp)) * growth * 32
        x = sol[b]
        assert np.max(np.abs(Kd @ x - h[b])) <= 1e-13 * growth * (np.linalg.norm(Kd, np.inf) * np.max(np.abs(x)) + np.max(np.abs(h[b])))
    kkt.close()
    pn.close()


def test_kkt_two_devices():
    """Row (e): problems are independent, a shard per device, no collective -- the KKT consumer follows the
    batch's shards. Needs 2 GPUs (skipped on a 1-GPU box; run with `gpurun --gpus 2`)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 CUDA devices")
    _two_device_case("cartpole", dict(T=101), 301, 2)
    _two_device_case("acrobot", dict(T=9), 70, 3)     # half bandwidth 14: > 48 KB shared memory, opt-in per device


def _two_device_case(name, kw, B, config):
    mo, osolver, pn, z, lam, sigma, w = _setup(name, kw, B, config)
    k1 = PK.KKTSystem(pn)
    sol1 = np.empty((B, k1.dim))
    k1.solve(sol1, variables=z, scaling=sigma, duals=lam)
    k1.close(); pn.close()
    pn2 = D.solver_from(M.BUILDERS[name](D, **kw), batch=B, devices=[0, 1]).nlp
    if pn2.num_parameter:
        pn2.set_parameters(w)
    k2 = PK.KKTSystem(pn2)
    sol2 = np.empty((B, k2.dim))
    k2.solve(sol2, variables=z, scaling=sigma, duals=lam)
    assert np.array_equal(sol1, sol2)
    sol3 = np.empty_like(sol2)
    k2.solve(sol3)                      # resident path on both devices
    assert np.array_equal(sol1, sol3)
    k2.close(); pn2.close()


def test_kkt_nan_and_singular_pass_through():
    """Reference behaviour: non-finite values are passed on unchecked (SURVEY 8b). A NaN in one problem's
    z makes that problem's solution non-finite and leaves the other problems' solutions bit-identical; a
    zero pivot (no regularisation, all-zero multipliers and a zero Hessian block) produces Inf/NaN, no hang."""
    name, kw, B = "pendulum", dict(), 6
    mo, osolver, pn, z, lam, sigma, w = _setup(name, kw, B, 1)
    kkt = PK.KKTSystem(pn)
    sol = np.empty((B, kkt.dim))
    kkt.solve(sol, variables=z, scaling=sigma, duals=lam)
    z2 = z.copy()
    z2[3, 5] = np.nan
    sol2 = np.empty_like(sol)
    kkt.solve(sol2, variables=z2, scaling=sigma, duals=lam)
    assert not np.all(np.isfinite(sol2[3]))
    keep = [b for b in range(B) if b != 3]
    assert np.array_equal(sol2[keep], sol[keep])
    kkt.close()
    k0 = PK.KKTSystem(pn, primal_reg=0.0, dual_reg=0.0)
    sol3 = np.empty_like(sol)
    k0.solve(sol3, variables=z, scaling=sigma, duals=lam)   # must return (finite or not), never hang
    assert sol3.shape == sol.shape
    k0.close()
    pn.close()


def test_kkt_state_errors():
    pn = D.solver_from(M.BUILDERS["pendulum"](D), batch=2).nlp
    kkt = PK.KKTSystem(pn)
    with pytest.raises(Exception):
        kkt.solution()          # nothing solved yet
    with pytest.raises(Exception):
        kkt.solve(np.empty((2, kkt.dim)))  # no z resident
    kkt.close()
    pn.close()


def test_per_problem_regularisation_inertia_and_subset_launch():
    """Solver hooks of the KKT consumer: (i) a per-problem primal regularisation array replaces the scalar, problem by
    problem (checked against the assembled matrix and a dense solve); (ii) the negative-pivot count of D equals the
    number of negative eigenvalues of K (Sylvester), also when the Hessian block is made indefinite; (iii)
    dto_kkt_launch_subset re-factors only the selected problems and leaves every other problem's solution, factor
    and pivot count bit-identical."""
    import torch
    name, kw, B = "cartpole", dict(T=11), 23
    mo, osolver, pn, z, lam, sigma, w = _setup(name, kw, B, 2)
    kkt = PK.KKTSystem(pn, primal_reg=0.0, dual_reg=1.0e-6)
    dev = torch.device("cuda", pn.shard_device(0))
    reg = np.linspace(1.0e-3, 2.0, B)
    kkt.set_primal_reg(reg)
    sol = np.empty((B, kkt.dim))
    kkt.solve(sol, variables=z, scaling=sigma, duals=10.0 * lam)       # large multipliers: indefinite Hessian blocks
    nneg = kkt.inertia()
    h = kkt.rhs()
    N_z = pn.num_variables
    for b in (0, 7, B - 1):
        K = kkt.matrix(b)
        assert np.allclose(np.diag(K)[:N_z] - np.diag(kkt_matrix_without_reg(kkt, pn, b, reg[b]))[:N_z], reg[b], rtol=1e-12, atol=1e-14)
        assert nneg[b] == int((np.linalg.eigvalsh(K) < 0).sum())
        ref = np.linalg.solve(K, h[b])
        assert np.max(np.abs(sol[b] - ref)) <= 1e-6 * max(1.0, np.max(np.abs(ref)))
    # the chunk-pipelined host call cuts the shard into sub-batches: the per-problem arrays must follow the chunks
    sol_c = np.empty_like(sol)
    kkt.solve(sol_c, variables=z, scaling=sigma, duals=10.0 * lam, chunks=5)
    assert np.array_equal(sol_c, sol) and np.array_equal(kkt.inertia(), nneg)
    # subset: new regularisation for three problems only
    pick = np.array([2, 11, 19], dtype=np.int32)
    reg2 = reg.copy()
    reg2[pick] = 50.0
    sol_before, nneg_before = kkt.solution(), kkt.inertia()
    kkt.set_primal_reg(reg2)
    idx = torch.as_tensor(pick, device=dev)
    kkt.launch_subset(idx.data_ptr(), len(pick))
    pn.sync()
    sol_after, nneg_after = kkt.solution(), kkt.inertia()
    keep = np.setdiff1d(np.arange(B), pick)
    assert np.array_equal(sol_after[keep], sol_before[keep]) and np.array_equal(nneg_after[keep], nneg_before[keep])
    kkt.launch(False)                                   # everything with reg2: the picked rows must agree bit for bit
    pn.sync()
    sol_full = kkt.solution()
    assert np.array_equal(sol_full[pick], sol_after[pick]) and np.array_equal(sol_full[keep], sol_before[keep])
    assert np.all(kkt.inertia()[pick] == pn.num_constraint)            # +50 on the diagonal: quasi-definite
    kkt.close()
    pn.close()


def kkt_matrix_without_reg(kkt, pn, b, reg_b):
    K = kkt.matrix(b).copy()
    K[np.arange(pn.num_variables), np.arange(pn.num_variables)] -= reg_b
    return K


def test_pinned_variables_get_identity_rows():
    """dto_kkt_set_fixed: variables pinned by equal bounds -- K's rows and columns of those variables are the identity,
    their right-hand-side entries zero; the solve returns exactly 0 for them and the reduced system's solution for the
    rest (dense reference); un-pinning restores the full system."""
    name, kw, B = "acrobot", dict(T=9), 5
    mo, osolver, pn, z, lam, sigma, w = _setup(name, kw, B, 3)
    kkt = PK.KKTSystem(pn, primal_reg=1.0e-3, dual_reg=1.0e-3)
    N_z = pn.num_variables
    full = np.empty((B, kkt.dim))
    kkt.solve(full, variables=z, scaling=sigma, duals=lam)
    K0, h0 = kkt.matrix(2), kkt.rhs()[2]
    fixed = np.zeros(N_z, dtype=bool)
    fixed[[0, 1, 2, 3, N_z - 4, N_z - 2]] = True
    kkt.set_fixed(fixed)
    sol = np.empty((B, kkt.dim))
    kkt.solve(sol, variables=z, scaling=sigma, duals=lam)
    K1, h1 = kkt.matrix(2), kkt.rhs()[2]
    fx = np.nonzero(fixed)[0]
    Kref, href = K0.copy(), h0.copy()
    Kref[fx, :] = 0.0
    Kref[:, fx] = 0.0
    Kref[fx, fx] = 1.0
    href[fx] = 0.0
    assert np.array_equal(K1, Kref) and np.array_equal(h1, href)
    assert np.all(sol[:, fx] == 0.0)
    ref = np.linalg.solve(Kref, href)
    assert np.max(np.abs(sol[2] - ref)) <= 1e-9 * max(1.0, np.max(np.abs(ref)))
    kkt.set_fixed(None)
    again = np.empty_like(full)
    kkt.solve(again, variables=z, scaling=sigma, duals=lam)
    assert np.array_equal(again, full)
    kkt.close()
    pn.close()


@pytest.mark.parametrize("name,kw", [("cartpole", dict(T=11)), ("acrobot", dict(T=9)), ("car", dict(T=12, obstacle="general"))])
def test_resolve_with_stored_factor_is_bit_identical_to_refactorising(name, kw):
    """dto_kkt_resolve: K stays, the right-hand side changes (a second-order correction overwrites c on the device).
    Forward and backward solves with the stored factor must give the very bits of factorising again -- for the whole
    batch and for a problem list (the others keep their solution) -- and the dense solve of the assembled matrix."""
    import torch
    from dto_b200 import sqp
    from dto_b200.evaluator import A_C
    B = 19
    mo, osolver, pn, z, lam, sigma, w = _setup(name, kw, B, 2)
    kkt = PK.KKTSystem(pn, primal_reg=1.0e-2, dual_reg=1.0e-6)
    dev = torch.device("cuda", pn.shard_device(0))
    sol0 = np.empty((B, kkt.dim))
    kkt.solve(sol0, variables=z, scaling=sigma, duals=lam)
    nneg0 = kkt.inertia()
    N_c = pn.num_constraint
    d_c = torch.as_tensor(sqp._CudaArray(pn.device_pointer(A_C, 0), (B, N_c)), device=dev)
    stream = torch.cuda.ExternalStream(pn.stream_pointer(0), device=dev)
    rng = np.random.default_rng(8)
    c_new = torch.as_tensor(rng.normal(size=(B, N_c)), device=dev)
    with torch.cuda.stream(stream):
        c_old = d_c.clone()
        d_c.copy_(c_new)
    kkt.resolve()
    pn.sync()
    got = kkt.solution()
    kkt.launch(False)                       # factorise again with the new right-hand side
    pn.sync()
    ref = kkt.solution()
    assert np.array_equal(got, ref) and not np.array_equal(got, sol0)
    K, h = kkt.matrix(3), kkt.rhs()[3]
    dense = np.linalg.solve(K, h)
    assert np.max(np.abs(got[3] - dense)) <= 1e-6 * max(1.0, np.max(np.abs(dense)))
    # problem list: back to the old c for three problems only
    pick = np.array([1, 8, 17], dtype=np.int32)
    idx = torch.as_tensor(pick, device=dev)
    with torch.cuda.stream(stream):
        d_c[idx.long()] = c_old[idx.long()]
    kkt.resolve(idx.data_ptr(), len(pick))
    pn.sync()
    part = kkt.solution()
    keep = np.setdiff1d(np.arange(B), pick)
    assert np.array_equal(part[keep], ref[keep]) and np.array_equal(part[pick], sol0[pick])
    assert np.array_equal(kkt.inertia(), nneg0)      # the pivot counts are re-read from the stored factor, not changed
    kkt.close()
    pn.close()

"""Row N1 / BASELINE config 3: the lock-step batched Newton-KKT solver (dto_b200/sqp.py). The device arm
(callbacks, KKT assembly, banded LDL', trial evaluations: this package's CUDA kernels through the C ABI) must
walk through the same iterates as the very same algorithm driven by the CPU oracle (tests/sqp_oracle.py:
oracle callbacks + the oracle's banded LDL' in the product's ordering), and the full solves must meet the
reference's own acceptance (/root/reference/test/solve.jl:134-137). Ipopt itself is absent: its iterates are
NOT what is compared here (unverifiable), the algorithm is this repository's."""
import numpy as np
import pytest

import dto_b200 as D
from dto_b200 import kkt as PK
from dto_b200 import sqp
from examples import models as M
from oracle import api as O

from sqp_oracle import OracleBackend

pytestmark = pytest.mark.gpu


def _np(x):
    return x.detach().cpu().numpy() if hasattr(x, "detach") else np.asarray(x)


def _guess(model, B, seed):
    T, n, m = model["T"], model["n"], model["m"]
    rng = np.random.default_rng(seed)
    z = np.zeros((B, T * n + (T - 1) * m))
    for t in range(T):
        o = t * (n + m)
        z[:, o:o + n] = model["x1"] + (model["xT"] - model["x1"]) * t / (T - 1)
        if t < T - 1:
            z[:, o + n:o + n + m] = rng.normal(size=(B, m))
    return z


@pytest.mark.parametrize("name,kw,B,iters", [("pendulum", dict(), 4, 12), ("acrobot", dict(T=9), 3, 25), ("acrobot", dict(T=21), 2, 30)])
def test_device_iterates_match_oracle_driven_algorithm(name, kw, B, iters):
    import torch
    mo, mp = M.BUILDERS[name](O, **kw), M.BUILDERS[name](D, **kw)
    osolver, psolver = O.solver_from(mo), D.solver_from(mp, batch=B)
    pn = psolver.nlp
    z0 = _guess(mp, B, 5)
    # dual_reg = 1e-6 keeps cond(K) near 1e7: the two arms factor K in different operation orders, so intermediate
    # iterates can only agree to about cond(K) * eps; the converged objectives are then compared at 1e-8
    opts = sqp.SQPOptions(max_iter=iters, dual_reg=1.0e-6)
    perm, bw = PK.analyze(pn)
    ref = sqp.solve(OracleBackend(osolver, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band"), z0, options=opts, record=True)
    be = sqp.DeviceBackend(pn, dual_reg=opts.dual_reg)
    got = sqp.solve(be, torch.as_tensor(z0, device=be.xp.device), options=opts, record=True)
    be.close()
    assert len(got.history) == len(ref.history)
    for hg, hr in zip(got.history, ref.history):
        scale = np.maximum(1.0, np.abs(hr["z"]))
        assert np.max(np.abs(hg["z"] - hr["z"]) / scale) < 1e-7, (name, hg["it"])
        assert np.array_equal(hg["done"], hr["done"]), (name, hg["it"])
        assert np.allclose(hg["f"], hr["f"], rtol=1e-7, atol=1e-10), (name, hg["it"])
    both = got.converged.cpu().numpy() & ref.converged
    assert np.allclose(got.objective.cpu().numpy()[both], ref.objective[both], rtol=1e-8)
    pn.close()


def test_acrobot_full_solves_meet_reference_acceptance():
    """config 3 at a test-sized batch: >= 95 % of the seeded problems reach ||c||_inf < 1e-6 with both end points
    within 1e-3 (test/solve.jl:134-137); tools/solve_config3.py runs the full 4096."""
    import sys, os
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    import solve_config3
    out = solve_config3.run(B=256, T=101, max_iter=300)
    assert out["accepted_frac"] >= 0.95, out
    assert out["gpu_launches"] > 100


def test_solver_api_runs_sqp_on_device():
    """Solver.solve() (src/solver.jl:45-47) picks the device solver for an equality-constrained problem with exact
    Hessians; get_trajectory returns the final iterate (src/solver.jl:41-43)."""
    mp = M.build_pendulum(D)
    s = D.solver_from(mp, batch=5)
    s.initialize_states(D.linear_interpolation(mp["x1"], mp["xT"], mp["T"]))
    s.initialize_controls([np.array([0.1 * (t + 1)]) for t in range(mp["T"] - 1)])
    res = s.solve()
    assert bool(res.converged.all()) and s.sqp_launches > 0
    xs, us = s.get_trajectory(3)
    assert np.linalg.norm(xs[0] - mp["x1"]) < 1e-6 and np.linalg.norm(xs[-1] - mp["xT"]) < 1e-6 and len(us) == mp["T"] - 1
    s.nlp.close()


def test_repacking_on_the_device_changes_no_result():
    """Same property as tests/test_sqp_cpu.py on the device arm: a smaller batch of the same shape is created for the
    unconverged problems (parameters copied device to device, CUDA graph re-captured); final iterates are bit-identical
    to the run that keeps every problem in the batch. Half of the problems start at a solution so that they converge
    in the first iteration and the batch really shrinks."""
    import torch
    mp = M.BUILDERS["pendulum"](D)
    B = 12
    pn0 = D.solver_from(mp, batch=2).nlp
    be0 = sqp.DeviceBackend(pn0)
    first = sqp.solve(be0, torch.as_tensor(_guess(mp, 2, 9), device=be0.xp.device), options=sqp.SQPOptions(max_iter=200))
    assert bool(first.converged[0])
    zs, ls = first.z[0].cpu().numpy(), first.lam[0].cpu().numpy()
    be0.close(); pn0.close()
    z0 = _guess(mp, B, 10)
    lam0 = np.zeros((B, len(ls)))
    z0[::2], lam0[::2] = zs, ls
    out = {}
    for repack in (False, True):
        pn = D.solver_from(mp, batch=B).nlp
        be = sqp.DeviceBackend(pn)
        res = sqp.solve(be, torch.as_tensor(z0, device=be.xp.device), torch.as_tensor(lam0, device=be.xp.device),
                        options=sqp.SQPOptions(max_iter=120, repack=repack, repack_min=2))
        out[repack] = (res.z.cpu().numpy(), res.iterations.cpu().numpy(), res.converged.cpu().numpy(), res.backend.B, res.backend.total_launches())
        if res.backend is not be:
            res.backend.close()
        be.close()
        pn.close()
    assert out[True][3] < B == out[False][3]
    assert np.array_equal(out[True][2], out[False][2]) and np.array_equal(out[True][1], out[False][1])
    assert np.array_equal(out[True][0], out[False][0])
    assert out[True][4] > 0 and out[True][1][0] == 0


def test_reference_solve_tests_with_bound_pinned_end_points():
    """/root/reference/test/solve.jl verbatim problem set-ups: end points pinned by Bound(state_lower = x1,
    state_upper = x1) -- Ipopt removes such variables; here their rows/columns of K are the identity
    (dto_kkt_set_fixed) so their step is exactly zero. (i) :227-296 "general constraint": double integrator, x1 by
    bound, xT by a GeneralConstraint -- device iterates equal the oracle-driven twin's and meet the test's acceptance;
    (ii) :1-138 acrobot T=101 with both end points by bounds: >= 90 % of 64 seeded problems meet the acceptance."""
    import torch
    kw = dict(reference_exact=True)
    mo, mp = M.build_linear_general(O, **kw), M.build_linear_general(D, **kw)
    B = 4
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    z0 = _guess(mp, B, 21)
    perm, bw = PK.analyze(pn)
    opts = sqp.SQPOptions(max_iter=20, dual_reg=1.0e-6)
    ref = sqp.solve(OracleBackend(osolver, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band"), z0, options=opts, record=True)
    be = sqp.DeviceBackend(pn, dual_reg=opts.dual_reg)
    got = sqp.solve(be, torch.as_tensor(z0, device=be.xp.device), options=opts, record=True)
    be.close()
    assert bool(got.converged.all()) and ref.converged.all() and len(got.history) == len(ref.history)
    Z = got.z.cpu().numpy()
    assert np.allclose(Z, ref.z, rtol=1e-8, atol=1e-10)
    n = mp["n"]
    assert np.array_equal(Z[:, :n], np.tile(mp["x1"], (B, 1)))                       # pinned: exactly the bound
    assert np.all(np.linalg.norm(Z[:, -n:] - mp["xT"], axis=1) < 1e-3)               # test/solve.jl:294-295
    pn.close()
    # (ii) acrobot, end points by bounds
    ma = M.build_acrobot(D, T=101, stage_endpoint_constraints=False)
    B = 64
    s = D.solver_from(ma, batch=B)
    s.initialize_states(D.linear_interpolation(ma["x1"], ma["xT"], 101))
    rng = np.random.default_rng(4)
    for b in range(B):
        s.initialize_controls([rng.normal(size=1) for _ in range(100)], problem=b)
    res = s.solve(options=dict(max_iter=300), method="sqp")
    ok = 0
    for b in range(B):
        xs, _ = s.get_trajectory(b)
        ok += int(np.linalg.norm(xs[0] - ma["x1"]) < 1e-3 and np.linalg.norm(xs[-1] - ma["xT"]) < 1e-3 and float(res.constraint_violation[b]) < 1e-6)
    assert ok >= 0.9 * B, ok
    s.nlp.close()


# ----------------------------------------------------------------------------------------------------------------------
# native arm: dto_sqp_solve (csrc/dto_sqp_host.inc + dto_sqp.cu) -- the same algorithm inside libdto.so, no torch
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,kw,B,iters", [("pendulum", dict(), 4, 12), ("acrobot", dict(T=9), 3, 25)])
def test_native_solver_walks_through_the_oracle_driven_iterates(name, kw, B, iters):
    """dto_sqp_solve stopped after k iterations must stand where the oracle-driven twin stood after k iterations, for
    every k (the native arm keeps no history, so it is simply run with max_iter = k); final multipliers, residuals and
    iteration counts must match too."""
    mo, mp = M.BUILDERS[name](O, **kw), M.BUILDERS[name](D, **kw)
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    z0 = _guess(mp, B, 5)
    perm, bw = PK.analyze(pn)
    opts = sqp.SQPOptions(max_iter=iters, dual_reg=1.0e-6)
    ref = sqp.solve(OracleBackend(osolver, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band"), z0, options=opts, record=True)
    for k in range(1, len(ref.history)):
        got = sqp.solve_native(pn, z0, options=sqp.SQPOptions(max_iter=k, dual_reg=opts.dual_reg))
        hr = ref.history[k]
        scale = np.maximum(1.0, np.abs(hr["z"]))
        assert np.max(np.abs(got.z - hr["z"]) / scale) < 1e-7, (name, k)
        assert np.allclose(got.lam, hr["lam"], rtol=1e-5, atol=1e-7), (name, k)
    got = sqp.solve_native(pn, z0, options=opts)
    assert np.array_equal(got.converged, ref.converged) and np.array_equal(got.iterations, ref.iterations)
    assert got.stats["iterations"] == len(ref.history) and got.stats["launches"] > 0
    both = got.converged & ref.converged
    assert np.allclose(got.objective[both], ref.objective[both], rtol=1e-8)
    assert np.allclose(got.constraint_violation, ref.constraint_violation, atol=1e-9)
    # the final iterate is the batch's resident z (get_trajectory, src/solver.jl:41-43)
    assert np.array_equal(pn.last_x(B - 1), got.z[B - 1])
    pn.close()


def test_native_solver_pinned_end_points_and_scope():
    """test/solve.jl:227-296 set-up (x1 pinned by equal bounds, xT by a GeneralConstraint) through dto_sqp_solve: same
    result as the oracle-driven twin, pinned variables exactly at the bound; inequality bounds switch the native solver
    to its interior-point mode (iterates strictly inside), inconsistent bounds are an argument error."""
    from dto_b200 import _lib
    kw = dict(reference_exact=True)
    mo, mp = M.build_linear_general(O, **kw), M.build_linear_general(D, **kw)
    B = 4
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    z0 = _guess(mp, B, 21)
    perm, bw = PK.analyze(pn)
    opts = sqp.SQPOptions(max_iter=20, dual_reg=1.0e-6)
    ref = sqp.solve(OracleBackend(osolver, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band"), z0, options=opts, record=True)
    got = sqp.solve_native(pn, z0, options=opts)
    assert got.converged.all() and ref.converged.all() and got.stats["iterations"] == len(ref.history)
    assert np.allclose(got.z, ref.z, rtol=1e-8, atol=1e-10)
    n = mp["n"]
    assert np.array_equal(got.z[:, :n], np.tile(mp["x1"], (B, 1)))
    assert np.all(np.linalg.norm(got.z[:, -n:] - mp["xT"], axis=1) < 1e-3)
    pn.close()
    pb = D.solver_from(M.build_cartpole(D, T=11), batch=2).nlp        # |u| <= 3: inequality bounds -> interior-point mode
    pb.set_parameters(np.tile(np.concatenate([np.zeros(4), [0.0, np.pi, 0.0, 0.0]]), (2, 1)))
    rb = sqp.solve_native(pb, np.zeros((2, pb.num_variables)), options=sqp.SQPOptions(max_iter=15))
    ub = np.stack([rb.z[:, t * 5 + 4] for t in range(10)], axis=1)
    assert np.all(np.abs(ub) < 3.0) and np.all(np.isfinite(rb.z))      # (T = 11 is too short to swing up: only the bounds are checked)
    with pytest.raises(_lib.DtoError) as e:                          # lower > upper is an argument error, not a scope question
        lo, up = pb.variable_bounds
        lo2 = lo.copy(); lo2[4] = 5.0
        z0 = np.zeros((2, pb.num_variables))
        out = [np.empty((2, pb.num_variables)), np.empty((2, pb.num_constraint))]
        _lib.check(_lib.lib().dto_sqp_solve(pb.handle, None, z0.ctypes.data, None, lo2.ctypes.data, np.ascontiguousarray(up).ctypes.data,
                                            out[0].ctypes.data, out[1].ctypes.data, None, None, None, None, None, None))
    assert e.value.status == -1
    pb.close()


def test_native_solver_full_solves_and_solver_api():
    """Solver.solve(method='native') on the reference's acrobot test (end points pinned by bounds, T = 101): the
    acceptance of test/solve.jl:134-137 for >= 90 % of 64 seeded problems, and the same success set as the torch arm
    on a smaller batch."""
    ma = M.build_acrobot(D, T=101, stage_endpoint_constraints=False)
    B = 64
    s = D.solver_from(ma, batch=B)
    s.initialize_states(D.linear_interpolation(ma["x1"], ma["xT"], 101))
    rng = np.random.default_rng(4)
    for b in range(B):
        s.initialize_controls([rng.normal(size=1) for _ in range(100)], problem=b)
    res = s.solve(options=dict(max_iter=300), method="native")
    ok = 0
    for b in range(B):
        xs, _ = s.get_trajectory(b)
        ok += int(np.linalg.norm(xs[0] - ma["x1"]) < 1e-3 and np.linalg.norm(xs[-1] - ma["xT"]) < 1e-3 and float(res.constraint_violation[b]) < 1e-6)
    assert ok >= 0.9 * B, ok
    assert s.sqp_launches > 100 and res.stats["syncs"] < res.stats["launches"]
    s.nlp.close()


def test_native_one_pass_line_search_equals_sequential_rounds(monkeypatch):
    """After the first round the native solver evaluates every remaining step length of the still-open problems in ONE
    pass over trial slots and takes the first that passes -- which is what the sequential rounds do one host round trip
    at a time (DTO_SQP_MULTI=0). Same trial points, same kernels, same test: the two must agree bit for bit, on a
    batch whose searches do backtrack (acrobot swing-up from random controls)."""
    ma = M.build_acrobot(D, T=101, stage_endpoint_constraints=False)
    B = 48
    pn = D.solver_from(ma, batch=B).nlp
    z0 = _guess(ma, B, 12)
    opts = sqp.SQPOptions(max_iter=60)
    one = sqp.solve_native(pn, z0, options=opts)
    monkeypatch.setenv("DTO_SQP_MULTI", "0")
    seq = sqp.solve_native(pn, z0, options=opts)
    assert one.stats["multi_trial_passes"] > 0 and seq.stats["multi_trial_passes"] == 0
    assert seq.stats["search_rounds"] > one.stats["search_rounds"]          # the searches did go past the first round
    assert np.array_equal(one.z, seq.z) and np.array_equal(one.lam, seq.lam)
    assert np.array_equal(one.iterations, seq.iterations) and np.array_equal(one.constraint_violation, seq.constraint_violation)
    pn.close()


def test_native_inertia_ladder_equals_one_try_per_pass(monkeypatch):
    """Inertia correction: the native solver factorises the next four regularisations of every bad problem side by side
    (candidate slots of the factor kernel) and keeps the first that gives N_c negative pivots; DTO_SQP_LADDER=1 tries
    the values one factorisation pass at a time. Same ladder, same factor kernel: bit-identical iterates, fewer passes."""
    ma = M.build_acrobot(D, T=101, stage_endpoint_constraints=False)
    B = 48
    pn = D.solver_from(ma, batch=B).nlp
    z0 = _guess(ma, B, 12)
    opts = sqp.SQPOptions(max_iter=60)
    lad = sqp.solve_native(pn, z0, options=opts)      # the default: ladder in candidate slots after the first check
    monkeypatch.setenv("DTO_SQP_LADDER", "1")
    seq = sqp.solve_native(pn, z0, options=opts)
    assert lad.stats["refactorisations"] < seq.stats["refactorisations"]
    assert np.array_equal(lad.z, seq.z) and np.array_equal(lad.lam, seq.lam)
    assert np.array_equal(lad.iterations, seq.iterations) and np.array_equal(lad.dual_residual, seq.dual_residual)
    pn.close()


def test_native_solver_leaves_converged_problems_out_of_the_factorisation(monkeypatch):
    """Once half of the batch has converged, the first factorisation of an iteration runs over the list of problems that
    have not (DTO_SQP_SKIP_DONE=0: always everything). A converged problem's step is never taken, so nothing may change:
    iterates, iteration counts, residuals bit for bit -- on a batch whose problems converge at different iterations."""
    ma = M.build_acrobot(D, T=101, stage_endpoint_constraints=False)
    B = 32
    pn = D.solver_from(ma, batch=B).nlp
    z0 = _guess(ma, B, 12)
    opts = sqp.SQPOptions(max_iter=260)
    on = sqp.solve_native(pn, z0, options=opts)
    monkeypatch.setenv("DTO_SQP_SKIP_DONE", "0")
    off = sqp.solve_native(pn, z0, options=opts)
    assert 2 * on.converged.sum() > B and len(set(on.iterations[on.converged].tolist())) >= 3
    assert np.array_equal(on.z, off.z) and np.array_equal(on.lam, off.lam) and np.array_equal(on.iterations, off.iterations)
    assert np.array_equal(on.constraint_violation, off.constraint_violation) and np.array_equal(on.dual_residual, off.dual_residual)
    assert np.array_equal(on.objective, off.objective)
    pn.close()


def test_interior_point_mode_with_active_control_bounds_matches_oracle_twin():
    """Inequality bounds on variables (Bound(action_lower, action_upper), src/bounds.jl): `sqp.solve` treats them by a
    primal-dual interior point on the same Newton-KKT step -- the barrier term Sigma = z_L/(x-l) + z_U/(u-x) is added to
    H's diagonal INSIDE the factor kernel (per-problem, per-variable array, dto_kkt_device_pointer(k, 5)). Pendulum
    swing-up with |u| <= 15 (the unconstrained optimum peaks at 18.6): the device arm walks through the oracle-driven
    twin's iterates, converges, respects the bounds strictly, has controls AT the bound, and pays for it in the
    objective; the KKT matrix the kernel assembled carries the diagonal."""
    import torch
    kw = dict(u_bnd=15.0)
    mo, mp = M.build_pendulum(O, **kw), M.build_pendulum(D, **kw)
    B = 3
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    z0 = _guess(mp, B, 5)
    perm, bw = PK.analyze(pn)
    opts = sqp.SQPOptions(max_iter=40, dual_reg=1.0e-6)
    ref = sqp.solve(OracleBackend(osolver, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band", options=opts), z0, options=opts, record=True)
    be = sqp.DeviceBackend(pn, dual_reg=opts.dual_reg, options=opts)
    assert be.bounds is not None and int(be.bounds["hasL"].sum()) == mp["T"] - 1
    got = sqp.solve(be, torch.as_tensor(z0, device=be.xp.device), options=opts, record=True)
    K = be.kkt.matrix(1)
    diag = be.d_diag[1, :pn.num_variables].cpu().numpy()      # (the array is [B, dim]: constraint rows carry the slack terms, none here)
    assert float(be.d_diag[:, pn.num_variables:].abs().max()) == 0.0
    be.close()
    assert bool(got.converged.all()) and ref.converged.all() and len(got.history) == len(ref.history)
    for hg, hr in zip(got.history, ref.history):
        assert np.max(np.abs(hg["z"] - hr["z"]) / np.maximum(1.0, np.abs(hr["z"]))) < 1e-9, hg["it"]
    Z = got.z.cpu().numpy()
    n, m, T = mp["n"], mp["m"], mp["T"]
    U = np.stack([Z[:, t * (n + m) + n] for t in range(T - 1)], axis=1)
    assert np.all(np.abs(U) < 15.0) and np.any(np.abs(U) > 15.0 - 1e-5)
    assert np.allclose(got.objective.cpu().numpy(), ref.objective, rtol=1e-9)
    # unconstrained optimum of the same problem for comparison (native arm): lower objective, |u| beyond 15
    pf = D.solver_from(M.build_pendulum(D), batch=B).nlp
    free = sqp.solve_native(pf, z0)
    assert free.converged.all() and np.all(free.objective < got.objective.cpu().numpy() - 1.0)
    pf.close()
    # the barrier diagonal is part of the assembled matrix: positive exactly on the bounded variables
    isu = np.zeros(pn.num_variables, dtype=bool)
    isu[[t * (n + m) + n for t in range(T - 1)]] = True
    assert np.all(diag[isu] > 0.0) and np.all(diag[~isu] == 0.0) and np.all(np.diag(K)[:pn.num_variables][isu] >= diag[isu] * (1 - 1e-12))
    pn.close()


def test_reference_cartpole_example_with_control_bounds_solves_on_the_device():
    """/root/reference/examples/cartpole/cartpole.jl as published -- T = 101, |u| <= 3 as Bound(action_lower, action_upper),
    the state pinned at both ends, the example's own guess (constant controls 0.01, states of an explicit rollout) -- for
    a batch, through Solver.solve(): bounds on variables select the interior-point mode of the lock-step solver. Every
    problem must converge to a KKT point of the bounded problem: dynamics satisfied (checked with the
    constraint callback at the returned point), end points met, |u| strictly within 3 with a good part of the controls AT the bound."""
    import examples.cartpole_swingup as ex
    B, T = 24, 101
    model = M.build_cartpole(D, T=T)
    n, m, x1, xT = model["n"], model["m"], model["x1"], model["xT"]
    s = D.solver_from(model, batch=B)
    s.nlp.set_parameters(np.tile(np.concatenate([x1, xT]), (B, 1)))
    rng = np.random.default_rng(0)
    for b in range(B):
        u0 = np.array([0.01 * (1.0 + 0.2 * rng.normal())])
        xs = [x1.astype(float)]
        for _ in range(T - 1):
            xs.append(np.array(M.cartpole_rk3_explicit(xs[-1], u0, np.zeros(0)), dtype=float))
        s.initialize_states(xs, problem=b)
        s.initialize_controls([u0] * (T - 1), problem=b)
    res = s.solve(options=dict(max_iter=600))                 # method="auto" -> the native solver's interior-point mode: no broker
    assert s.broker is None and s.sqp_launches > 100
    assert bool(_np(res.converged).all()), res.iterations
    Z = _np(res.z)
    c = np.zeros((B, s.nlp.num_constraint))
    s.nlp.eval_constraint(c, Z)
    assert np.max(np.abs(c)) < 1e-7
    U = np.stack([Z[:, t * (n + m) + n] for t in range(T - 1)], axis=1)
    assert np.all(np.abs(U) < 3.0) and (np.abs(U) > 3.0 - 1e-4).mean() > 0.1
    assert np.max(np.abs(Z[:, :n] - x1)) < 1e-6 and np.max(np.abs(Z[:, -n:] - xT)) < 1e-6
    s.nlp.close()
    assert callable(ex.main)


def test_reference_car_example_with_obstacle_inequalities_solves_on_the_device():
    """/root/reference/examples/car/car.jl as published (T = 51, |u| <= 0.5, pinned end states, one obstacle INEQUALITY row
    per knot, the example's guess) for a batch through Solver.solve(): inequality rows and bounds select the
    interior-point mode; its (2,2)-block diagonal -t_i/lam_i is added inside the factor kernel like the bounds' Sigma. The
    direct solve fails on some guesses (controls run into their bounds first); the bound continuation of `solve_bounded`
    picks those up. Every converged problem: dynamics satisfied, obstacle rows <= 0 and touched, controls within the bounds and at them."""
    B, T = 12, 51
    model = M.build_car(D, T=T, obstacle="stage")
    n, m, x1, xT = model["n"], model["m"], model["x1"], model["xT"]
    s = D.solver_from(model, batch=B)
    s.initialize_states(D.linear_interpolation(x1, xT, T))
    rng = np.random.default_rng(2)
    for b in range(B):
        s.initialize_controls([0.001 * rng.normal(size=m) for _ in range(T - 1)], problem=b)
    res = s.solve(options=dict(max_iter=300))
    conv = _np(res.converged)
    assert s.broker is None and conv.sum() >= B - 1, conv          # (99.7 % of 1024 guesses: tools/ip_car.py)
    Z = _np(res.z)
    c = np.zeros((B, s.nlp.num_constraint))
    s.nlp.eval_constraint(c, Z)
    clo, cup = s.nlp.constraint_bounds
    ineq = clo != cup
    Z, c = Z[conv], c[conv]
    assert ineq.sum() == T and np.max(np.abs(c[:, ~ineq])) < 1e-7
    assert np.max(c[:, ineq]) < 1e-7 and np.all((c[:, ineq] > -1e-5).sum(axis=1) >= 1)
    U = np.concatenate([Z[:, t * (n + m) + n: t * (n + m) + n + m] for t in range(T - 1)], axis=1)
    assert np.all(np.abs(U) < 0.5) and np.all((np.abs(U) > 0.5 - 1e-4).sum(axis=1) >= 3)
    assert np.array_equal(Z[:, :n], np.tile(x1, (len(Z), 1))) and np.array_equal(Z[:, -n:], np.tile(xT, (len(Z), 1)))
    s.nlp.close()


def test_interior_point_inequality_rows_device_iterates_match_oracle_twin():
    """Inequality rows in the interior-point mode: the -t_i/lam_i entries of K's (2,2) block and the shifted right-hand side
    are applied on the device (factor kernel, DIAG instantiation; constraint array) and densely in the oracle-driven twin.
    Car with obstacle rows, control bounds and pinned end states at the small test shape (T = 7; too short to reach the goal,
    which is irrelevant here): the two arms must walk through the same iterates."""
    import torch
    kw = dict(T=7, obstacle="stage")
    mo, mp = M.build_car(O, **kw), M.build_car(D, **kw)
    B = 3
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    z0 = _guess(mp, B, 8) * 0.05
    n, m, T = mp["n"], mp["m"], mp["T"]
    for t in range(T):
        z0[:, t * (n + m): t * (n + m) + n] = mp["x1"] + (mp["xT"] - mp["x1"]) * t / (T - 1)
    perm, bw = PK.analyze(pn)
    opts = sqp.SQPOptions(max_iter=12, dual_reg=1.0e-6)
    ref = sqp.solve(OracleBackend(osolver, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band", options=opts), z0, options=opts, record=True)
    be = sqp.DeviceBackend(pn, dual_reg=opts.dual_reg, options=opts)
    assert int(be.bounds["hasI"].sum()) == T and int(be.bounds["hasL"].sum()) == (T - 1) * m
    got = sqp.solve(be, torch.as_tensor(z0, device=be.xp.device), options=opts, record=True)
    assert float(be.d_diag[:, pn.num_variables:].abs().max()) > 0.0          # the slack terms reached the kernel's array
    be.close()
    assert len(got.history) == len(ref.history) == 12
    for hg, hr in zip(got.history, ref.history):
        assert np.max(np.abs(hg["z"] - hr["z"]) / np.maximum(1.0, np.abs(hr["z"]))) < 1e-7, hg["it"]
        assert np.allclose(hg["f"], hr["f"], rtol=1e-7, atol=1e-9), hg["it"]
    pn.close()


@pytest.mark.parametrize("case", ["pendulum_bounds", "cartpole_example", "car_example"])
def test_native_interior_point_agrees_with_the_torch_glued_arm(case):
    """The interior-point mode exists in both arms: `sqp.solve` (torch glue; equal to the oracle-driven twin iterate by
    iterate, tests above) and dto_sqp_solve (kernels k_ip_* of csrc/dto_sqp.cu). Same algorithm, different summation
    orders: the two must converge for the same problems, in (nearly) the same number of iterations, to the same points."""
    import torch
    if case == "pendulum_bounds":
        model, B, iters = M.build_pendulum(D, u_bnd=15.0), 4, 60
    elif case == "cartpole_example":
        model, B, iters = M.build_cartpole(D, T=101), 8, 400
    else:
        model, B, iters = M.build_car(D, T=51, obstacle="stage"), 8, 300
    n, m, T, x1, xT = model["n"], model["m"], model["T"], model["x1"], model["xT"]
    s = D.solver_from(model, batch=B)
    rng = np.random.default_rng(5)
    if case == "cartpole_example":
        s.nlp.set_parameters(np.tile(np.concatenate([x1, xT]), (B, 1)))
        for b in range(B):
            u0 = np.array([0.01 * (1.0 + 0.2 * rng.normal())])
            xs = [x1.astype(float)]
            for _ in range(T - 1):
                xs.append(np.array(M.cartpole_rk3_explicit(xs[-1], u0, np.zeros(0)), dtype=float))
            s.initialize_states(xs, problem=b)
            s.initialize_controls([u0] * (T - 1), problem=b)
    else:
        s.initialize_states(D.linear_interpolation(x1, xT, T))
        for b in range(B):
            s.initialize_controls([(0.3 if case == "pendulum_bounds" else 0.001) * rng.normal(size=m) for _ in range(T - 1)], problem=b)
    nat = s.solve(options=dict(max_iter=iters), method="native")
    tor = s.solve(options=dict(max_iter=iters), method="sqp")
    cn, ct = _np(nat.converged), _np(tor.converged)
    assert cn.sum() >= B - 1 and ct.sum() >= B - 1
    both = cn & ct
    zn, zt = _np(nat.z)[both], _np(tor.z)[both]
    assert np.max(np.abs(zn - zt) / np.maximum(1.0, np.abs(zt))) < 1e-5
    assert np.allclose(_np(nat.objective)[both], _np(tor.objective)[both], rtol=1e-6, atol=1e-8)
    direct = both & ~_np(getattr(nat, "staged", np.zeros(B, bool))) & ~_np(getattr(tor, "staged", torch.zeros(B, dtype=torch.bool)))
    assert np.max(np.abs(_np(nat.iterations)[direct] - _np(tor.iterations)[direct])) <= 3
    s.nlp.close()


def test_one_sided_bounds_in_both_device_arms():
    """A bound on one side only (Bound(action_lower = [-10]), no upper bound): the interior-point mode must treat the missing
    side as absent (no barrier term, no push, never scaled by the continuation). Pendulum swing-up, whose unconstrained optimum
    dips to u = -16.7: both device arms converge to the same point, u >= -10 strictly, the bound is active somewhere, and the
    upper side is free to exceed +10."""
    model = M.build_pendulum(D)
    n, m, T = model["n"], model["m"], model["T"]
    model["bounds"] = [D.Bound(n, m, action_lower=[-10.0])] * (T - 1) + [D.Bound(n, 0)]
    B = 3
    s = D.solver_from(model, batch=B)
    lo, up = s.nlp.variable_bounds
    assert np.isfinite(lo).sum() == T - 1 and not np.isfinite(up).any()
    s.initialize_states(D.linear_interpolation(model["x1"], model["xT"], T))
    rng = np.random.default_rng(3)
    for b in range(B):
        s.initialize_controls([0.3 * rng.normal(size=m) for _ in range(T - 1)], problem=b)
    nat = s.solve(options=dict(max_iter=80), method="native")
    tor = s.solve(options=dict(max_iter=80), method="sqp")
    assert _np(nat.converged).all() and _np(tor.converged).all()
    zn, zt = _np(nat.z), _np(tor.z)
    assert np.max(np.abs(zn - zt) / np.maximum(1.0, np.abs(zt))) < 1e-5
    U = np.stack([zn[:, t * (n + m) + n] for t in range(T - 1)], axis=1)
    assert np.all(U > -10.0) and np.any(U < -10.0 + 1e-4) and np.any(U > 10.0)
    s.nlp.close()


def test_solve_over_several_devices_equals_the_single_device_solve():
    """Row (e) for the solver: a batch spread over all visible devices is solved by one dto_sqp_solve per device, side by side
    (sqp.solve_native_sharded), no collective. Problems are independent and every kernel gives a problem the same bits wherever
    it sits, so the result must equal the one-device solve bit for bit -- with per-problem parameters and bounds in play
    (cartpole example) and without (pendulum). Needs >= 2 GPUs (`gpurun --gpus 2`)."""
    import torch
    ndev = torch.cuda.device_count()
    if ndev < 2:
        pytest.skip("needs at least 2 GPUs")
    for case in ("pendulum", "cartpole"):
        B = 2 * ndev + 1                                   # ragged shards
        outs = []
        for devices in ([0], list(range(ndev))):
            if case == "pendulum":
                model = M.build_pendulum(D)
                s = D.solver_from(model, batch=B, devices=devices)
                s.initialize_states(D.linear_interpolation(model["x1"], model["xT"], model["T"]))
                for b in range(B):
                    s.initialize_controls([np.array([0.05 * (b + 1)]) for _ in range(model["T"] - 1)], problem=b)
                opts = dict(max_iter=60)
            else:
                model = M.build_cartpole(D, T=101)
                T, x1, xT = 101, model["x1"], model["xT"]
                s = D.solver_from(model, batch=B, devices=devices)
                W = np.tile(np.concatenate([x1, xT]), (B, 1))
                W[:, 5] += 0.01 * np.arange(B)             # per-problem goal angles: the parameter slices must follow the shards
                s.nlp.set_parameters(W)
                for b in range(B):
                    u0 = np.array([0.01 * (1.0 + 0.1 * b)])
                    xs = [x1.astype(float)]
                    for _ in range(T - 1):
                        xs.append(np.array(M.cartpole_rk3_explicit(xs[-1], u0, np.zeros(0)), dtype=float))
                    s.initialize_states(xs, problem=b)
                    s.initialize_controls([u0] * (T - 1), problem=b)
                opts = dict(max_iter=300)
            assert s.nlp.num_shards == len(devices)
            res = s.solve(options=opts)
            assert s.broker is None and _np(res.converged).all()
            xs_last, _ = s.get_trajectory(B - 1)
            outs.append((_np(res.z).copy(), _np(res.iterations).copy(), np.concatenate(xs_last)))
            if len(devices) > 1:
                assert res.stats["devices"] == devices
            s.nlp.close()
        assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1]) and np.array_equal(outs[0][2], outs[1][2])

"""CPU side of the native solver's walks at shipped sizes (tests/test_sqp_scale_gpu.py): the twin's batched banded solve against
the problem-by-problem one, its C-twin evaluation with per-problem parameters against the oracle, and, for every walk case of
tests/scale_cases.py, that the twin runs as long as the walk expects and takes the branch of dto_sqp_host.inc the case claims to
reach -- so that a case cannot pass on the GPU at a smaller size or without its branch."""
import numpy as np
import pytest

from examples import models as M
from oracle import api as O
from oracle import cgen

from scale_cases import CASES, ITERATIONS, Case
from sqp_oracle import OracleBackend, band_ldl_solve, band_ldl_solve_batched
from util import assert_close


def _banded_indefinite(rng, B, n, bw):
    """B symmetric matrices whose permutation P K P' has half bandwidth bw and indefinite diagonal blocks of either sign,
    dominant enough that no pivot of the unpivoted LDL' vanishes; and that permutation"""
    perm = rng.permutation(n)
    A = np.zeros((B, n, n))
    for k in range(1, bw + 1):
        v = rng.uniform(-1.0, 1.0, (B, n - k))
        i = np.arange(n - k)
        A[:, i, i + k] = v
        A[:, i + k, i] = v
    sign = np.where(rng.uniform(size=(B, n)) < 0.4, -1.0, 1.0)
    A[:, np.arange(n), np.arange(n)] = sign * rng.uniform(2.0 * bw, 3.0 * bw, (B, n))
    K = np.empty_like(A)
    K[:, perm[:, None], perm[None, :]] = A          # K[perm][:, perm] = A
    return K, perm


@pytest.mark.parametrize("n", [56, 912])
@pytest.mark.parametrize("bw", [6, 30])
def test_batched_band_solve_gives_the_bits_of_the_problem_by_problem_solve(n, bw):
    rng = np.random.default_rng(n + bw)
    B = 5
    K, perm = _banded_indefinite(rng, B, n, bw)
    h = rng.normal(size=(B, n))
    x, nneg = band_ldl_solve_batched(K, h, perm, bw)
    for b in range(B):
        xb, nb = band_ldl_solve(K[b], h[b], perm, bw)
        assert nneg[b] == nb > 0
        assert np.array_equal(x[b], xb), b
        r = K[b] @ xb - h[b]
        assert np.max(np.abs(r)) < 1e-12 * np.max(np.abs(K[b])) * max(1.0, np.max(np.abs(xb)))


def test_batched_band_solve_sees_the_same_inertia_as_the_eigenvalues():
    rng = np.random.default_rng(3)
    K, perm = _banded_indefinite(rng, 4, 56, 6)
    _, nneg = band_ldl_solve_batched(K, rng.normal(size=(4, 56)), perm, 6)
    assert np.array_equal(nneg, (np.linalg.eigvalsh(K) < 0).sum(axis=1))


@pytest.mark.parametrize("name,kw", [("pendulum", dict()), ("linear_general", dict(reference_exact=True))])
def test_batched_newton_step_gives_the_bits_of_the_problem_by_problem_step(name, kw):
    """the whole Newton step of the twin (assembly with regularisation, barrier diagonal and pinned variables, then the solve)"""
    import dto_b200 as D
    from dto_b200 import kkt as PK
    mo = M.BUILDERS[name](O, **kw)
    osolver, pn = O.solver_from(mo), D.solver_from(M.BUILDERS[name](D, **kw), batch=1).nlp
    perm, bw = PK.analyze(pn)
    B = 4
    rng = np.random.default_rng(7)
    z, lam = rng.normal(size=(B, pn.num_variables)), rng.normal(size=(B, pn.num_constraint))
    delta, diag = rng.uniform(0.0, 1e-2, B), rng.uniform(0.0, 1.0, (B, pn.num_variables))
    out = []
    for linear in ("band", "band-batched"):
        be = OracleBackend(osolver, B, dual_reg=1e-6, perm=perm - 1, bw=bw, linear=linear)
        assert be.fixed.any() == (name == "linear_general")
        be.callbacks(z, lam, lam, delta, diag=diag)
        out.append(be.newton(delta))
    for a, b in zip(*out):
        assert np.array_equal(a, b)
    pn.close()


@pytest.fixture(scope="module")
def cartpole_twin():
    mo = M.build_cartpole(O, T=11, u_bnd=None)
    osolver = O.solver_from(mo)
    osolver.set_parameters([np.zeros(8) for _ in range(mo["T"])] + [np.zeros(0)])
    co = cgen.build_c_oracle(osolver, "scale_cartpole11", shared_parameters=True, cse=True)
    return mo, osolver, co


def _cartpole_point(osolver, B, seed):
    rng = np.random.default_rng(seed)
    nlp = osolver.nlp
    return rng.uniform(-1.0, 1.0, (B, nlp.num_variables)), rng.normal(size=(B, nlp.num_constraint))


def test_c_twin_with_per_problem_parameters_equals_the_oracle_on_a_shared_parameter_batch(cartpole_twin):
    mo, osolver, co = cartpole_twin
    B = 4
    w0 = np.concatenate([[0.05, -0.02, 0.01, 0.0], [0.1, np.pi - 0.05, 0.0, 0.02]])
    osolver.set_parameters([w0.copy() for _ in range(mo["T"])] + [np.zeros(0)])
    z, lam = _cartpole_point(osolver, B, 1)
    twin = OracleBackend(osolver, B, c_twin=co, w=np.tile(w0, (B, 1)))._eval(z, lam, 31)
    ref = OracleBackend(osolver, B)._eval(z, lam, 31)
    for k in ("f", "g", "c", "J", "H"):
        assert_close(f"C twin {k}", twin[k], ref[k], rtol=1e-12, atol=1e-14)


def test_c_twin_gives_every_problem_its_own_parameters(cartpole_twin):
    mo, osolver, co = cartpole_twin
    B = 5
    rng = np.random.default_rng(2)
    w = np.concatenate([rng.normal(0.0, 0.1, (B, 4)), mo["xT"] + rng.normal(0.0, 0.1, (B, 4))], axis=1)
    z, lam = _cartpole_point(osolver, B, 3)
    twin = OracleBackend(osolver, B, c_twin=co, w=w)._eval(z, lam, 31)
    for b in range(B):
        osolver.set_parameters([w[b].copy() for _ in range(mo["T"])] + [np.zeros(0)])
        ref = OracleBackend(osolver, 1)._eval(z[b:b + 1], lam[b:b + 1], 31)
        for k in ("f", "g", "c", "J", "H"):
            assert_close(f"C twin problem {b} {k}", twin[k][b:b + 1], ref[k], rtol=1e-12, atol=1e-14)
    # the constraint rows x_1 - w[0:4] and x_T - w[4:8] carry each problem's own end points
    assert len(np.unique(twin["c"], axis=0)) == B
    with pytest.raises(ValueError):
        OracleBackend(osolver, B, w=w)                          # per-problem parameters need the C twin


@pytest.fixture(scope="module")
def cases():
    made = {}

    def get(key):
        if key not in made:
            made[key] = Case(key)
        return made[key]

    yield get
    for c in made.values():
        c.close()


@pytest.mark.parametrize("key", list(CASES))
def test_walk_case_runs_at_its_size_for_its_iterations(cases, key):
    c = cases(key)
    assert c.N_z > 128 and c.N_c > 128 and c.B > 4, (c.N_z, c.N_c, c.B)
    assert c.iterations == ITERATIONS[key]
    assert np.all(np.isfinite(c.ref.z))


def test_case_a_factorises_a_subset_from_the_first_iteration_on(cases):
    c = cases("a_pendulum_alist")
    assert c.B == 37 and c.B % 4 != 0
    open_ = c.open_after_check()
    assert 2 * open_[0] < c.B and all(2 * n < c.B for n in open_)
    assert np.all(c.ref.iterations[::2] == 0) and np.all(c.ref.iterations[1::2] > 0) and c.ref.converged.all()


def test_case_b_takes_the_full_inertia_ladder(cases):
    c = cases("b_band_ladder")
    assert c.bw == 30
    assert any(1 <= n <= c.B // 4 for n in c.be.retries)        # m = min(4, B / n_retry) = 4 candidates per problem
    assert any(n > c.B // 4 for n in c.be.retries)               # ... and shorter ladders while many problems need it


def test_case_c_uses_corrections_and_per_problem_trial_slots(cases):
    c = cases("c_cartpole_w")
    assert c.w.shape == (c.B, 8) and len(np.unique(c.w, axis=0)) == c.B
    assert any(h["soc"].any() for h in c.ref.history if "soc" in h)
    assert any(np.any(h["alpha"] <= 0.5) for h in c.ref.history if "alpha" in h)
    assert c.one_pass_search_after_first_round()


def test_case_d_runs_the_interior_point_mode_with_and_without_inequality_rows(cases):
    pend, car = cases("d_pendulum_bounds"), cases("d_car_obstacle")
    for c in (pend, car):
        assert c.be.bounds is not None and c.be.bounds["hasL"].sum() > 0
    assert pend.be.bounds["hasI"].sum() == 0 and car.be.bounds["hasI"].sum() == 41
    assert len(pend.be.retries) > 0 and len(car.be.retries) > 0


@pytest.mark.parametrize("key", ["e_pendulum_knot_bfgs", "e_pendulum_partitioned_bfgs"])
def test_case_e_updates_every_block_over_20_iterations(cases, key):
    c = cases(key)
    assert c.iterations >= 20
    assert not any(f.any() for f in c.be.first)                  # every knot / element block of every problem took an update


def test_case_f_reaches_every_branch_on_the_shipped_shape(cases):
    c = cases("f_acrobot")
    assert (c.N_z, c.N_c) == (504, 408)
    assert len(c.be.retries) > 0
    assert any(h["soc"].any() for h in c.ref.history if "soc" in h)
    assert c.one_pass_search_after_first_round()

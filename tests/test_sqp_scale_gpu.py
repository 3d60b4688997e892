"""The native solver (dto_sqp_solve) walks through the iterates of its float64 twin at the sizes it ships at: rows of more than
128 entries (the second and later trips of the warp-per-problem kernels of csrc/dto_sqp.cu), batches of several CTAs, per-problem
parameters in the trial slots, and every branch of the search that only a large batch takes. The cases, and what each reaches,
are those of tests/scale_cases.py; tests/test_sqp_scale_cpu.py checks on the twin alone that each case takes the branch it claims.

Every walk stops the native solver after k iterations, for every k the twin ran, and compares its iterate with the twin's after
k iterations, with the tolerances of the walks at toy sizes (tests/test_sqp_gpu.py): z to 1e-7 relative to max(1, |z|), the
multipliers to rtol 1e-5 and atol 1e-7; then convergence flags and iteration counts must be equal and the objectives of the
problems both converged agree to 1e-8."""
import numpy as np
import pytest

from scale_cases import ITERATIONS, Case

pytestmark = pytest.mark.gpu


def _first_split(case, k, got):
    """where the native iterate left the twin's after k iterations: the first problem, and the twin's decisions of the
    iteration before (the quantities to compare when a walk fails)"""
    hr = case.ref.history[k]
    err = np.max(np.abs(got.z - hr["z"]) / np.maximum(1.0, np.abs(hr["z"])), axis=1)
    b = int(np.argmax(err > 1e-7)) if (err > 1e-7).any() else int(np.argmax(err))
    prev = case.ref.history[k - 1]
    keys = ("nu", "slope", "alpha", "delta", "soc", "done")
    return f"{case.key}: k = {k}, problem {b}, z error {err[b]:.3e}; twin at k - 1: " + ", ".join(
        f"{q} = {prev[q][b]!r}" for q in keys if q in prev)


def walk(case):
    """the native solver stopped after k iterations stands where the twin stood, for every k; then the full run"""
    ref = case.ref
    for k in range(1, len(ref.history)):
        got = case.solve_native(k)
        hr = ref.history[k]
        assert np.max(np.abs(got.z - hr["z"]) / np.maximum(1.0, np.abs(hr["z"]))) < 1e-7, _first_split(case, k, got)
        assert np.allclose(got.lam, hr["lam"], rtol=1e-5, atol=1e-7), (case.key, k)
    got = case.solve_native(case.opts.max_iter)
    assert np.array_equal(got.converged, ref.converged) and np.array_equal(got.iterations, ref.iterations), case.key
    assert got.stats["iterations"] == len(ref.history)
    both = got.converged & ref.converged
    assert np.allclose(got.objective[both], ref.objective[both], rtol=1e-8)
    print(f"{case.key}: B = {case.B}, N_z = {case.N_z}, N_c = {case.N_c}, {len(ref.history)} iterations, "
          f"{int(got.converged.sum())} converged; " + ", ".join(f"{q} {got.stats[q]}" for q in
                                                             ("refactorisations", "corrections", "multi_trial_passes", "search_rounds")))
    return got


@pytest.fixture
def case(request):
    c = Case(request.param)
    assert c.N_z > 128 and c.N_c > 128 and c.B > 4, (c.N_z, c.N_c, c.B)
    assert c.iterations == ITERATIONS[c.key]
    yield c
    c.close()


@pytest.mark.parametrize("case", ["a_pendulum_alist"], indirect=True)
def test_subset_factorisation_with_converged_problems_inside_ctas(case):
    """pendulum T = 101, B = 37 (ten CTAs, the last partial): half of the problems start converged, so the first factorisation of
    every later iteration runs over the list of open problems, and converged and open problems alternate inside every CTA"""
    assert any(2 * n < case.B for n in case.open_after_check())
    got = walk(case)
    assert got.stats["refactorisations"] > 0 and got.stats["corrections"] > 0 and got.stats["multi_trial_passes"] > 0
    assert np.all(got.iterations[::2] == 0) and np.all(got.iterations[1::2] > 0)


@pytest.mark.parametrize("case", ["b_band_ladder"], indirect=True)
def test_full_inertia_ladder_with_32_lane_rows(case):
    """band model (15, 2, 14, False) at T = 10: KKT rows of half bandwidth 30, an indefinite reduced Hessian; inertia correction
    with four candidates per problem once at most a quarter of the batch needs it"""
    assert case.bw == 30
    assert any(1 <= n <= case.B // 4 for n in case.be.retries)
    got = walk(case)
    assert got.stats["refactorisations"] > 0 and got.stats["corrections"] > 0


@pytest.mark.parametrize("case", ["c_cartpole_w"], indirect=True)
def test_trial_slots_carry_each_problems_parameters(case):
    """cartpole T = 41 with its own start and goal per problem (w = [x1; xT]) and free controls: one-pass searches over trial
    slots (k_multi_trial copies each problem's w; the objective and constraint kernels evaluate the slots with it) and
    second-order corrections"""
    assert len(np.unique(case.w, axis=0)) == case.B
    got = walk(case)
    assert got.stats["multi_trial_passes"] > 0 and got.stats["corrections"] > 0


@pytest.mark.parametrize("case", ["d_pendulum_bounds", "d_car_obstacle"], indirect=True)
def test_interior_point_over_long_rows(case):
    """k_ip_* over rows of more than 128 entries: bounds on the pendulum's controls, and the car's obstacle rows (any_ineq)"""
    got = walk(case)
    assert np.all(np.isfinite(got.z)) and got.stats["refactorisations"] > 0


@pytest.mark.parametrize("case", ["e_pendulum_knot_bfgs", "e_pendulum_partitioned_bfgs"], indirect=True)
def test_quasi_newton_modes_over_101_knots(case):
    """k_qn_update, k_pqn_update (z_prev alternating with the iteration's parity) and k_pqn_assemble over T = 101 knots for at
    least 20 iterations"""
    assert case.iterations >= 20 and not any(f.any() for f in case.be.first)
    walk(case)


@pytest.mark.parametrize("case", ["f_acrobot"], indirect=True)
def test_acrobot_at_the_shipped_shape(case):
    """acrobot T = 101 (N_z = 504, N_c = 408), the model and length the benchmark solves, for the 15 iterations over which the
    iterates stay within the shared tolerance (see tests/scale_cases.py: they separate gradually, no decision differs)"""
    assert (case.N_z, case.N_c) == (504, 408)
    got = walk(case)
    assert got.stats["refactorisations"] > 0 and got.stats["corrections"] > 0 and got.stats["multi_trial_passes"] > 0

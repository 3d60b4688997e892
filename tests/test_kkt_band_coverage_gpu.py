"""The banded KKT kernels (csrc/dto_kkt.cu) at every compiled bandwidth bound and the first bandwidth past each, and the
native solver's 32-lane paths, against float64 references on the host.

The models are the synthetic band family of tests/band_models.py (bandwidths pinned by tests/test_band_coverage_cpu.py).
For every bandwidth, in the exact-Hessian mode and in the knot-block mode:

  * assembly: K and h bit for bit against the host assembly of the GPU's own g, c, J, H (or blocks);
  * factor: P K P' = L D L' to rounding, L and D against the oracle's QDLDL in the product's ordering within cond-scaled
    rounding, the negative-pivot count against the eigenvalues (indefinite H included);
  * solution: backward error and forward error against the QDLDL solve;
  * variants: the single-row-set kernel and the fused right-hand side give the default kernel's bits, and a re-solve with
    the stored factor gives the bits of factorising again;
  * options: per-problem regularisation, subset launches, pinned variables and the barrier diagonal (DIAG kernels);
  * the batch: odd, one full CTA (4 * 32 / W problems) plus a remainder (the dead second group of a 16-lane warp), and B = 1.

Then the native solver where the KKT matrix needs 32 lanes: exact Hessian at BW = 20 and BW = 31 (free end states, so the
double well makes the reduced Hessian indefinite and the inertia ladder runs in candidate slots: the VIRT kernels), the interior-point mode (DIAG + VIRT), and the knot-block BFGS mode with 17-variable
blocks (k_qn_update<32>), each walking through the iterates of the oracle-driven twin."""
import numpy as np
import pytest

import dto_b200 as D
from dto_b200 import _lib
from dto_b200 import kkt as PK
from dto_b200 import sqp
from oracle import api as O
from oracle import kkt as OK

from band_models import BAND_CASES, QN_BAND, band_kwargs, build_band, case_id
from sqp_oracle import OracleBackend
from test_sqp_qn_cpu import QNOracleBackend

pytestmark = pytest.mark.gpu

MODES = ("exact", "knot-blocks")
KKT_CASES = [(key, mode) for key in BAND_CASES for i, mode in enumerate(MODES) if BAND_CASES[key][i] is not None and BAND_CASES[key][i] <= 31]
REG = 1.0e-4


@pytest.fixture(scope="module")
def nlps():
    """one product batch per (model, batch size, Hessian) for the whole module: each model library is traced and loaded once"""
    cache = {}

    def get(key, B, hessian=True):
        k = (key, B, hessian)
        if k not in cache:
            cache[k] = D.solver_from(build_band(D, **band_kwargs(key), evaluate_hessian=hessian), batch=B).nlp
        return cache[k]

    yield get
    for pn in cache.values():
        pn.close()


def _inputs(pn, B, seed, mode):
    """z, multipliers and (knot-block mode) blocks; large multipliers / non-SPD blocks on every other problem make H indefinite"""
    rng = np.random.default_rng(seed)
    z = rng.uniform(-1.0, 1.0, (B, pn.num_variables))
    lam = rng.normal(size=(B, pn.num_constraint)) * np.where(np.arange(B) % 2 == 0, 30.0, 1.0)[:, None]
    blocks = None
    if mode == "knot-blocks":
        xs, nx, _, nu = pn.knot_layout()
        rows = []
        for b in range(B):
            row = []
            for t in range(pn.T):
                n = int(nx[t] + nu[t])
                A = rng.normal(size=(n, n))
                S = A @ A.T + n * np.eye(n) if b % 2 else A
                row.append((0.5 * (S + S.T)).ravel())          # bitwise symmetric
            rows.append(np.concatenate(row))
        blocks = np.array(rows)
    return z, lam, blocks


def _evaluate(pn, mode):
    """the callback outputs at the resident (z, multipliers) of every problem, as the KKT launch consumed them"""
    B = pn.batch
    cb = dict(g=np.empty((B, pn.num_variables)), c=np.empty((B, pn.num_constraint)), J=np.empty((B, pn.num_jacobian)))
    pn.eval_objective_gradient(cb["g"])
    pn.eval_constraint(cb["c"])
    if mode == "exact":
        cb["H"] = np.empty((B, pn.num_hessian))
        pn.eval_jacobian_hessian(cb["J"], cb["H"])
    else:
        pn.eval_constraint_jacobian(cb["J"])
    return cb


def _host_system(pn, mode, cb, b, lam, blocks, preg, dreg):
    """K and h of problem b: the oracle's assembly of the GPU's callback outputs `cb` (knot-block mode: of the blocks, in
    the order of hessian_block_structure)"""
    nz, ny = pn.num_variables, pn.num_constraint
    if mode == "exact":
        hs, H = pn.hessian_lagrangian_structure(), cb["H"][b]
    else:
        r, c = pn.hessian_block_structure()
        hs, H = list(zip(r.tolist(), c.tolist())), blocks[b]
    return OK.assemble(nz, ny, pn.jacobian_structure(), hs, cb["g"][b], cb["c"][b], cb["J"][b], H, lam[b], preg, dreg)


def _check_factor(kkt, b, K, h, perm, sol):
    """P K P' = L D L', L and D against QDLDL in the same ordering, inertia against the eigenvalues, backward / forward error"""
    Lm, Dv = kkt.factor(b)
    Kp = K[np.ix_(perm, perm)]
    scale = np.max(np.abs(Kp))
    growth = max(1.0, np.max(np.abs(Lm)) ** 2 * np.max(np.abs(Dv)) / scale)
    assert np.max(np.abs(Lm @ np.diag(Dv) @ Lm.T - Kp)) <= 1e-13 * scale * growth * kkt.row_width, b
    Lr, Dr, Dinv, _ = OK.qdldl_factor(K, perm)
    # the two factorisations sum in different orders; without pivoting an indefinite K has element growth, which scales
    # the difference of their rounding errors like cond(K) does
    cond = np.linalg.cond(K)
    tol = 50 * cond * growth * np.finfo(float).eps
    assert np.array_equal(Dv > 0, Dr > 0), b
    assert np.max(np.abs(Dv - Dr) / np.abs(Dr)) <= tol, b
    assert np.max(np.abs(Lm - Lr)) <= tol * max(1.0, np.max(np.abs(Lr))), b
    ev = np.linalg.eigvalsh(K)
    assert kkt.inertia()[b] == int((ev < 0).sum()) == int((Dv < 0).sum()), b
    x = sol[b]
    assert np.max(np.abs(K @ x - h)) <= 1e-13 * growth * (np.linalg.norm(K, np.inf) * np.max(np.abs(x)) + np.max(np.abs(h))), b
    ref = OK.qdldl_solve(Lr, Dinv, h, perm)
    assert np.max(np.abs(x - ref)) <= tol * max(1.0, np.max(np.abs(ref))), b


def _make(pn, mode, blocks, preg=REG, dreg=REG):
    kkt = PK.KKTSystem(pn, preg, dreg, hessian=mode)
    if blocks is not None:
        kkt.set_hessian_blocks(blocks)
    return kkt


@pytest.mark.parametrize("key,mode", KKT_CASES, ids=[f"{case_id(k)}-{m}" for k, m in KKT_CASES])
def test_kkt_kernels_at_every_bandwidth(key, mode, nlps, monkeypatch):
    bw = BAND_CASES[key][MODES.index(mode)]
    W = 16 if bw <= 15 else 32
    B = 4 * (32 // W) + 3
    for batch in (B, 1):
        pn = nlps(key, batch)
        z, lam, blocks = _inputs(pn, batch, 11 + bw, mode)
        kkt = _make(pn, mode, blocks)
        assert kkt.bandwidth == bw and kkt.row_width == W
        perm = kkt.permutation() - 1
        sol = np.full((batch, kkt.dim), np.nan)
        kkt.solve(sol, variables=z, scaling=np.ones(batch), duals=lam)
        assert np.array_equal(kkt.solution(), sol)
        h = kkt.rhs()
        cb = _evaluate(pn, mode)
        indefinite = 0
        for b in range(batch):
            K, hh = _host_system(pn, mode, cb, b, lam, blocks, REG, REG)
            assert np.array_equal(kkt.matrix(b), K), f"problem {b}: assembled K differs from the host assembly"
            assert np.array_equal(h[b], hh), f"problem {b}: right-hand side differs"
            _check_factor(kkt, b, K, hh, perm, sol)
            nz = pn.num_variables
            indefinite += int(np.linalg.eigvalsh(K[:nz, :nz])[0] < 0.0)
        if batch > 1:
            assert indefinite > 0, "no indefinite Hessian block in the batch"
        factors = [kkt.factor(b) for b in range(batch)]
        kkt.close()
        # the single-row-set kernel (where the bound has one) and the fused right-hand side: the same bits
        for var, val in (("DTO_KKT_VARIANT", "single"), ("DTO_KKT_FUSE_RHS", "1")):
            monkeypatch.setenv(var, val)
            other = _make(pn, mode, blocks)
            s2 = np.empty_like(sol)
            other.solve(s2, variables=z, scaling=np.ones(batch), duals=lam)
            assert np.array_equal(s2, sol), var
            assert np.array_equal(other.rhs(), h), var
            for b in range(batch):
                L2, D2 = other.factor(b)
                assert np.array_equal(L2, factors[b][0]) and np.array_equal(D2, factors[b][1]), (var, b)
            other.close()
            monkeypatch.delenv(var)


@pytest.mark.parametrize("key,mode", KKT_CASES, ids=[f"{case_id(k)}-{m}" for k, m in KKT_CASES])
def test_kkt_options_at_every_bandwidth(key, mode, nlps):
    """resolve (whole batch, problem list), per-problem regularisation, launch_subset, set_fixed and the DIAG kernels"""
    import torch
    from dto_b200.evaluator import A_C
    bw = BAND_CASES[key][MODES.index(mode)]
    W = 16 if bw <= 15 else 32
    B = 4 * (32 // W) + 3
    pn = nlps(key, B)
    nz, ny = pn.num_variables, pn.num_constraint
    z, lam, blocks = _inputs(pn, B, 23 + bw, mode)
    kkt = _make(pn, mode, blocks, 0.0, 1.0e-6)
    dev = torch.device("cuda", pn.shard_device(0))
    stream = torch.cuda.ExternalStream(pn.stream_pointer(0), device=dev)
    perm = kkt.permutation() - 1
    # per-problem primal regularisation
    reg = np.linspace(1.0e-3, 3.0, B)
    kkt.set_primal_reg(reg)
    sol0 = np.empty((B, kkt.dim))
    kkt.solve(sol0, variables=z, scaling=np.ones(B), duals=lam)
    nneg0 = kkt.inertia()
    cb = _evaluate(pn, mode)
    for b in (0, B // 2, B - 1):
        K, hh = _host_system(pn, mode, cb, b, lam, blocks, reg[b], 1.0e-6)
        assert np.array_equal(kkt.matrix(b), K), b
        _check_factor(kkt, b, K, hh, perm, sol0)
    # resolve with a new c: the bits of factorising again, for the batch and for a problem list
    d_c = torch.as_tensor(sqp._CudaArray(pn.device_pointer(A_C, 0), (B, ny)), device=dev)
    c_new = torch.as_tensor(np.random.default_rng(bw).normal(size=(B, ny)), device=dev)
    with torch.cuda.stream(stream):
        c_old = d_c.clone()
        d_c.copy_(c_new)
    kkt.resolve()
    pn.sync()
    got = kkt.solution()
    kkt.launch(False)
    pn.sync()
    ref = kkt.solution()
    assert np.array_equal(got, ref) and not np.array_equal(got, sol0)
    pick = np.array([1, B // 2, B - 1], dtype=np.int32)
    idx = torch.as_tensor(pick, device=dev)
    with torch.cuda.stream(stream):
        d_c[idx.long()] = c_old[idx.long()]
    kkt.resolve(idx.data_ptr(), len(pick))
    pn.sync()
    part = kkt.solution()
    keep = np.setdiff1d(np.arange(B), pick)
    assert np.array_equal(part[keep], ref[keep]) and np.array_equal(part[pick], sol0[pick])
    assert np.array_equal(kkt.inertia(), nneg0)
    with torch.cuda.stream(stream):
        d_c.copy_(c_old)
    # subset launch: new regularisation for the picked problems only; the others keep their bits
    kkt.launch(False)
    pn.sync()
    before, nneg_before = kkt.solution(), kkt.inertia()
    reg2 = reg.copy()
    reg2[pick] = 50.0
    kkt.set_primal_reg(reg2)
    kkt.launch_subset(idx.data_ptr(), len(pick))
    pn.sync()
    after = kkt.solution()
    assert np.array_equal(after[keep], before[keep]) and np.array_equal(kkt.inertia()[keep], nneg_before[keep])
    kkt.launch(False)
    pn.sync()
    full = kkt.solution()
    assert np.array_equal(full[pick], after[pick]) and np.array_equal(full[keep], before[keep])
    kkt.set_primal_reg(None)
    # barrier diagonal (DIAG kernels): random values on variable and constraint rows, K checked against the host
    diag = np.random.default_rng(bw + 1).uniform(0.0, 2.0, (B, kkt.dim))
    diag[:, nz:] *= -1.0
    d_diag = torch.as_tensor(sqp._CudaArray(kkt.device_pointer(5), (B, kkt.dim)), device=dev)
    with torch.cuda.stream(stream):
        d_diag.copy_(torch.as_tensor(diag, device=dev))
    kkt.launch(False)
    pn.sync()
    sol_d = kkt.solution()
    ii = np.arange(kkt.dim)
    shift = np.where(ii < nz, 0.0, -1.0e-6)
    for b in (0, B // 2, B - 1):
        Kd, hh = _host_system(pn, mode, cb, b, lam, blocks, 0.0, 0.0)
        Kd[ii, ii] = Kd[ii, ii] + (shift + diag[b])          # the kernel adds (regularisation + diagonal) to the entry
        assert np.array_equal(kkt.matrix(b), Kd), b
        _check_factor(kkt, b, Kd, hh, perm, sol_d)
    with torch.cuda.stream(stream):
        d_diag.zero_()
    # pinned variables: identity rows and columns, zero right-hand side, the reduced system's solution
    kkt.launch(False)
    pn.sync()
    K0, h0 = kkt.matrix(2), kkt.rhs()[2]
    full = kkt.solution()
    n, m = key[0], key[1]
    fixed = np.zeros(nz, dtype=bool)
    fixed[:n] = True                                     # the first knot's states
    fixed[nz - n + 1] = True                             # and one of the last knot's
    kkt.set_fixed(fixed)
    kkt.launch(False)
    pn.sync()
    sol_f = kkt.solution()
    fx = np.nonzero(fixed)[0]
    Kref, href = K0.copy(), h0.copy()
    Kref[fx, :] = 0.0
    Kref[:, fx] = 0.0
    Kref[fx, fx] = 1.0
    href[fx] = 0.0
    assert np.array_equal(kkt.matrix(2), Kref) and np.array_equal(kkt.rhs()[2], href)
    assert np.all(sol_f[:, fx] == 0.0)
    dense = np.linalg.solve(Kref, href)
    assert np.max(np.abs(sol_f[2] - dense)) <= 1e3 * np.linalg.cond(Kref) * np.finfo(float).eps * max(1.0, np.max(np.abs(dense)))
    kkt.set_fixed(None)
    kkt.launch(False)
    pn.sync()
    assert np.array_equal(kkt.solution(), full)
    kkt.close()


def test_exact_mode_refuses_bandwidth_32(nlps):
    key = next(k for k, v in BAND_CASES.items() if v[0] == 32)
    pn = nlps(key, 3)
    pn.sync()
    l0 = pn.launch_count()
    with pytest.raises(_lib.DtoError) as e:
        PK.KKTSystem(pn)
    assert e.value.status == -7 and "exceeds 31" in str(e.value)
    assert pn.launch_count() == l0


# ----------------------------------------------------------------------------------------------------------------------
# the native solver with 32-lane KKT rows
# ----------------------------------------------------------------------------------------------------------------------
WIDE = (15, 2, 14, False)    # exact mode: half bandwidth 30 -> BW = 31
MID = (10, 2, 9, False)      # exact mode: half bandwidth 20 -> BW = 20


def _guess(model, B, seed):
    T, n, m = model["T"], model["n"], model["m"]
    rng = np.random.default_rng(seed)
    z = np.zeros((B, T * n + (T - 1) * m))
    for t in range(T):
        o = t * (n + m)
        z[:, o:o + n] = model["x1"] + (model["xT"] - model["x1"]) * t / (T - 1) + 0.3 * rng.normal(size=(B, n))
        if t < T - 1:
            z[:, o + n:o + n + m] = rng.normal(size=(B, m))
    return z


def _walk_exact(key, B, iters, u_bnd=None):
    kw = dict(band_kwargs(key), u_bnd=u_bnd)
    mo, mp = build_band(O, **kw), build_band(D, **kw)
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    z0 = _guess(mp, B, 5)
    perm, bw = PK.analyze(pn)
    assert bw == BAND_CASES[key][0]
    opts = sqp.SQPOptions(max_iter=iters, dual_reg=1.0e-6)
    ref = sqp.solve(OracleBackend(osolver, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band", options=opts), z0,
                    options=opts, record=True)
    native = lambda k: sqp.SQPOptions(max_iter=k, dual_reg=opts.dual_reg, bound_relax=1.0)     # noqa: E731
    for k in range(1, len(ref.history)):
        got = sqp.solve_native(pn, z0, options=native(k))
        hr = ref.history[k]
        assert np.max(np.abs(got.z - hr["z"]) / np.maximum(1.0, np.abs(hr["z"]))) < 1e-7, k
        assert np.allclose(got.lam, hr["lam"], rtol=1e-5, atol=1e-7), k
    got = sqp.solve_native(pn, z0, options=native(iters))
    assert np.array_equal(got.converged, ref.converged) and np.array_equal(got.iterations, ref.iterations)
    assert got.stats["iterations"] == len(ref.history)
    return pn, z0, native(iters), got, ref


@pytest.mark.parametrize("key", [WIDE, MID], ids=["bw30", "bw20"])
def test_native_solver_with_32_lane_rows_walks_through_the_oracle_twin(key, monkeypatch):
    """the inertia ladder runs (candidate slots: VIRT kernels at W = 32), and one try per pass gives the same bits"""
    pn, z0, opts, got, ref = _walk_exact(key, 5, 25)
    assert got.stats["refactorisations"] > 0
    both = got.converged & ref.converged
    assert both.any() and np.allclose(got.objective[both], ref.objective[both], rtol=1e-8)
    monkeypatch.setenv("DTO_SQP_LADDER", "1")
    seq = sqp.solve_native(pn, z0, options=opts)
    assert seq.stats["refactorisations"] > got.stats["refactorisations"]
    assert np.array_equal(seq.z, got.z) and np.array_equal(seq.lam, got.lam) and np.array_equal(seq.iterations, got.iterations)
    pn.close()


def test_native_interior_point_with_32_lane_rows_walks_through_the_oracle_twin():
    """|u| <= 0.5 (active) on the BW = 31 model: the barrier diagonal (DIAG) and candidate slots (DIAG + VIRT) at W = 32"""
    pn, z0, opts, got, ref = _walk_exact(WIDE, 3, 25, u_bnd=0.5)
    assert np.all(np.isfinite(got.z))
    n, m, T = WIDE[0], WIDE[1], band_kwargs(WIDE)["T"]
    U = np.stack([got.z[:, t * (n + m) + n + j] for t in range(T - 1) for j in range(m)], axis=1)
    assert np.all(np.abs(U) < 0.5)
    pn.close()


def test_native_knot_bfgs_with_17_variable_blocks_walks_through_the_oracle_twin():
    """knot blocks of 17 variables (k_qn_update with 32 lanes; the last knot's block has 15) in a KKT matrix of half
    bandwidth 31; B * T odd"""
    B, iters = 3, 25
    kw = dict(band_kwargs(QN_BAND), evaluate_hessian=False)
    mo, mp = build_band(O, **kw), build_band(D, **kw)
    osolver, pn = O.solver_from(mo), D.solver_from(mp, batch=B).nlp
    assert (B * mp["T"]) % 2 == 1
    perm, bw = PK.analyze(pn, hessian="knot-blocks")
    assert bw == 31
    xs, nx, _, nu = pn.knot_layout()
    assert max(int(nx[t] + nu[t]) for t in range(pn.T)) == 17
    opts = sqp.SQPOptions(max_iter=iters, dual_reg=1.0e-6)
    be = QNOracleBackend(osolver, pn, B, dual_reg=opts.dual_reg, perm=perm - 1, bw=bw, linear="band", options=opts)
    z0 = _guess(mp, B, 7)
    ref = sqp.solve(be, z0, options=opts, record=True)
    native = lambda k: sqp.SQPOptions(max_iter=k, dual_reg=opts.dual_reg, hessian_approximation="knot-bfgs", bound_relax=1.0)  # noqa: E731
    for k in range(1, len(ref.history)):
        got = sqp.solve_native(pn, z0, options=native(k))
        hr = ref.history[k]
        assert np.max(np.abs(got.z - hr["z"]) / np.maximum(1.0, np.abs(hr["z"]))) < 1e-7, k
        assert np.allclose(got.lam, hr["lam"], rtol=1e-5, atol=1e-5), k
    got = sqp.solve_native(pn, z0, options=native(iters))
    assert np.array_equal(got.converged, ref.converged) and np.array_equal(got.iterations, ref.iterations)
    assert not any(f.any() for f in be.first)          # every block of the twin took an update
    pn.close()

"""GPU tests beyond small-case parity: golden fixtures, full BASELINE sizes against the oracle's C
twin, size-independent properties (determinism, fused == separate, shard invariance, sigma
linearity), edge cases and C-ABI state errors. Everything goes through libdto.so."""
import os

import numpy as np
import pytest

import dto_b200 as D
from dto_b200 import _lib
from dto_b200.evaluator import A_H, A_J, A_Z
from examples import models as M
from golden.make_golden import GOLDEN, tag
from oracle import api as O
from oracle import cgen
from util import KERNEL_VARIANTS, assert_close, make_inputs

pytestmark = pytest.mark.gpu
HERE = os.path.join(os.path.dirname(__file__), "golden")


def _eval_all(pn, z, lam, sigma, w):
    B = z.shape[0]
    if pn.num_parameter:
        pn.set_parameters(w)
    out = dict(f=pn.eval_objective(z), g=np.full((B, pn.num_variables), np.nan), c=np.full((B, pn.num_constraint), np.nan),
               J=np.full((B, pn.num_jacobian), np.nan), H=np.full((B, pn.num_hessian), np.nan))
    pn.eval_objective_gradient(out["g"])
    pn.eval_constraint(out["c"])
    pn.eval_constraint_jacobian(out["J"])
    if pn.hessian_lagrangian:
        pn.eval_hessian_lagrangian(out["H"], None, sigma, lam)
    else:  # evaluate_hessian=False problems (src/moi.jl:122: features without :Hess): no slots, no values
        out["H"] = np.zeros((B, 0))
    return out


@pytest.mark.parametrize("name,kw,B,config", GOLDEN, ids=[tag(g[0], g[1]) for g in GOLDEN])
def test_cuda_matches_golden(name, kw, B, config):
    fx = np.load(os.path.join(HERE, tag(name, kw) + ".npz"))
    pn = D.solver_from(M.BUILDERS[name](D, **kw), batch=B).nlp
    r, c = pn.jacobian_structure_arrays()
    assert np.array_equal(np.stack([r, c], 1), fx["jac_structure"])
    out = _eval_all(pn, fx["z"], fx["lam"], fx["sigma"], fx["w"])
    for k in ("f", "g", "c", "J") + (("H",) if pn.hessian_lagrangian else ()):
        assert_close(f"{name} {k}", out[k], fx[k])
    pn.close()


FULL = [
    ("cartpole", dict(T=101), 4096, 2),          # BASELINE configs[1]
    ("acrobot", dict(T=101), 4096, 3),           # configs[2] (callbacks)
    ("car", dict(T=201, obstacle="general"), 16384, 4),  # configs[3]
    ("cartpole", dict(T=1001), 257, 5),          # configs[4] long horizon, ragged batch
]


@pytest.mark.parametrize("name,kw,B,config", FULL, ids=[f"{f[0]}-T{f[1]['T']}-B{f[2]}" for f in FULL])
def test_full_size_vs_c_oracle_and_properties(name, kw, B, config):
    mo = M.BUILDERS[name](O, **kw)
    mp = M.BUILDERS[name](D, **kw)
    osolver = O.solver_from(mo)
    shared = bool(mo.get("shared_parameters"))
    if shared:
        osolver.set_parameters([np.zeros(8) for _ in range(mo["T"])] + [np.zeros(0)])
    co = cgen.build_c_oracle(osolver, tag(name, kw), shared_parameters=shared, cse=True)
    pn = D.solver_from(mp, batch=B).nlp
    z, lam, sigma, w = make_inputs(name, mp, pn.num_variables, pn.num_constraint, pn.num_parameter, B, config)
    ref = co.eval(31, z, lam, sigma, w)
    out = _eval_all(pn, z, lam, sigma, w)
    for k in ("f", "g", "c", "J", "H"):
        assert_close(f"{name} {k}", out[k], ref[k])
    # fused pass vs separate passes: same values (separately compiled programs may contract FMAs
    # differently, so this is a tolerance check); repeat runs are bit-identical (fixed gather order)
    J2, H2 = np.empty_like(out["J"]), np.empty_like(out["H"])
    pn.eval_jacobian_hessian(J2, H2)
    assert_close("fused J", J2, ref["J"])
    assert_close("fused H", H2, ref["H"])
    assert np.allclose(J2, out["J"], rtol=1e-13, atol=1e-15) and np.allclose(H2, out["H"], rtol=1e-13, atol=1e-15)
    J3, H3 = np.empty_like(J2), np.empty_like(H2)
    pn.eval_jacobian_hessian(J3, H3)
    assert np.array_equal(J3, J2) and np.array_equal(H3, H2)
    # shard invariance: three logical shards on one device give the identical bits (no cross-problem coupling)
    ps = pn.new_batch(devices=[0, 0, 0])
    if ps.num_parameter:
        ps.set_parameters(w)
    J4, H4 = np.empty_like(J2), np.empty_like(H2)
    ps.eval_jacobian_hessian(J4, H4, z, sigma, lam)
    assert _lib.lib().dto_batch_num_shards(ps.handle) == 3
    assert np.array_equal(J4, J2) and np.array_equal(H4, H2)
    # one-problem read-back (per-Ipopt driver path) and get_trajectory semantics
    b = B // 2
    row = np.empty(pn.num_hessian)
    _lib.check(_lib.lib().dto_get_problem(pn.handle, A_H, b, row.ctypes.data))
    assert np.array_equal(row, H2[b])
    assert np.array_equal(pn.last_x(b), z[b])
    ps.close()
    pn.close()


def test_in_process_shards_over_all_visible_devices_are_bit_identical():
    """The in-process multi-device path of libdto.so (one host thread, one stream per shard, contiguous shards,
    host gather = each shard's D2H into its slice; SURVEY 8e): the batch is spread over EVERY visible device --
    and over at least three shards, so the path is exercised on a one-GPU box too (a device may be listed more
    than once) -- and all five callbacks + the fused pass + the KKT consumer must reproduce the one-shard bits."""
    from dto_b200 import kkt as PK
    ndev = _lib.lib().dto_device_count()
    devices = [d % ndev for d in range(max(3, ndev))]
    name, kw, B, config = "cartpole", dict(T=11), 1000, 2     # 1000 problems: ragged shards (334, 334, 332)
    mp = M.BUILDERS[name](D, **kw)
    one = D.solver_from(mp, batch=B, devices=[0]).nlp
    many = D.solver_from(mp, batch=B, devices=devices).nlp
    assert many.num_shards == len(devices) and sorted({many.shard_device(i) for i in range(many.num_shards)}) == sorted(set(devices))
    assert sum(many.shard_range(i)[1] for i in range(many.num_shards)) == B
    z, lam, sigma, w = make_inputs(name, mp, one.num_variables, one.num_constraint, one.num_parameter, B, config)
    a, b = _eval_all(one, z, lam, sigma, w), _eval_all(many, z, lam, sigma, w)
    for k in ("f", "g", "c", "J", "H"):
        assert np.array_equal(a[k], b[k]), k
    Ja, Ha, Jb, Hb = (np.empty_like(a[k]) for k in ("J", "H", "J", "H"))
    one.eval_jacobian_hessian(Ja, Ha, z, sigma, lam)
    many.eval_jacobian_hessian(Jb, Hb, z, sigma, lam)
    assert np.array_equal(Ja, Jb) and np.array_equal(Ha, Hb)
    k1, k2 = PK.KKTSystem(one), PK.KKTSystem(many)
    s1, s2 = np.empty((B, k1.dim)), np.empty((B, k2.dim))
    k1.solve(s1, variables=z, scaling=sigma, duals=lam)
    k2.solve(s2, variables=z, scaling=sigma, duals=lam)
    assert np.array_equal(s1, s2)
    assert np.array_equal(k1.inertia(), k2.inertia()) and np.all(k1.inertia() == one.num_constraint)
    k1.close(); k2.close(); one.close(); many.close()


def test_sigma_linearity_and_dual_linearity():
    """H(sigma, lambda) = sigma * H_cost + H_constraints(lambda), linear in each."""
    mp = M.build_acrobot(D, T=21)
    B = 37
    pn = D.solver_from(mp, batch=B).nlp
    z, lam, sigma, w = make_inputs("acrobot", mp, pn.num_variables, pn.num_constraint, 0, B, 3)
    H = {}
    for key, (s, l) in {"00": (0.0, 0 * lam), "10": (1.0, 0 * lam), "20": (2.0, 0 * lam), "01": (0.0, lam), "02": (0.0, 2 * lam),
                        "11": (1.0, lam)}.items():
        H[key] = np.empty((B, pn.num_hessian))
        pn.eval_hessian_lagrangian(H[key], z, s, l)
    assert np.all(H["00"] == 0.0)
    assert np.allclose(H["20"], 2 * H["10"], rtol=1e-15, atol=0)
    assert np.allclose(H["02"], 2 * H["01"], rtol=1e-13, atol=1e-15)
    assert np.allclose(H["11"], H["10"] + H["01"], rtol=1e-13, atol=1e-15)
    pn.close()


@pytest.mark.parametrize("B", [1, 2, 31, 32, 33, 65])
def test_ragged_batches_and_min_horizon(B):
    """Warp tiles straddle problem boundaries: every batch size / horizon must give the same rows."""
    for name, kw in (("pendulum", dict(T=2)), ("pendulum", dict(T=3)), ("cartpole", dict(T=7))):
        mo, mp = M.BUILDERS[name](O, **kw), M.BUILDERS[name](D, **kw)
        osolver = O.solver_from(mo)
        shared = bool(mo.get("shared_parameters"))
        if shared:
            osolver.set_parameters([np.zeros(8) for _ in range(mo["T"])] + [np.zeros(0)])
        co = cgen.build_c_oracle(osolver, tag(name, kw), shared_parameters=shared, cse=True)
        pn = D.solver_from(mp, batch=B).nlp
        z, lam, sigma, w = make_inputs(name, mp, pn.num_variables, pn.num_constraint, pn.num_parameter, B, 8)
        ref = co.eval(31, z, lam, sigma, w)
        out = _eval_all(pn, z, lam, sigma, w)
        for k in ("f", "g", "c", "J", "H"):
            assert_close(f"{name}{kw} B={B} {k}", out[k], ref[k])
        pn.close()


def test_state_errors_and_hessian_switch():
    mp = M.build_pendulum(D)
    pn = D.solver_from(mp, batch=2).nlp
    with pytest.raises(_lib.DtoError) as e:
        pn.eval_objective()
    assert e.value.status == -6  # before dto_set_x
    z = np.zeros((2, pn.num_variables))
    pn.eval_objective(z)
    H = np.empty((2, pn.num_hessian))
    with pytest.raises(_lib.DtoError) as e:
        pn.eval_hessian_lagrangian(H)
    assert e.value.status == -6  # before dto_set_duals
    with pytest.raises(ValueError):
        pn.set_x(np.zeros((3, pn.num_variables)))
    pn.close()
    # a Cost without evaluate_hessian: the reference throws (Q9); we return DTO_ERR_NO_HESSIAN
    mp = M.build_cartpole(D, T=5, evaluate_hessian=False)
    pn = D.solver_from(mp, batch=2).nlp
    pn.set_parameters(np.zeros((2, 8)))
    pn.set_x(np.zeros((2, pn.num_variables)))
    pn.set_duals(1.0, np.zeros((2, pn.num_constraint)))
    with pytest.raises(_lib.DtoError) as e:
        pn.eval_hessian_lagrangian(np.empty((2, 0)))
    assert e.value.status == -5
    J = np.empty((2, pn.num_jacobian))
    pn.eval_constraint_jacobian(J)  # Jacobian still fine
    assert np.isfinite(J).all()
    pn.close()


def test_nan_inf_pass_through():
    """Non-finite values are handed back unchanged, like the reference (no status codes for them)."""
    mp = M.build_pendulum(D)
    pn = D.solver_from(mp, batch=3).nlp
    z = np.random.default_rng(0).uniform(size=(3, pn.num_variables))
    z[1, 0] = np.nan
    z[2, 3] = np.inf
    f = pn.eval_objective(z)
    assert np.isfinite(f[0]) and np.isnan(f[1]) and not np.isfinite(f[2])
    pn.close()


@pytest.mark.parametrize("mode", ["sympy", "dag"])
def test_symbolic_derivative_mode_matches(mode, monkeypatch):
    """DTO_DERIV=sympy lowers the expanded symbolic derivative expressions (the literal form the
    reference's closures hold), DTO_DERIV=dag the plain forward propagation without cut nodes; both must
    agree with the oracle like the default hierarchical mode does."""
    monkeypatch.setenv("DTO_DERIV", mode)
    for name, kw, B, config in [("pendulum", dict(), 4, 1), ("cartpole", dict(T=11), 3, 2)]:
        fx = np.load(os.path.join(HERE, tag(name, kw) + ".npz"))
        pn = D.solver_from(M.BUILDERS[name](D, **kw), batch=B).nlp
        out = _eval_all(pn, fx["z"], fx["lam"], fx["sigma"], fx["w"])
        for k in ("f", "g", "c", "J", "H"):
            assert_close(f"sympy-mode {name} {k}", out[k], fx[k])
        pn.close()


def test_table_gather_fallback_matches(monkeypatch):
    """Shapes whose per-knot recipes are not compiled into the model library use the generic
    table-driven Hessian gather; force it and check it against the golden fixtures too."""
    monkeypatch.setenv("DTO_TABLE_GATHER", "1")
    for name, kw, B, config in [("acrobot", dict(T=9), 3, 3), ("car", dict(T=12, obstacle="general"), 3, 4),
                                ("acrobot_hessian_test", dict(), 5, 6)]:
        fx = np.load(os.path.join(HERE, tag(name, kw) + ".npz"))
        pn = D.solver_from(M.BUILDERS[name](D, **kw), batch=B).nlp
        assert not pn.compiled_gather()
        out = _eval_all(pn, fx["z"], fx["lam"], fx["sigma"], fx["w"])
        for k in ("f", "g", "c", "J", "H"):
            assert_close(f"table-gather {name} {k}", out[k], fx[k])
        pn.close()
    monkeypatch.delenv("DTO_TABLE_GATHER")
    pn = D.solver_from(M.build_acrobot(D, T=9), batch=3).nlp
    assert pn.compiled_gather()


VARIANT_MODELS = [("pendulum", dict(), 1), ("cartpole", dict(T=11), 2), ("acrobot", dict(T=9), 3),
                  ("car", dict(T=12, obstacle="general"), 4)]


@pytest.mark.parametrize("tune", KERNEL_VARIANTS)
def test_kernel_variants_match_golden_and_each_other(tune, monkeypatch):
    """The three per-knot kernels (plain one-tile-per-warp, persistent bulk-copy pipeline, warp-specialised)
    run the same generated element code and the same += order, so they must agree with the golden
    fixtures AND with the default selection to a few ulps (the compiler may contract a multiply of an
    element term into the slot sum in one kernel and not in another, so not bit for bit), on batches
    large enough for many tiles that straddle problem boundaries. DTO_TUNE forces: the plain kernel everywhere / the persistent kernel
    for every Hessian pass / the specialised kernel for every Hessian pass (also of light models)."""
    for name, kw, config in VARIANT_MODELS:
        fx = np.load(os.path.join(HERE, tag(name, kw) + ".npz"))
        B0 = fx["z"].shape[0]
        reps = 40  # B0*reps problems: dozens of warp tiles
        z, lam, sigma, w = (np.tile(fx[k], (reps,) + (1,) * (fx[k].ndim - 1)) for k in ("z", "lam", "sigma", "w"))
        res = {}
        for t in ("", tune):
            if t:
                monkeypatch.setenv("DTO_TUNE", t)
            else:
                monkeypatch.delenv("DTO_TUNE", raising=False)
            pn = D.solver_from(M.BUILDERS[name](D, **kw), batch=B0 * reps).nlp
            out = _eval_all(pn, z, lam, sigma, w)
            J2, H2 = np.full_like(out["J"], np.nan), np.full_like(out["H"], np.nan)
            pn.eval_jacobian_hessian(J2, H2, z, sigma, lam)
            out["J2"], out["H2"] = J2, H2
            res[t] = out
            pn.close()
        monkeypatch.delenv("DTO_TUNE", raising=False)
        for k in ("f", "g", "c", "J", "H"):
            assert_close(f"{tune} {name} {k}", res[tune][k][:B0], fx[k])
        # same element code in every kernel: a few ulps; bf=0 swaps the branch-free sin/cos/reciprocal of the
        # default build for the library's (each < 1 ulp, but not the same bits), so it is held to the oracle
        # tolerance instead
        rt, at = (1e-12, 1e-14) if "bf=0" in tune else (1e-14, 1e-16)
        for k in ("g", "c", "J", "H", "J2", "H2"):
            assert_close(f"{tune} vs default {name} {k}", res[tune][k], res[""][k], rtol=rt, atol=at)
        assert_close(f"{tune} fused J {name}", res[tune]["J2"], res[tune]["J"], rtol=1e-14, atol=1e-16)
        assert_close(f"{tune} fused H {name}", res[tune]["H2"], res[tune]["H"], rtol=1e-14, atol=1e-16)


def test_branch_free_math_falls_back_outside_its_domain(monkeypatch):
    """The default build (DTO_TUNE bf=1) replaces sin/cos/reciprocal inside the generated element programs by
    branch-free versions (one basic block); arguments outside their domain (|angle| >= 2^31, NaN, Inf, reciprocals of
    denormal / huge values) must re-evaluate with the library functions and give the default path's
    values, problem by problem."""
    name, kw = "cartpole", dict(T=11)
    fx = np.load(os.path.join(HERE, tag(name, kw) + ".npz"))
    z, lam, sigma, w = (np.tile(fx[k], (4,) + (1,) * (fx[k].ndim - 1)).copy() for k in ("z", "lam", "sigma", "w"))
    z[1, 1] = 3.0e10       # pole angle far beyond 2^31 at knot 0
    z[2, 6] = -7.5e12      # and at knot 1
    z[3, 3] = np.nan
    z[4, 11] = np.inf
    z[5, 1] = 2.0 ** 31    # boundary of the fast path
    res = {}
    for t in ("bf=0,emit=0", ""):
        if t:
            monkeypatch.setenv("DTO_TUNE", t)
        else:
            monkeypatch.delenv("DTO_TUNE", raising=False)
        pn = D.solver_from(M.BUILDERS[name](D, **kw), batch=z.shape[0]).nlp
        res[t] = _eval_all(pn, z, lam, sigma, w)
        pn.close()
    monkeypatch.delenv("DTO_TUNE", raising=False)
    for k in ("c", "J", "H"):
        a, b = res[""][k], res["bf=0,emit=0"][k]
        assert np.array_equal(np.isnan(a), np.isnan(b)), f"{k}: NaN pattern differs"
        fin = np.isfinite(b)
        assert_close(f"bf=1 {k}", a[fin], b[fin], rtol=1e-12, atol=1e-14)
    assert np.isfinite(res[""]["J"][1]).all() and np.isfinite(res[""]["H"][2]).all()
    assert "dto_sincos_bf" in open(D.solver_from(M.BUILDERS[name](D, **kw), batch=1).model.path.replace(".so", ".cu")).read()

"""Host-side checks of the derivative synthesis (ir.py): the hierarchical (cut-based) derivatives are the
same functions as the plain second-order forward propagation and as sympy's expanded derivatives -- the
expressions the reference's Symbolics closures evaluate (/root/reference/src/dynamics.jl:24-35) -- and the
user-Jacobian constructor (src/dynamics.jl:59-101) lowers the USER's expressions, exact or not."""
import numpy as np
import pytest
import sympy as sp

import dto_b200 as D
from dto_b200 import codegen
from dto_b200.ir import Graph, choose_cuts, count_ops, hierarchical
from examples import models as M


def _graph(el):
    g, sym = Graph(), {}
    for cname, syms in el.args.items():
        for i, s_ in enumerate(syms):
            sym[s_] = g.inp(cname, i)
    memo = {}
    res = [g.from_sympy(e, sym, memo) for e in el.evaluate]
    wrt = [sym[v] for v in el.vars]
    L = res[0] if el.role == "cost" else g.sum(g.mul(sym[l], rn) for l, rn in zip(el.lam, res))
    return g, sym, res, wrt, L


def _patterns(el):
    hpat = [(min(r, c) - 1, max(r, c) - 1) for r, c in zip(el.hess_rows, el.hess_cols)]
    jpat = [(r - 1, c - 1) for r, c in zip(el.jac_rows, el.jac_cols)]
    return jpat, hpat, (lambda j, H, h: [j[r].get(c, h.ZERO) for r, c in jpat] + [H.get(k, h.ZERO) for k in hpat])


def _inputs(el, rng):
    return {(cname, i): float(rng.normal() * 1.3) for cname, syms in el.args.items() for i in range(len(syms))}


@pytest.mark.parametrize("name,kw,max_evals", [("cartpole", dict(T=4), 700), ("acrobot", dict(T=4), 700),
                                                ("acrobot_hessian_test", dict(), 400), ("pendulum", dict(), 50)])
def test_hierarchical_equals_plain_forward(name, kw, max_evals):
    mp = M.BUILDERS[name](D, **kw)
    el = mp["dynamics"][0].spec
    g, sym, res, wrt, L = _graph(el)
    jpat, hpat, fused = _patterns(el)
    cuts, st = choose_cuts(g, res, L, wrt, fused, max_evals=max_evals)
    j0, H0 = hierarchical(g, res, L, wrt, [])
    j1, H1 = hierarchical(g, res, L, wrt, cuts)
    assert set(H1) <= set(hpat) and all(set(j1[i]) <= {c for r, c in jpat if r == i} for i in range(len(res)))
    n0, n1 = fused(j0, H0, g), fused(j1, H1, g)
    assert sum(count_ops(g, n1).values()) == st["ops"] <= st["plain"] == sum(count_ops(g, n0).values())
    if name in ("cartpole", "acrobot"):
        assert cuts and st["ops"] < 0.85 * st["plain"]  # the cuts are what the default mode is for
    rng = np.random.default_rng(7)
    for _ in range(8):
        inp = _inputs(el, rng)
        a, b = np.array(g.evaluate(n0, inp)), np.array(g.evaluate(n1, inp))
        assert np.all(np.abs(a - b) <= 1e-12 * np.maximum(1.0, np.abs(a))), (name, np.max(np.abs(a - b)))


def test_hierarchical_equals_sympy_derivatives():
    """against the expanded symbolic derivatives (what Symbolics hands to build_function) in 40-digit arithmetic"""
    import mpmath
    mp = M.BUILDERS["acrobot"](D, T=4)
    el = mp["dynamics"][0].spec
    g, sym, res, wrt, L = _graph(el)
    jpat, hpat, fused = _patterns(el)
    cuts, _ = choose_cuts(g, res, L, wrt, fused, max_evals=500)
    j1, H1 = hierarchical(g, res, L, wrt, cuts)
    nodes = fused(j1, H1, g)
    exact = list(el.jac) + list(el.hess)
    allsyms = [s_ for syms in el.args.values() for s_ in syms]
    f = sp.lambdify(allsyms, exact, modules="mpmath")
    rng = np.random.default_rng(11)
    mpmath.mp.dps = 40
    for _ in range(3):
        inp = _inputs(el, rng)
        vals = [mpmath.mpf(inp[(cname, i)]) for cname, syms in el.args.items() for i in range(len(syms))]
        ref = np.array([float(v) for v in f(*vals)])
        got = np.array(g.evaluate(nodes, inp))
        assert np.all(np.abs(got - ref) <= 1e-12 * np.abs(ref) + 1e-14), np.max(np.abs(got - ref))


def _user_jac_dynamics(scale):
    def f(y, x, u, w):
        return y - (x + 0.1 * M.arr(x[1], u[0] - M.sin(x[0])))

    def fj(J, y, x, u, w):  # scale != 1: deliberately NOT the derivative of f
        J[0, 0], J[0, 1], J[0, 3] = -1.0, -0.1, 1.0
        J[1, 0], J[1, 1], J[1, 2], J[1, 4] = scale * 0.1 * M.cos(x[0]), -1.0, -0.1, 1.0

    return D.Dynamics(f, fj, 2, 2, 1)


@pytest.mark.parametrize("mode", ["hier", "dag", "sympy"])
def test_user_jacobian_is_what_gets_lowered(mode, monkeypatch):
    """ADVICE r1: the reference calls the user's closure (src/dynamics.jl:59-64); every derivative mode must
    emit THOSE expressions, and two user Jacobians for one f are two different model libraries."""
    monkeypatch.setenv("DTO_DERIV", mode)
    srcs, hashes = [], []
    for scale in (1.0, 3.0):
        d = _user_jac_dynamics(scale)
        assert d.spec.user_jac
        spec = codegen.ModelSpec(name="uj", dyn=[d.spec], cost=[], stage=[])
        hashes.append(codegen.spec_hash(spec))
        src, _ = codegen.emit_model(spec, hashes[-1])
        srcs.append(src[src.index("dyn0_jac("):src.index("dyn0_hess(")])
    assert hashes[0] != hashes[1]
    assert srcs[0] != srcs[1]
    assert "0.3" in srcs[1] or "dto_k" in srcs[1]  # 3 * 0.1 * cos(x0): the scaled coefficient reached the code
    if mode != "sympy":
        d = _user_jac_dynamics(3.0)
        g, sym, res, wrt, L = _graph(d.spec)
        nodes = [g.from_sympy(e, sym, {}) for e in d.spec._jac]
        inp = {("y", 0): 0.1, ("y", 1): 0.2, ("x", 0): 0.7, ("x", 1): -0.4, ("u", 0): 0.3}
        vals = g.evaluate(nodes, inp)
        assert abs(vals[1] - 3.0 * 0.1 * np.cos(0.7)) < 1e-15 and len(vals) == 10


@pytest.mark.parametrize("tune", ["pdl_plain=0", "emit=1", "ws_helpers=3", "ws=yes", "ws"])
def test_unsupported_tuning_is_refused(tune, monkeypatch):
    """A retired or misspelt DTO_TUNE key, or a value no build supports, is an error naming the accepted keys: it must
    not build the default kernels under a new content hash."""
    monkeypatch.setenv("DTO_TUNE", tune)
    with pytest.raises(ValueError, match=r"accepted: ws=1\|0, persist=1\|0"):
        codegen._tuning()
    monkeypatch.setenv("DTO_TUNE", "ws=0, persist=0")
    t = codegen._tuning()
    assert (t["ws"], t["persist"], t["emit"]) == (0, 0, 2)

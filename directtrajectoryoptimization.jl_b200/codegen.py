"""Code generator: element expressions -> CUDA device functions -> model library (.so).

This is the "new codegen stage" of the north star: it takes the symbolic expressions the
element constructors build (what /root/reference/src/dynamics.jl:24-35, src/costs.jl:19-27,
src/constraints.jl:28-40, src/general_constraint.jl:24-36 feed to `build_function`) and,
instead of `eval`-ing one un-shared closure per output, lowers ALL outputs that are
evaluated at the same knot in the same pass (e.g. Jacobian + Hessian of one dynamics
element) through one common-subexpression-eliminated straight-line FP64 program, emitted as
a `__device__` function that the hand-written kernels of csrc/dto_kernels.cuh inline.

One model library = one translation unit = generated `struct DtoModel` + dto_kernels.cuh,
compiled by nvcc for sm_100a and exporting `dto_model_entry()` (csrc/dto_model_abi.h).
Libraries are content-addressed (the reference's "#TODO: option to load/save methods",
src/dynamics.jl:22) and cached in-tree under _models/.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import sympy as sp

CODEGEN_VERSION = "9"
PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
MODEL_DIR = os.path.join(PKG_DIR, "_models")
# libraries (and cut searches) missing from MODEL_DIR are generated here; DTO_CACHE_DIR points it elsewhere, so that a
# process that must not write into the source tree (bench.py) still reuses what the build left in MODEL_DIR
CACHE_DIR = os.environ.get("DTO_CACHE_DIR") or MODEL_DIR
NVCC = os.environ.get("DTO_NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]


def _deriv_mode() -> str:
    """"hier" (default): derivatives synthesised on the residual DAG with automatically chosen cut
    nodes as local differentiation variables (ir.hierarchical; cartpole-RK3: 698 instead of 1241 FP64
    operations per knot). "dag": the same without cuts = plain sparse second-order forward propagation.
    "sympy": lower the expanded symbolic derivative expressions (what the reference's Symbolics closures
    hold) through tree CSE -- the literal drop-in input, kept as a cross-check path. All three are CUDA."""
    m = os.environ.get("DTO_DERIV", "hier")
    if m not in ("hier", "dag", "sympy"):
        raise ValueError("DTO_DERIV must be 'hier', 'dag' or 'sympy'")
    return m


# DTO_TUNE keys: the accepted values, the default first. ws / persist: use the warp-specialised / persistent kernel
# where the shape allows; ws_all: the warp-specialised kernel for the passes without a Hessian too; ws_plan: its
# precomputed tile plans; ws_helpers: its helper warps; bf: branch-free sin/cos/reciprocal; emit: statement order of
# the element programs (2: register-pressure-aware list scheduling, 0: DFS post-order)
TUNE_VALUES = {"ws": (1, 0), "persist": (1, 0), "ws_all": (0, 1), "ws_plan": (1, 0), "ws_helpers": (8, 4), "bf": (1, 0),
               "emit": (2, 0)}


def _tuning() -> Dict[str, int]:
    """Compile-time kernel selection (part of the content hash); override with DTO_TUNE="ws=0,persist=0"."""
    t = {k: v[0] for k, v in TUNE_VALUES.items()}
    for kv in os.environ.get("DTO_TUNE", "").split(","):
        if not kv.strip():
            continue
        k, _, v = kv.partition("=")
        k = k.strip()
        if k not in TUNE_VALUES or not v.strip().lstrip("-").isdigit() or int(v) not in TUNE_VALUES[k]:
            raise ValueError(f"DTO_TUNE: {kv.strip()!r} is not supported; accepted: "
                             + ", ".join(f"{n}={'|'.join(map(str, vs))}" for n, vs in TUNE_VALUES.items()))
        t[k] = int(v)
    return t


# ----------------------------------------------------------------------------- specs
@dataclass
class ElementSpec:
    """One element kind. `args` maps C argument name -> list of symbols (in order)."""
    role: str                      # 'dyn' | 'cost' | 'stage'
    n_out: int
    nx: int
    nu: int
    nw: int
    args: Dict[str, Sequence[sp.Symbol]]
    evaluate: List[sp.Expr]
    jac_rows: List[int]
    jac_cols: List[int]
    has_hess: bool
    hess_rows: List[int] = field(default_factory=list)
    hess_cols: List[int] = field(default_factory=list)
    ineq: List[int] = field(default_factory=list)
    vars: Sequence[sp.Symbol] = ()         # differentiation variables in order ([x;u;y] or [x;u])
    lam: Sequence[sp.Symbol] = ()          # multipliers of the element's outputs (not for costs)
    _jac: Optional[List[sp.Expr]] = None   # expanded symbolic derivatives, built on demand
    user_jac: bool = False                 # _jac holds the USER's Jacobian expressions (Dynamics(f, jacobian, ...))
    _hess: Optional[List[sp.Expr]] = None  # (only the "sympy" derivative mode lowers these)

    @property
    def nnz_jac(self) -> int:
        return len(self.jac_rows)

    @property
    def nnz_hess(self) -> int:
        return len(self.hess_rows) if self.has_hess else 0

    @property
    def lagrangian(self) -> sp.Expr:
        if self.role == "cost":
            return self.evaluate[0]
        acc = sp.Integer(0)
        for l, e in zip(self.lam, self.evaluate):
            acc = acc + l * e
        return acc

    @property
    def jac(self) -> List[sp.Expr]:
        if self._jac is None:
            from . import symbolic as S
            self._jac = S.jacobian_values(self.evaluate, list(self.vars), self.jac_rows, self.jac_cols)
        return self._jac

    @property
    def hess(self) -> List[sp.Expr]:
        if self._hess is None:
            from . import symbolic as S
            self._hess = (S.hessian_values(self.lagrangian, list(self.vars), self.hess_rows, self.hess_cols)
                          if self.has_hess else [])
        return self._hess


@dataclass
class GeneralSpec:
    num_variables: int
    num_parameter: int
    args: Dict[str, Sequence[sp.Symbol]]   # 'z', 'w', 'lam'
    evaluate: List[sp.Expr]
    jac_rows: List[int]
    jac_cols: List[int]
    jac: List[sp.Expr]
    has_hess: bool
    hess_rows: List[int] = field(default_factory=list)
    hess_cols: List[int] = field(default_factory=list)
    hess: List[sp.Expr] = field(default_factory=list)
    ineq: List[int] = field(default_factory=list)


@dataclass
class ModelSpec:
    name: str
    dyn: List[ElementSpec]
    cost: List[ElementSpec]
    stage: List[ElementSpec]
    general: Optional[GeneralSpec] = None
    hg_classes: List[tuple] = field(default_factory=list)   # compiled gather recipes (recipes.py)
    hg_meta: List[tuple] = field(default_factory=list)      # per class: (own cost terms, own dynamics terms, previous knot's cost terms)


# ----------------------------------------------------------------------------- C printing
_CFUN = {"sin": "sin", "cos": "cos", "tan": "tan", "exp": "exp", "log": "log", "atan": "atan", "asin": "asin",
         "acos": "acos", "sinh": "sinh", "cosh": "cosh", "tanh": "tanh", "Abs": "fabs", "atan2": "atan2",
         "sign": "dto_sign"}


def _lit(v: float) -> str:
    r = repr(float(v))
    if "e" not in r and "." not in r and "inf" not in r and "nan" not in r:
        r += ".0"
    return r


def cstr(e: sp.Expr, names: Dict[sp.Symbol, str]) -> str:
    """Fully parenthesised C for one expression; numbers printed with repr (17 digits)."""
    if e.is_Symbol:
        return names[e]
    if e.is_Number or e.is_NumberSymbol:
        v = float(e)
        return _lit(v) if v >= 0 else f"({_lit(v)})"
    if e.is_Add:
        return "(" + " + ".join(cstr(a, names) for a in e.args) + ")"
    if e.is_Mul:
        num, den = [], []
        for a in e.args:
            if a.is_Pow and a.args[1].is_Integer and int(a.args[1]) < 0:
                den.append(_pow_c(a.args[0], -int(a.args[1]), names))
            else:
                num.append(cstr(a, names))
        n = "*".join(num) if num else "1.0"
        if den:
            d = "*".join(den)
            return f"(({n})/({d}))" if len(den) > 1 or len(num) > 1 else f"({n}/{d})"
        return "(" + n + ")"
    if e.is_Pow:
        b, p = e.args
        if p.is_Integer:
            k = int(p)
            if k < 0:
                return f"(1.0/{_pow_c(b, -k, names)})"
            return _pow_c(b, k, names)
        if p == sp.Rational(1, 2) or (p.is_Float and float(p) == 0.5):
            return f"sqrt({cstr(b, names)})"
        if p.is_Float and float(p) == int(float(p)):
            k = int(float(p))
            return f"(1.0/{_pow_c(b, -k, names)})" if k < 0 else _pow_c(b, k, names)
        return f"pow({cstr(b, names)}, {cstr(p, names)})"
    if isinstance(e, sp.Piecewise):
        out = "0.0"
        for val, cond in reversed(e.args):
            out = cstr(val, names) if cond is sp.true else f"(({cstr(cond, names)}) ? {cstr(val, names)} : {out})"
        return out
    if e.is_Relational:
        return f"({cstr(e.lhs, names)} {e.rel_op} {cstr(e.rhs, names)})"
    if e.is_Function:
        fn = _CFUN.get(e.func.__name__)
        if fn is None:
            raise NotImplementedError(f"no CUDA lowering for function {e.func}")
        return fn + "(" + ", ".join(cstr(a, names) for a in e.args) + ")"
    raise NotImplementedError(f"no CUDA lowering for node {type(e)}")


def _pow_c(b: sp.Expr, k: int, names) -> str:
    bs = cstr(b, names)
    if k == 1:
        return bs
    return f"dto_powi<{k}>({bs})"


# ----------------------------------------------------------------------------- lowering
def lower(outputs: List[Tuple[str, sp.Expr]], names: Dict[sp.Symbol, str], loads: Dict[sp.Symbol, str],
          indent: str = "    ") -> Tuple[List[str], int]:
    """outputs: [(lhs, expr)] -> C statements of one CSE'd straight-line program, op count.
    `loads` maps input symbols to their memory expression (e.g. x[1]); each used input is
    loaded into a register once."""
    exprs = [sp.sympify(e) for _, e in outputs]
    if not exprs:
        return [], 0
    repl, red = sp.cse(exprs, symbols=sp.numbered_symbols("t_"), order="none")
    used = set()
    for _, e in repl:
        used |= e.free_symbols
    for e in red:
        used |= e.free_symbols
    local = dict(names)
    lines: List[str] = []
    for s in sorted((s for s in used if s in loads), key=lambda s: loads[s]):
        lines.append(f"{indent}const double {names[s]} = {loads[s]};")
    ops = 0
    for s, e in repl:
        local[s] = str(s)
        lines.append(f"{indent}const double {s} = {cstr(e, local)};")
        ops += int(sp.count_ops(e))
    for (lhs, _), e in zip(outputs, red):
        lines.append(f"{indent}{lhs} = {cstr(e, local)};")
        ops += int(sp.count_ops(e))
    return lines, ops


# ----------------------------------------------------------------------------- emission
_PREAMBLE = r"""// GENERATED by directtrajectoryoptimization.jl_b200/codegen.py -- do not edit.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include "dto_model_abi.h"

template <int K>
__device__ __forceinline__ double dto_powi(double x)
{
    if constexpr (K == 0) return 1.0;
    else if constexpr (K == 1) return x;
    else if constexpr (K % 2 == 0) { const double h = dto_powi<K / 2>(x); return h * h; }
    else return x * dto_powi<K - 1>(x);
}
__device__ __forceinline__ double dto_sign(double x) { return (x > 0.0) - (x < 0.0); }

// Branch-free sin/cos and reciprocal for the straight-line element programs (tune bf=1). Outside
// their domain they set `bad`; the generated function then re-evaluates itself with the library
// functions, so results stay defined for every double (NaN / Inf / huge arguments included).
// sincos: Cody-Waite reduction by pi/2 in three FMA steps (|x| < 2^31), fdlibm kernel polynomials
// (< 1 ulp on [-pi/4, pi/4]), quadrant by selects.
__device__ __forceinline__ void dto_sincos_bf(double x, double* sp, double* cp, unsigned& bad)
{
    bad |= (unsigned)((__double2hiint(x) & 0x7fffffff) >= 0x41e00000);  // |x| >= 2^31, Inf, NaN
    const int k = __double2int_rn(x * 0.63661977236758138);
    const double kd = (double)k;
    double r = fma(-kd, __longlong_as_double(0x3ff921fb54442d18LL), x);
    r = fma(-kd, __longlong_as_double(0x3c91a62633145c00LL), r);
    r = fma(-kd, __longlong_as_double(0x397b839a252049c0LL), r);
    const double z = r * r;
    const double v = z * r;
    double p = fma(z, 1.58969099521155010221e-10, -2.50507602534068634195e-08);
    p = fma(z, p, 2.75573137070700676789e-06);
    p = fma(z, p, -1.98412698298579493134e-04);
    p = fma(z, p, 8.33333333332248946124e-03);
    const double sr = fma(v, fma(z, p, -1.66666666666666324348e-01), r);
    double q = fma(z, -1.13596475577881948265e-11, 2.08757232129817482790e-09);
    q = fma(z, q, -2.75573143513906633035e-07);
    q = fma(z, q, 2.48015872894767294178e-05);
    q = fma(z, q, -1.38888888888741095749e-03);
    q = fma(z, q, 4.16666666666666019037e-02);
    const double hz = 0.5 * z;
    const double w1 = 1.0 - hz;
    const double cr = w1 + (((1.0 - w1) - hz) + z * (z * q));
    const double a = (k & 1) ? cr : sr;
    const double b = (k & 1) ? sr : cr;
    *sp = (k & 2) ? -a : a;
    *cp = ((k + 1) & 2) ? -b : b;
}
// reciprocal: hardware seed (2^-23) + two Newton steps (~1 ulp); flags denormal / huge / non-finite
__device__ __forceinline__ double dto_rcp_bf(double x, unsigned& bad)
{
    const unsigned e = ((unsigned)__double2hiint(x) >> 20) & 0x7ffu;
    bad |= (unsigned)((e - 3u) > 2040u);
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double t = fma(-x, r, 1.0);
    r = fma(r, t, r);
    t = fma(-x, r, 1.0);
    r = fma(r, t, r);
    t = fma(-x, r, 1.0);
    return fma(r, t, r);
}
"""


def _names_loads(args: Dict[str, Sequence[sp.Symbol]]):
    names, loads = {}, {}
    for cname, syms in args.items():
        for i, s in enumerate(syms):
            names[s] = f"{cname}_{i}"
            loads[s] = f"{cname}[{i}]"
    return names, loads


_SIG = {
    "dyn": "const double* __restrict__ y, const double* __restrict__ x, const double* __restrict__ u, const double* __restrict__ w",
    "cost": "const double* __restrict__ x, const double* __restrict__ u, const double* __restrict__ w",
    "stage": "const double* __restrict__ x, const double* __restrict__ u, const double* __restrict__ w",
}
_CALL = {"dyn": "y, x, u, w", "cost": "x, u, w", "stage": "x, u, w"}


def _emit_element(el: ElementSpec, k: int, out: List[str], stats: dict, cpool: Optional[dict] = None) -> None:
    if _deriv_mode() in ("hier", "dag"):
        try:
            _emit_element_dag(el, k, out, stats, cpool)
            return
        except NotImplementedError as e:  # a function the DAG has no rule for: lower sympy's derivatives instead
            stats[f"{el.role}{k}_dag_fallback"] = str(e)
    _emit_element_sympy(el, k, out, stats)


def _cached_cuts(el: ElementSpec, g, res, L, wrt, fused):
    """choose_cuts with an in-tree cache: the search depends on the element's expressions only, while one
    model is rebuilt for many tuning variants (the node ids are stable: the DAG is built deterministically)."""
    import json
    from .ir import choose_cuts
    max_evals = int(os.environ.get("DTO_CUT_EVALS", "6000"))
    h = hashlib.sha256(("cuts1|%d|" % max_evals).encode())
    with open(os.path.join(PKG_DIR, "ir.py"), "rb") as f:
        h.update(f.read())
    h.update(repr((el.role, [str(v) for v in el.vars], el.jac_rows, el.jac_cols, el.hess_rows, el.hess_cols)).encode())
    for e in el.evaluate:
        h.update(sp.srepr(e).encode())
    fname = f"cuts_{h.hexdigest()[:16]}.json"
    for p in (os.path.join(MODEL_DIR, fname), os.path.join(CACHE_DIR, fname)):
        if os.path.exists(p):
            with open(p) as f:
                d = json.load(f)
            return d["cuts"], d["stats"]
    cuts, st = choose_cuts(g, res, L, wrt, fused, max_evals=max_evals)
    path = os.path.join(CACHE_DIR, fname)
    os.makedirs(CACHE_DIR, exist_ok=True)
    with open(path + ".tmp", "w") as f:
        json.dump({"cuts": cuts, "stats": st}, f)
    os.replace(path + ".tmp", path)
    return cuts, st


def _emit_element_dag(el: ElementSpec, k: int, out: List[str], stats: dict, cpool: Optional[dict] = None) -> None:
    """Derivative synthesis on the residual DAG (ir.py): first/second-order sparse forward
    propagation, all outputs of one pass share one hash-consed graph."""
    from .ir import Graph, choose_cuts, count_ops, emit, hierarchical

    g = Graph()
    sym: Dict[sp.Symbol, int] = {}
    load: Dict[Tuple[str, int], str] = {}
    for cname, syms in el.args.items():
        for i, s_ in enumerate(syms):
            sym[s_] = g.inp(cname, i)
            load[(cname, i)] = f"{cname}[{i}]"
    memo: dict = {}
    res = [g.from_sympy(e, sym, memo) for e in el.evaluate]
    wrt = [sym[v] for v in el.vars]
    pre = f"{el.role}{k}"
    sig = _SIG[el.role]
    LAM = ", const double* __restrict__ lam"
    chunks: List[str] = []

    def fn(name, extra_sig, outputs, ret=None):
        c = count_ops(g, [n for _, n in outputs])
        stats[f"{pre}_{name}"] = sum(v for kk, v in c.items())
        stats[f"{pre}_{name}_mix"] = c
        chunks.append(f"__device__ __forceinline__ {'double' if ret else 'void'} {pre}_{name}({sig}{extra_sig})\n{{")
        tune = _tuning()
        use_bf = bool(tune["bf"]) and not ret and any(c.get(k_, 0) for k_ in ("sin", "cos", "rcp"))
        if use_bf:
            # fast path: one basic block; slow path (library sin/cos, IEEE division) only when an argument
            # left the domain of the branch-free functions
            chunks.append("    unsigned dto_bad = 0u;")
            chunks.extend(emit(g, outputs, load, cpool=cpool, order=tune["emit"], bf=True))
            chunks.append("    if (__builtin_expect(dto_bad != 0u, 0)) {")
            chunks.extend(emit(g, outputs, load, indent="        ", prefix="s", cpool=cpool, order=tune["emit"]))
            chunks.append("    }")
        else:
            chunks.extend(emit(g, outputs, load, cpool=cpool, order=tune["emit"]))
        if ret:
            chunks.append(f"    return {ret};")
        chunks.append("}\n")

    L = None
    if el.has_hess:
        L = res[0] if el.role == "cost" else g.sum(g.mul(sym[l], rn) for l, rn in zip(el.lam, res))
    hpat = [(min(r, c) - 1, max(r, c) - 1) for r, c in zip(el.hess_rows, el.hess_cols)] if el.has_hess else []
    jpat = [(r - 1, c - 1) for r, c in zip(el.jac_rows, el.jac_cols)]

    def fused(jac_, H_, h_):
        return [jac_[r].get(c, h_.ZERO) for r, c in jpat] + [H_.get(k_, h_.ZERO) for k_ in hpat]

    cuts: List[int] = []
    if _deriv_mode() == "hier" and el.has_hess and el.role != "cost":
        cuts, cst = _cached_cuts(el, g, res, L, wrt, fused)
        stats[f"{pre}_cuts"] = cst
    jacd, Hd = hierarchical(g, res, L, wrt, cuts, second=el.has_hess)
    # Jacobian / gradient entries in pattern order; every derivative must sit inside the pattern
    if el.user_jac:
        # Dynamics(f, jacobian, ...): the user's own Jacobian expressions are what the reference calls
        # (src/dynamics.jl:59-64), whether or not they are the derivative of f
        jac_nodes = [g.from_sympy(e, sym, memo) for e in el._jac]
    else:
        allowed = {}
        for r, c in jpat:
            allowed.setdefault(r, set()).add(c)
        for i in range(len(res)):
            extra = set(jacd[i]) - allowed.get(i, set())
            if extra:
                raise RuntimeError(f"{pre}: derivative of output {i} w.r.t. variables {sorted(extra)} is outside the structural "
                                   "Jacobian pattern")
        jac_nodes = [jacd[r].get(c, g.ZERO) for r, c in jpat]
    hess_nodes = []
    if el.has_hess:
        extra = set(Hd) - set(hpat)
        if extra:
            raise RuntimeError(f"{pre}: second derivatives {sorted(extra)} are outside the structural Hessian pattern")
        hess_nodes = [Hd.get(k_, g.ZERO) for k_ in hpat]

    if el.role == "cost":
        fn("val", "", [("const double v", res[0])], ret="v")
        fn("grad", ", double* __restrict__ G", [(f"G[{i}]", n) for i, n in enumerate(jac_nodes)])
        sg = g.inp("sigma", 0)
        load[("sigma", 0)] = "sigma"
        fn("hess", ", const double sigma, double* __restrict__ H", [(f"H[{i}]", g.mul(sg, n)) for i, n in enumerate(hess_nodes)])
    else:
        jo = [(f"J[{i}]", n) for i, n in enumerate(jac_nodes)]
        ho = [(f"H[{i}]", n) for i, n in enumerate(hess_nodes)]
        fn("res", ", double* __restrict__ R", [(f"R[{i}]", n) for i, n in enumerate(res)])
        fn("jac", ", double* __restrict__ J", jo)
        fn("hess", LAM + ", double* __restrict__ H", ho)
        fn("jac_hess", LAM + ", double* __restrict__ J, double* __restrict__ H", jo + ho)
    out.extend(chunks)


def _emit_element_sympy(el: ElementSpec, k: int, out: List[str], stats: dict) -> None:
    names, loads = _names_loads(el.args)
    pre = f"{el.role}{k}"
    sig = _SIG[el.role]
    LAM = ", const double* __restrict__ lam"

    def fn(name, extra_sig, outputs):
        body, ops = lower(outputs, names, loads)
        stats[f"{pre}_{name}"] = ops
        out.append(f"__device__ __forceinline__ void {pre}_{name}({sig}{extra_sig})\n{{")
        out.extend(body)
        out.append("}\n")

    if el.role == "cost":
        body, ops = lower([("const double v", el.evaluate[0])], names, loads)
        stats[f"{pre}_val"] = ops
        out.append(f"__device__ __forceinline__ double {pre}_val({sig})\n{{")
        out.extend(body)
        out.append("    return v;\n}\n")
        fn("grad", ", double* __restrict__ G", [(f"G[{i}]", e) for i, e in enumerate(el.jac)])
        sigma = sp.Symbol("sigma")
        names[sigma] = "sigma"
        fn("hess", ", const double sigma, double* __restrict__ H",
           [(f"H[{i}]", sigma * e) for i, e in enumerate(el.hess)] if el.has_hess else [])
        return
    fn("res", ", double* __restrict__ R", [(f"R[{i}]", e) for i, e in enumerate(el.evaluate)])
    jo = [(f"J[{i}]", e) for i, e in enumerate(el.jac)]
    ho = [(f"H[{i}]", e) for i, e in enumerate(el.hess)] if el.has_hess else []
    fn("jac", ", double* __restrict__ J", jo)
    fn("hess", LAM + ", double* __restrict__ H", ho)
    fn("jac_hess", LAM + ", double* __restrict__ J, double* __restrict__ H", jo + ho)


def _dispatch(role: str, n: int, name: str, ret: str, extra_sig: str, extra_call: str) -> List[str]:
    sig = _SIG[role]
    call = _CALL[role]
    lines = [f"    __device__ __forceinline__ static {ret} {role}_{name}(int k, {sig}{extra_sig})", "    {",
             "        switch (k) {"]
    for k in range(n):
        r = "return " if ret != "void" else ""
        tail = "" if ret != "void" else " break;"
        lines.append(f"        case {k}: {r}{role}{k}_{name}({call}{extra_call});{tail}")
    lines.append("        default: break;")
    lines.append("        }")
    if ret != "void":
        lines.append("        return 0.0;")
    lines.append("    }")
    return lines


def _int_array(name: str, vals: Sequence[int]) -> str:
    body = ", ".join(str(int(v)) for v in vals) if len(vals) else "0"
    return f"static const int32_t {name}[] = {{{body}}};"


def _general_templates(gen: GeneralSpec):
    """De-duplicate general-constraint outputs by index shift: an output expression whose z,
    w and lambda indices are renumbered relative to their minima is a TEMPLATE; outputs with
    identical templates share one device function (SURVEY: rolled codegen)."""
    zi = {s: i for i, s in enumerate(gen.args["z"])}
    wi = {s: i for i, s in enumerate(gen.args["w"])}
    li = {s: i for i, s in enumerate(gen.args.get("lam", []))}
    canon_z = [sp.Symbol(f"gz{i}") for i in range(len(zi) + 1)]
    canon_w = [sp.Symbol(f"gw{i}") for i in range(len(wi) + 1)]
    canon_l = [sp.Symbol(f"gl{i}") for i in range(len(li) + 1)]
    templates: List[List[sp.Expr]] = [[], [], []]
    lookup: List[Dict[sp.Expr, int]] = [{}, {}, {}]
    inst = [[], [], []]  # per class: (tmpl, zbase, wbase, lbase)
    for cls, exprs in enumerate([gen.evaluate, gen.jac, gen.hess if gen.has_hess else []]):
        for e in exprs:
            e = sp.sympify(e)
            fs = e.free_symbols
            zs = [zi[s] for s in fs if s in zi]
            ws = [wi[s] for s in fs if s in wi]
            ls = [li[s] for s in fs if s in li]
            zb, wb, lb = (min(zs) if zs else 0), (min(ws) if ws else 0), (min(ls) if ls else 0)
            sub = {}
            for s in fs:
                if s in zi:
                    sub[s] = canon_z[zi[s] - zb]
                elif s in wi:
                    sub[s] = canon_w[wi[s] - wb]
                elif s in li:
                    sub[s] = canon_l[li[s] - lb]
            ce = e.xreplace(sub)
            t = lookup[cls].get(ce)
            if t is None:
                t = len(templates[cls])
                templates[cls].append(ce)
                lookup[cls][ce] = t
            inst[cls].append((t, zb, wb, lb))
    names, loads = {}, {}
    for i, s in enumerate(canon_z):
        names[s], loads[s] = f"z_{i}", f"z[{i}]"
    for i, s in enumerate(canon_w):
        names[s], loads[s] = f"w_{i}", f"w[{i}]"
    for i, s in enumerate(canon_l):
        names[s], loads[s] = f"lam_{i}", f"lam[{i}]"
    return templates, inst, names, loads


def emit_model(spec: ModelSpec, source_hash: str) -> Tuple[str, dict]:
    out: List[str] = [_PREAMBLE, "/*CPOOL*/"]
    stats: dict = {}
    cpool: Dict[float, int] = {}
    for role, els in (("dyn", spec.dyn), ("cost", spec.cost), ("stage", spec.stage)):
        for k, el in enumerate(els):
            _emit_element(el, k, out, stats, cpool)
    vals = sorted(cpool, key=cpool.get)
    out[1] = ("// FP64 literals whose low word is non-zero live in the constant bank (direct c[][] operands)\n"
              "__constant__ double dto_k[] = {" + (", ".join(_lit(v) for v in vals) if vals else "0.0") + "};\n")
    stats["const_pool"] = len(vals)

    # general constraint templates
    gen = spec.general
    gen_inst = None
    if gen is not None:
        templates, gen_inst, gnames, gloads = _general_templates(gen)
        for cls in range(3):
            for t, e in enumerate(templates[cls]):
                body, ops = lower([("const double v", e)], gnames, gloads)
                stats[f"gen{cls}_{t}"] = ops
                out.append(f"__device__ __forceinline__ double gen{cls}_{t}(const double* __restrict__ z, "
                           "const double* __restrict__ w, const double* __restrict__ lam)\n{")
                out.extend(body)
                out.append("    return v;\n}\n")
        stats["gen_templates"] = [len(t) for t in templates]

        def _span(e, prefix):
            idx = [int(str(s_)[len(prefix):]) for s_ in e.free_symbols if str(s_).startswith(prefix)]
            return max(idx) + 1 if idx else 0
        stats["gen_hess_span"] = [(_span(e, "gz"), _span(e, "gw"), _span(e, "gl")) for e in templates[2]]

    halo = 0
    for el in spec.dyn:
        if el.has_hess and any(r > el.nx + el.nu for r in el.hess_rows):
            halo = 1

    # ---- struct DtoModel
    # the struct name is unique per model: several model libraries live in one process and C++
    # template instantiations / inline statics with equal mangled names may be shared across them
    m: List[str] = [f"struct DtoModel_{source_hash} {{", f"    static constexpr int HESS_HALO = {halo};"]
    els_all = list(spec.dyn) + list(spec.cost) + list(spec.stage)
    m.append(f"    static constexpr int MAX_NX = {max([e.nx for e in els_all] + [e.n_out for e in spec.dyn] + [0])};")
    m.append(f"    static constexpr int MAX_NU = {max([e.nu for e in els_all] + [0])};")
    m.append(f"    static constexpr int MAX_NY = {max([e.n_out for e in spec.dyn] + [0])};")
    m.append(f"    static constexpr int MAX_NW = {max([e.nw for e in els_all] + [0])};")
    m.append(f"    static constexpr int MAX_NC = {max([e.n_out for e in spec.stage] + [0])};")
    m.append(f"    static constexpr int N_KINDS_MAX = {max(len(spec.dyn), len(spec.cost), len(spec.stage))};")
    ops_fused = max([stats.get(f"dyn{k}_jac_hess", 0) for k in range(len(spec.dyn))] + [0])
    m.append(f"    static constexpr int OPS_FUSED = {ops_fused};  // FP64 ops of the heaviest fused dynamics element")
    dyn_w = any(set(e.args["w"]) & set().union(*[x.free_symbols for x in e.evaluate]) for e in spec.dyn if len(e.args["w"]))
    m.append(f"    static constexpr bool DYN_USES_W = {'true' if dyn_w else 'false'};")
    for role, els in (("dyn", spec.dyn), ("cost", spec.cost), ("stage", spec.stage)):
        m.append(f"    __device__ __forceinline__ static int {role}_nh(int k)")
        m.append("    {")
        m.append("        switch (k) {")
        for k, el in enumerate(els):
            m.append(f"        case {k}: return {el.nnz_hess};")
        m.append("        default: return 0;")
        m.append("        }")
        m.append("    }")
    LAM = ", const double* __restrict__ lam"
    # compiled Hessian gather classes
    ncls = len(spec.hg_classes)
    vmax = max([len(r) for r in spec.hg_classes] + [0])
    m.append(f"    static constexpr int HG_NCLASS = {ncls};")
    m.append(f"    static constexpr int HG_VMAX = {vmax};")
    m.append(f"    __device__ __forceinline__ static void hg_compute(int cls, const double* __restrict__ own, "
             f"const double* __restrict__ prev, double (&v)[{max(vmax, 1)}])")
    m.append("    {")
    m.append("        switch (cls) {")

    def _src(k):
        return f"own[{k}]" if k >= 0 else f"prev[{-k - 2}]"

    for c, rec in enumerate(spec.hg_classes):
        m.append(f"        case {c}:")
        for j, srcs in enumerate(rec):
            terms = [_src(k) for k in srcs if k != -1]
            m.append(f"            v[{j}] = {' + '.join(terms) if terms else '0.0'};")
        m.append("            break;")
    m.append("        default: break;")
    m.append("        }")
    m.append("    }")
    m.append(f"    __device__ __forceinline__ static void hg_store(int cls, const double (&v)[{max(vmax, 1)}], double* __restrict__ dst)")
    m.append("    {")
    m.append("        switch (cls) {")
    for c, rec in enumerate(spec.hg_classes):
        m.append(f"        case {c}:")
        for j in range(len(rec)):
            m.append(f"            dst[{j}] = v[{j}];")
        m.append("            break;")
    m.append("        default: break;")
    m.append("        }")
    m.append("    }")
    # register-resident gather (warp-specialised kernel): own terms come from the per-role arrays the
    # element functions just filled, previous-knot terms (always dynamics terms) from shared memory
    maxc = max([e.nnz_hess for e in spec.cost] + [1])
    maxd = max([e.nnz_hess for e in spec.dyn] + [1])
    maxs = max([e.nnz_hess for e in spec.stage] + [1])
    m.append(f"    static constexpr int MAXC = {maxc};")
    m.append(f"    static constexpr int MAXD = {maxd};")
    m.append(f"    static constexpr int MAXS = {maxs};")
    # previous-knot dynamics terms any class reads: fetched from the lane below by warp shuffles
    prev_used = sorted({-k - 2 - (spec.hg_meta[c][2] if c < len(spec.hg_meta) else 0)
                        for c, rec in enumerate(spec.hg_classes) for srcs in rec for k in srcs if k <= -2})
    m.append(f"    __device__ __forceinline__ static void hg_prev_exchange(const double (&td)[{maxd}], double (&pd)[{maxd}])")
    m.append("    {")
    for i in prev_used:
        m.append(f"        pd[{i}] = __shfl_up_sync(0xffffffffu, td[{i}], 1);")
    m.append("    }")
    m.append(f"    __device__ __forceinline__ static void hg_compute_r(int cls, const double (&tc)[{maxc}], const double (&td)[{maxd}], "
             f"const double (&ts)[{maxs}], const double (&prevd)[{maxd}], double (&v)[{max(vmax, 1)}])")
    m.append("    {")
    m.append("        switch (cls) {")
    for c, rec in enumerate(spec.hg_classes):
        nc_, nd_, ncp_ = spec.hg_meta[c] if c < len(spec.hg_meta) else (0, 0, 0)

        def _srcr(k, nc_=nc_, nd_=nd_, ncp_=ncp_):
            if k >= 0:
                if k < nc_:
                    return f"tc[{k}]"
                if k < nc_ + nd_:
                    return f"td[{k - nc_}]"
                return f"ts[{k - nc_ - nd_}]"
            return f"prevd[{-k - 2 - ncp_}]"

        m.append(f"        case {c}:")
        for j, srcs in enumerate(rec):
            terms = [_srcr(k) for k in srcs if k != -1]
            m.append(f"            v[{j}] = {' + '.join(terms) if terms else '0.0'};")
        m.append("            break;")
    m.append("        default: break;")
    m.append("        }")
    m.append("    }")
    m += _dispatch("cost", len(spec.cost), "val", "double", "", "")
    m += _dispatch("cost", len(spec.cost), "grad", "void", ", double* __restrict__ G", ", G")
    m += _dispatch("cost", len(spec.cost), "hess", "void", ", const double sigma, double* __restrict__ H", ", sigma, H")
    for role, n in (("dyn", len(spec.dyn)), ("stage", len(spec.stage))):
        m += _dispatch(role, n, "res", "void", ", double* __restrict__ R", ", R")
        m += _dispatch(role, n, "jac", "void", ", double* __restrict__ J", ", J")
        m += _dispatch(role, n, "hess", "void", LAM + ", double* __restrict__ H", ", lam, H")
        m += _dispatch(role, n, "jac_hess", "void", LAM + ", double* __restrict__ J, double* __restrict__ H",
                       ", lam, J, H")
    m.append("    __device__ __forceinline__ static double gen_eval(int cls, int tmpl, const double* __restrict__ z, "
             "const double* __restrict__ w, const double* __restrict__ lam)")
    m.append("    {")
    if gen is not None:
        for cls in range(3):
            m.append(f"        if (cls == {cls}) {{")
            m.append("            switch (tmpl) {")
            for t in range(stats["gen_templates"][cls]):
                m.append(f"            case {t}: return gen{cls}_{t}(z, w, lam);")
            m.append("            default: break;")
            m.append("            }")
            m.append("        }")
    m.append("        return 0.0;")
    m.append("    }")
    m.append("};")
    m.append(f"using DtoModel = DtoModel_{source_hash};\n")
    out.extend(m)
    out.append('#include "dto_kernels.cuh"\n')

    # ---- descriptors
    d: List[str] = []

    def elem_desc(role: str, k: int, el: ElementSpec) -> str:
        p = f"{role}{k}"
        d.append(_int_array(f"{p}_jr", el.jac_rows))
        d.append(_int_array(f"{p}_jc", el.jac_cols))
        d.append(_int_array(f"{p}_hr", el.hess_rows if el.has_hess else []))
        d.append(_int_array(f"{p}_hc", el.hess_cols if el.has_hess else []))
        d.append(_int_array(f"{p}_iq", el.ineq))
        nj = el.nnz_jac
        nh = el.nnz_hess
        return (f"{{{el.n_out}, {el.nx}, {el.nu}, {el.nw}, {nj}, {p}_jr, {p}_jc, {int(el.has_hess)}, {nh}, "
                f"{p}_hr, {p}_hc, {len(el.ineq)}, {p}_iq}}")

    for role, els in (("dyn", spec.dyn), ("cost", spec.cost), ("stage", spec.stage)):
        rows = [elem_desc(role, k, el) for k, el in enumerate(els)]
        if not rows:
            rows = ["{0, 0, 0, 0, 0, nullptr, nullptr, 0, 0, nullptr, nullptr, 0, nullptr}"]
        d.append(f"static const dto_element_desc {role}_descs[] = {{\n    " + ",\n    ".join(rows) + "\n};")
    if gen is not None:
        d.append(_int_array("gen_jr", gen.jac_rows))
        d.append(_int_array("gen_jc", gen.jac_cols))
        d.append(_int_array("gen_hr", gen.hess_rows if gen.has_hess else []))
        d.append(_int_array("gen_hc", gen.hess_cols if gen.has_hess else []))
        d.append(_int_array("gen_iq", gen.ineq))
        for cls in range(3):
            for j, nm in enumerate(("tmpl", "zbase", "wbase", "lbase")):
                d.append(_int_array(f"gen_{nm}{cls}", [t[j] for t in gen_inst[cls]]))
        nh = len(gen.hess) if gen.has_hess else 0
        d.append(_int_array("gen_hspan", [v for t3 in stats.get("gen_hess_span", []) for v in t3]))
        d.append("static const dto_general_desc gen_desc = {"
                 f"{gen.num_variables}, {gen.num_parameter}, {len(gen.evaluate)}, {len(gen.jac)}, gen_jr, gen_jc, "
                 f"{int(gen.has_hess)}, {nh}, gen_hr, gen_hc, {len(gen.ineq)}, gen_iq, "
                 "{gen_tmpl0, gen_tmpl1, gen_tmpl2}, {gen_zbase0, gen_zbase1, gen_zbase2}, "
                 "{gen_wbase0, gen_wbase1, gen_wbase2}, {gen_lbase0, gen_lbase1, gen_lbase2}, "
                 f"{len(stats.get('gen_hess_span', []))}, gen_hspan}};")
    hg_ns = [len(r) for r in spec.hg_classes]
    hg_of, acc = [], 0
    for n_ in hg_ns:
        hg_of.append(acc)
        acc += n_
    d.append(_int_array("hg_nslots", hg_ns))
    d.append(_int_array("hg_ofs", hg_of))
    d.append(_int_array("hg_src", [k for r in spec.hg_classes for srcs in r for k in srcs]))
    d.append(_int_array("hg_meta", [v for c in range(len(spec.hg_classes)) for v in (spec.hg_meta[c] if c < len(spec.hg_meta) else (-1, -1, -1))]))
    fused = 0
    for k in range(len(spec.dyn)):
        fused = max(fused, stats.get(f"dyn{k}_jac_hess", 0))
    stats["ops_fused_per_knot"] = fused
    d.append(f"""
static int model_launch(int kernel_id, const dto_launch_args* a, void* stream) {{ return dto::launch<DtoModel>(kernel_id, a, stream); }}
static int64_t model_smem(int kernel_id, const dto_launch_args* a) {{ return dto::smem_bytes<DtoModel>(kernel_id, a); }}
static const dto_model_vtable model_vtable = {{
    DTO_MODEL_ABI_VERSION, "{spec.name}", "{source_hash}",
    {len(spec.dyn)}, {len(spec.cost)}, {len(spec.stage)},
    dyn_descs, cost_descs, stage_descs, {"&gen_desc" if gen is not None else "nullptr"},
    {halo}, DTO_WARPS, {fused},
    {len(spec.hg_classes)}, hg_nslots, hg_ofs, hg_src, hg_meta,
    model_launch, model_smem
}};
extern "C" __attribute__((visibility("default"))) const dto_model_vtable* dto_model_entry(void) {{ return &model_vtable; }}
""")
    out.extend(d)
    return "\n".join(out), stats


# ----------------------------------------------------------------------------- build
def spec_hash(spec: ModelSpec) -> str:
    h = hashlib.sha256()
    h.update(CODEGEN_VERSION.encode())
    h.update(repr(sorted(_tuning().items())).encode())
    h.update(_deriv_mode().encode())
    with open(os.path.join(PKG_DIR, "ir.py"), "rb") as f:
        h.update(f.read())
    for fname in ("dto_kernels.cuh", "dto_kernel_ws.cuh", "dto_model_abi.h"):
        with open(os.path.join(CSRC_DIR, fname), "rb") as f:
            h.update(f.read())

    def feed_el(el):
        h.update(repr((el.role, el.n_out, el.nx, el.nu, el.nw, el.jac_rows, el.jac_cols, el.has_hess, el.hess_rows,
                       el.hess_cols, el.ineq)).encode())
        for e in list(el.evaluate):
            h.update(sp.srepr(e).encode())
        if el.user_jac:  # Dynamics(f, jacobian, ...): two user Jacobians for one f are two different libraries
            h.update(b"userjac")
            for e in el._jac:
                h.update(sp.srepr(sp.sympify(e)).encode())

    for els in (spec.dyn, spec.cost, spec.stage):
        h.update(b"|")
        for el in els:
            feed_el(el)
    h.update(repr(spec.hg_classes).encode())
    h.update(repr(spec.hg_meta).encode())
    if spec.general is not None:
        g = spec.general
        h.update(repr((g.num_variables, g.num_parameter, g.jac_rows, g.jac_cols, g.has_hess, g.hess_rows, g.hess_cols,
                       g.ineq)).encode())
        for e in list(g.evaluate) + list(g.jac) + (list(g.hess) if g.has_hess else []):
            h.update(sp.srepr(e).encode())
    return h.hexdigest()[:16]


def build_model(spec: ModelSpec, verbose: bool = False, force: bool = False) -> str:
    """Generate + compile (or reuse) the model library; returns the path of the .so."""
    hsh = spec_hash(spec)
    prebuilt = os.path.join(MODEL_DIR, f"{spec.name}_{hsh}.so")
    if os.path.exists(prebuilt) and not force:
        return prebuilt
    os.makedirs(CACHE_DIR, exist_ok=True)
    base = os.path.join(CACHE_DIR, f"{spec.name}_{hsh}")
    so, cu = base + ".so", base + ".cu"
    if os.path.exists(so) and not force:
        return so
    # one builder at a time per library: the ranks of a torchrun launch that all miss the same model must not
    # race on the .cu / .so.tmp files (seen on an 8-GPU box); the others wait and then find the finished .so
    import fcntl
    with open(base + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if os.path.exists(so) and not force:
                return so
            return _build_model_locked(spec, hsh, base, so, cu, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_model_locked(spec: ModelSpec, hsh: str, base: str, so: str, cu: str, verbose: bool) -> str:
    t0 = time.time()
    src, stats = emit_model(spec, hsh)
    with open(cu, "w") as f:
        f.write(src)
    if not os.path.exists(NVCC):
        raise RuntimeError(f"nvcc not found at {NVCC}: the CUDA model library cannot be built (no CPU fallback exists)")
    tune = _tuning()
    # ws_helpers = 8, one helper warp per compute warp (16 warps per CTA, 128 registers per thread at launch; setmaxnreg
    # then gives helpers 40 and compute warps 216). Light models always needed it (a helper's ~300 latency-bound
    # integer instructions per tile would bound the kernel); since the hierarchical derivatives cut the
    # FP64 work per knot the heavy models do too: with one helper per TWO compute warps the cartpole compute
    # warps waited 22 % of their time for inputs (profiles/ncu_ws_r02_a.txt), 37.0 -> 33.5 us with 8 helpers.
    cmd = [NVCC, *NVCC_ARCH, f"-DDTO_PERSIST={tune['persist']}", f"-DDTO_WS={tune['ws']}", f"-DDTO_WS_PLAN={tune['ws_plan']}",
           f"-DDTO_WS_HELPERS={tune['ws_helpers']}", f"-DDTO_WS_ALL_MODES={tune['ws_all']}", "-O3", "-std=c++17", "-lineinfo",
           "--shared", "-Xcompiler", "-fPIC,-fvisibility=hidden", "-Xptxas", "-v", "-I", CSRC_DIR, "-o", so + ".tmp", cu]
    t1 = time.time()
    r = subprocess.run(cmd, capture_output=True, text=True)
    with open(base + ".log", "w") as f:
        f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr + f"\ncodegen {t1 - t0:.1f}s nvcc {time.time() - t1:.1f}s\n"
                + repr(stats) + "\n")
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for {cu}:\n{r.stderr[-4000:]}")
    os.replace(so + ".tmp", so)
    if verbose:
        print(f"[dto codegen] built {so} (codegen {t1 - t0:.1f}s, nvcc {time.time() - t1:.1f}s) ops={stats.get('ops_fused_per_knot')}")
    return so

"""ORACLE (test infrastructure only): plain-C twin of the CPU restatement.

Emits, for one assembled oracle Solver, a self-contained C file that restates the
reference's callback structure with the reference's loop shapes:

    trajectory!/duals! unpack   /root/reference/src/data.jl:258-278
    per-knot closure call + cache -> slice copy (+ fill!)
                                /root/reference/src/dynamics.jl:103-127, src/costs.jl:49-73,
                                src/constraints.jl:80-104, src/general_constraint.jl:73-91
    callback order + zero fill  /root/reference/src/moi.jl:1-120

Element functions come from the ORACLE's own symbolic expressions (oracle/elements.py),
printed here with full precision, in two variants:
    cse=False  one independent expression per output -- what Symbolics 0.1.x
               build_function emits (no CSE); this is the "reference-like" CPU baseline;
    cse=True   sympy.cse over each closure's outputs (a faster stand-in, also used as the
               large-batch checker because it compiles and runs quickly).
A batch is an OpenMP loop over problems with per-thread element caches (one Solver is not
thread-safe in the reference, SURVEY 2.1). Built with `gcc -O2 -fopenmp` into oracle/_build/.
Used only by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
from typing import Dict, List, Sequence

import numpy as np
import sympy as sp

BUILD_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_build")

_CF = {"sin": "sin", "cos": "cos", "tan": "tan", "exp": "exp", "log": "log", "atan": "atan", "asin": "asin",
       "acos": "acos", "sinh": "sinh", "cosh": "cosh", "tanh": "tanh", "Abs": "fabs", "atan2": "atan2"}


def _c(e: sp.Expr, names: Dict[sp.Symbol, str]) -> str:
    if e.is_Symbol:
        return names[e]
    if e.is_Number or e.is_NumberSymbol:
        v = float(e)
        r = repr(v)
        if "e" not in r and "." not in r and "inf" not in r and "nan" not in r:
            r += ".0"
        return r if v >= 0 else f"({r})"
    if e.is_Add:
        return "(" + " + ".join(_c(a, names) for a in e.args) + ")"
    if e.is_Mul:
        return "(" + "*".join(_c(a, names) for a in e.args) + ")"
    if e.is_Pow:
        b, p = e.args
        if p.is_Integer or (p.is_Float and float(p) == int(float(p))):
            k = int(p)
            bs = _c(b, names)
            if k == -1:
                return f"(1.0/{bs})"
            return f"powi({bs}, {k})"
        return f"pow({_c(b, names)}, {_c(p, names)})"
    if isinstance(e, sp.Piecewise):  # ifelse(c, a, b)
        out = "0.0"
        for val, cond in reversed(e.args):
            out = _c(val, names) if cond is sp.true else f"(({_c(cond, names)}) ? {_c(val, names)} : {out})"
        return out
    if e.is_Relational:
        return f"({_c(e.lhs, names)} {e.rel_op} {_c(e.rhs, names)})"
    if e.is_Function:
        return _CF[e.func.__name__] + "(" + ", ".join(_c(a, names) for a in e.args) + ")"
    raise NotImplementedError(type(e))


def _fn(name: str, sig: str, exprs: Sequence, names: Dict[sp.Symbol, str], cse: bool) -> str:
    lines = [f"static void {name}({sig})", "{"]
    exprs = [sp.sympify(e) for e in exprs]
    if cse and exprs:
        repl, red = sp.cse(exprs, symbols=sp.numbered_symbols("t_"), order="none")
        local = dict(names)
        for s, e in repl:
            local[s] = str(s)
            lines.append(f"    const double {s} = {_c(e, local)};")
        for k, e in enumerate(red):
            lines.append(f"    out[{k}] = {_c(e, local)};")
    else:
        for k, e in enumerate(exprs):
            lines.append(f"    out[{k}] = {_c(e, names)};")
    lines.append("}")
    return "\n".join(lines)


def _names(**arrays) -> Dict[sp.Symbol, str]:
    n = {}
    for cname, syms in arrays.items():
        for i, s in enumerate(syms):
            n[s] = f"{cname}[{i}]"
    return n


def _arr(name: str, vals, ctype="int") -> str:
    vals = list(vals)
    body = ", ".join(str(int(v)) for v in vals) if vals else "0"
    return f"static const {ctype} {name}[] = {{{body}}};"


_DRIVER = r"""
/* ---- reference loop structure, one problem ---- */
typedef struct { double* X; double* cache; double* dual; } scratch_t;

static void unpack(const double* z, double* X)
{   /* trajectory!: states[t] .= z[idx]; actions[t] .= z[idx] (src/data.jl:258-267) */
    for (int t = 0; t < T; ++t) { for (int i = 0; i < NX[t]; ++i) X[XOFS[t] + i] = z[STATE_IDX[t] - 1 + i]; }
    for (int t = 0; t < T - 1; ++t) { for (int i = 0; i < NU[t]; ++i) X[UOFS[t] + i] = z[ACTION_IDX[t] - 1 + i]; }
}

static double eval_objective_1(const double* z, const double* w, scratch_t* s)
{   /* src/moi.jl:1-13 -> src/costs.jl:49-56 */
    unpack(z, s->X);
    double Jv = 0.0;
    for (int t = 0; t < T; ++t) {
        cost_eval(COST_KIND[t], s->cache, s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t]);
        Jv += s->cache[0];
    }
    return Jv;
}

static void eval_gradient_1(double* g, const double* z, const double* w, scratch_t* s)
{   /* src/moi.jl:15-30 -> src/costs.jl:58-64 */
    for (int i = 0; i < NZ; ++i) g[i] = 0.0;
    unpack(z, s->X);
    for (int t = 0; t < T; ++t) {
        cost_grad(COST_KIND[t], s->cache, s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t]);
        for (int k = 0; k < NX[t] + NU[t]; ++k) g[STATE_IDX[t] - 1 + k] += s->cache[k];
    }
}

static void eval_constraint_1(double* c, const double* z, const double* w, scratch_t* s)
{   /* src/moi.jl:32-50 */
    for (int i = 0; i < NC; ++i) c[i] = 0.0;
    unpack(z, s->X);
    for (int t = 0; t < T - 1; ++t) {
        dyn_eval(DYN_KIND[t], s->cache, s->X + XOFS[t + 1], s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t]);
        for (int k = 0; k < DYN_NC[t]; ++k) { c[DYN_CIDX[t] - 1 + k] = s->cache[k]; s->cache[k] = 0.0; }
    }
    for (int t = 0; t < T; ++t) {
        if (STAGE_KIND[t] < 0) continue;
        stage_eval(STAGE_KIND[t], s->cache, s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t]);
        for (int k = 0; k < STAGE_NC[t]; ++k) { c[STAGE_CIDX[t] - 1 + k] = s->cache[k]; s->cache[k] = 0.0; }
    }
    if (GEN_NC != 0) {
        general_eval(s->cache, z, w);
        for (int k = 0; k < GEN_NC; ++k) { c[GEN_CIDX - 1 + k] = s->cache[k]; s->cache[k] = 0.0; }
    }
}

static void eval_jacobian_1(double* J, const double* z, const double* w, scratch_t* s)
{   /* src/moi.jl:52-70 */
    for (int i = 0; i < NJ; ++i) J[i] = 0.0;
    unpack(z, s->X);
    for (int t = 0; t < T - 1; ++t) {
        dyn_jac(DYN_KIND[t], s->cache, s->X + XOFS[t + 1], s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t]);
        for (int k = 0; k < DYN_NJ[t]; ++k) { J[DYN_JIDX[t] - 1 + k] = s->cache[k]; s->cache[k] = 0.0; }
    }
    for (int t = 0; t < T; ++t) {
        if (STAGE_KIND[t] < 0) continue;
        stage_jac(STAGE_KIND[t], s->cache, s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t]);
        for (int k = 0; k < STAGE_NJ[t]; ++k) { J[STAGE_JIDX[t] - 1 + k] = s->cache[k]; s->cache[k] = 0.0; }
    }
    if (GEN_NC != 0) {
        general_jac(s->cache, z, w);
        for (int k = 0; k < GEN_NJ; ++k) { J[GEN_JIDX - 1 + k] = s->cache[k]; s->cache[k] = 0.0; }
    }
}

static void eval_hessian_1(double* H, const double* z, double sigma, const double* lam, const double* w, scratch_t* s)
{   /* src/moi.jl:72-120: zero; duals!; cost (scaled in the cache); dynamics; stage; general */
    for (int i = 0; i < NH; ++i) H[i] = 0.0;
    unpack(z, s->X);
    for (int i = 0; i < NC; ++i) s->dual[i] = lam[i];
    for (int t = 0; t < T; ++t) {
        const int n = COST_NH[t];
        cost_hess(COST_KIND[t], s->cache, s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t]);
        for (int k = 0; k < n; ++k) s->cache[k] *= sigma;
        for (int k = 0; k < n; ++k) H[HIDX[COST_HPTR[t] + k] - 1] += s->cache[k];
    }
    for (int t = 0; t < T - 1; ++t) {
        const int n = DYN_NH[t];
        if (n == 0) continue;
        dyn_hess(DYN_KIND[t], s->cache, s->X + XOFS[t + 1], s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t], s->dual + DYN_CIDX[t] - 1);
        for (int k = 0; k < n; ++k) { H[HIDX[DYN_HPTR[t] + k] - 1] += s->cache[k]; s->cache[k] = 0.0; }
    }
    for (int t = 0; t < T; ++t) {
        const int n = STAGE_NH[t];
        if (n == 0) continue;
        stage_hess(STAGE_KIND[t], s->cache, s->X + XOFS[t], s->X + UOFS[t], w + WOFS[t], s->dual + STAGE_CIDX[t] - 1);
        for (int k = 0; k < n; ++k) { H[HIDX[STAGE_HPTR[t] + k] - 1] += s->cache[k]; s->cache[k] = 0.0; }
    }
    if (GEN_NH != 0) {
        general_hess(s->cache, z, w, s->dual + GEN_CIDX - 1);
        for (int k = 0; k < GEN_NH; ++k) { H[HIDX[GEN_HPTR + k] - 1] += s->cache[k]; s->cache[k] = 0.0; }
    }
}

/* ---- batch = OpenMP loop over problems ---- */
#include <stdlib.h>
#ifdef _OPENMP
#include <omp.h>
#endif

int oracle_dims(int* out) { out[0] = T; out[1] = NZ; out[2] = NC; out[3] = NJ; out[4] = NH; out[5] = NW; return 0; }
int oracle_max_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* what: bit 0 objective, 1 gradient, 2 constraint, 3 jacobian, 4 hessian */
int oracle_eval_batch(int what, long B, int nthreads, const double* z, const double* lam, const double* sigma, const double* w,
                      double* f, double* g, double* c, double* J, double* H)
{
#ifdef _OPENMP
    if (nthreads > 0) omp_set_num_threads(nthreads);
#endif
#pragma omp parallel
    {
        scratch_t s;
        s.X = (double*)malloc(sizeof(double) * (NZ + 1));
        s.cache = (double*)malloc(sizeof(double) * (CACHE_MAX + 1));
        s.dual = (double*)malloc(sizeof(double) * (NC + 1));
        for (int i = 0; i < CACHE_MAX + 1; ++i) s.cache[i] = 0.0;
#pragma omp for schedule(static)
        for (long b = 0; b < B; ++b) {
            const double* zb = z + b * NZ;
            const double* wb = w + b * NW;
            if (what & 1) f[b] = eval_objective_1(zb, wb, &s);
            if (what & 2) eval_gradient_1(g + b * NZ, zb, wb, &s);
            if (what & 4) eval_constraint_1(c + b * NC, zb, wb, &s);
            if (what & 8) eval_jacobian_1(J + b * NJ, zb, wb, &s);
            if (what & 16) eval_hessian_1(H + b * NH, zb, sigma[b], lam + b * NC, wb, &s);
        }
        free(s.X); free(s.cache); free(s.dual);
    }
    return 0;
}
"""


def emit_c(solver, shared_parameters: bool, cse: bool) -> str:
    """C source for one assembled oracle Solver (oracle/nlp.py)."""
    nlp = solver.nlp
    t = nlp.trajopt
    idx = nlp.indices
    T = len(t.objective)
    out: List[str] = ["/* GENERATED by oracle/cgen.py (test infrastructure; CPU restatement of the reference) */",
                      "#include <math.h>",
                      "static inline double powi(double x, int k) { if (k < 0) return 1.0 / powi(x, -k); double r = 1.0; "
                      "while (k) { if (k & 1) r *= x; x *= x; k >>= 1; } return r; }"]

    def uniq(elems):
        u, ids, kinds = [], {}, []
        for e in elems:
            if getattr(e, "sym", None) is None and not hasattr(e, "num_gradient"):
                kinds.append(-1)
                continue
            if id(e) not in ids:
                ids[id(e)] = len(u)
                u.append(e)
            kinds.append(ids[id(e)])
        return u, kinds

    dyn_u, dyn_k = uniq(t.dynamics)
    cost_u, cost_k = uniq(t.objective)
    stage_u, stage_k = uniq(t.constraints)
    cache_max = 1

    for k, e in enumerate(cost_u):
        s = e.sym
        nm = _names(x=s["x"], u=s["u"], w=s["w"])
        sig = "double* out, const double* x, const double* u, const double* w"
        out.append(_fn(f"cost{k}_eval", sig, s["evaluate"], nm, cse))
        out.append(_fn(f"cost{k}_grad", sig, s["gradient"], nm, cse))
        out.append(_fn(f"cost{k}_hess", sig, s.get("hessian", []), nm, cse))
        cache_max = max(cache_max, e.num_gradient, e.num_hessian)
    for k, e in enumerate(dyn_u):
        s = e.sym
        if s is None:
            raise NotImplementedError("user-closure Dynamics has no expressions to print")
        nm = _names(y=s["y"], x=s["x"], u=s["u"], w=s["w"], lam=s.get("lam", []))
        sig = "double* out, const double* y, const double* x, const double* u, const double* w"
        out.append(_fn(f"dyn{k}_eval", sig, s["evaluate"], nm, cse))
        out.append(_fn(f"dyn{k}_jac", sig, s["jacobian"], nm, cse))
        out.append(_fn(f"dyn{k}_hess", sig + ", const double* lam", s.get("hessian", []), nm, cse))
        cache_max = max(cache_max, e.num_next_state, e.num_jacobian, e.num_hessian)
    for k, e in enumerate(stage_u):
        s = e.sym
        nm = _names(x=s["x"], u=s["u"], w=s["w"], lam=s.get("lam", []))
        sig = "double* out, const double* x, const double* u, const double* w"
        out.append(_fn(f"stage{k}_eval", sig, s["evaluate"], nm, cse))
        out.append(_fn(f"stage{k}_jac", sig, s["jacobian"], nm, cse))
        out.append(_fn(f"stage{k}_hess", sig + ", const double* lam", s.get("hessian", []), nm, cse))
        cache_max = max(cache_max, e.num_constraint, e.num_jacobian, e.num_hessian)
    gen = nlp.general_constraint
    if gen.num_constraint:
        s = gen.sym
        nm = _names(z=s["z"], w=s["w"], lam=s.get("lam", []))
        sig = "double* out, const double* z, const double* w"
        out.append(_fn("general_eval", sig, s["evaluate"], nm, cse))
        out.append(_fn("general_jac", sig, s["jacobian"], nm, cse))
        out.append(_fn("general_hess", sig + ", const double* lam", s.get("hessian", []), nm, cse))
        cache_max = max(cache_max, gen.num_constraint, gen.num_jacobian, gen.num_hessian)
    else:
        out.append("static void general_eval(double* out, const double* z, const double* w) {}")
        out.append("static void general_jac(double* out, const double* z, const double* w) {}")
        out.append("static void general_hess(double* out, const double* z, const double* w, const double* lam) {}")

    def dispatch(role, n, name, sig, call):
        lines = [f"static void {role}_{name}(int k, {sig})", "{", "    switch (k) {"]
        for k in range(n):
            lines.append(f"    case {k}: {role}{k}_{name}({call}); break;")
        lines += ["    default: break;", "    }", "}"]
        return "\n".join(lines)

    csig = "double* out, const double* x, const double* u, const double* w"
    dsig = "double* out, const double* y, const double* x, const double* u, const double* w"
    for nme in ("eval", "grad", "hess"):
        out.append(dispatch("cost", len(cost_u), nme, csig, "out, x, u, w"))
    out.append(dispatch("dyn", len(dyn_u), "eval", dsig, "out, y, x, u, w"))
    out.append(dispatch("dyn", len(dyn_u), "jac", dsig, "out, y, x, u, w"))
    out.append(dispatch("dyn", len(dyn_u), "hess", dsig + ", const double* lam", "out, y, x, u, w, lam"))
    out.append(dispatch("stage", len(stage_u), "eval", csig, "out, x, u, w"))
    out.append(dispatch("stage", len(stage_u), "jac", csig, "out, x, u, w"))
    out.append(dispatch("stage", len(stage_u), "hess", csig + ", const double* lam", "out, x, u, w, lam"))

    # ---- tables (1-based index values exactly as the oracle / reference hold them)
    sd, ad = t.state_dimensions, t.action_dimensions
    xofs, uofs, acc = [], [], 0
    for tt in range(T):
        xofs.append(acc)
        acc += sd[tt]
        uofs.append(acc)
        acc += ad[tt]
    pdims = [len(p) for p in t.parameters[:T]]
    if shared_parameters:
        wofs, nw = [0] * T, (max(pdims) if pdims else 0)
    else:
        wofs, nw, a2 = [], 0, 0
        for tt in range(T):
            wofs.append(a2)
            a2 += pdims[tt]
        nw = a2
    hidx: List[int] = []
    cost_hptr, dyn_hptr, stage_hptr = [], [], []
    for tt in range(T):
        cost_hptr.append(len(hidx))
        hidx.extend(idx.objective_hessians[tt])
    for tt in range(T - 1):
        dyn_hptr.append(len(hidx))
        hidx.extend(idx.dynamics_hessians[tt])
    for tt in range(T):
        stage_hptr.append(len(hidx))
        hidx.extend(idx.stage_hessians[tt])
    gen_hptr = len(hidx)
    hidx.extend(idx.general_hessian)
    NH = len(nlp.hessian_lagrangian_sparsity)
    first = lambda lst, default=1: (lst[0] if len(lst) else default)  # noqa: E731
    out += [
        f"enum {{ T = {T}, NZ = {nlp.num_variables}, NC = {nlp.num_constraint}, NJ = {nlp.num_jacobian}, NH = {NH}, "
        f"NW = {nw}, CACHE_MAX = {cache_max}, GEN_NC = {gen.num_constraint}, GEN_NJ = {gen.num_jacobian}, "
        f"GEN_NH = {gen.num_hessian}, GEN_CIDX = {first(idx.general_constraint)}, GEN_JIDX = {first(idx.general_jacobian)}, "
        f"GEN_HPTR = {gen_hptr} }};",
        _arr("NX", sd), _arr("NU", ad), _arr("XOFS", xofs), _arr("UOFS", uofs), _arr("WOFS", wofs),
        _arr("STATE_IDX", [first(v) for v in idx.states]),
        _arr("ACTION_IDX", [first(v) for v in idx.actions] + [1]),
        _arr("COST_KIND", cost_k), _arr("DYN_KIND", dyn_k + [-1]), _arr("STAGE_KIND", stage_k),
        _arr("DYN_NC", [d.num_next_state for d in t.dynamics]),
        _arr("DYN_CIDX", [first(v) for v in idx.dynamics_constraints]),
        _arr("DYN_NJ", [d.num_jacobian for d in t.dynamics]),
        _arr("DYN_JIDX", [first(v) for v in idx.dynamics_jacobians]),
        _arr("STAGE_NC", [c.num_constraint for c in t.constraints]),
        _arr("STAGE_CIDX", [first(v) for v in idx.stage_constraints]),
        _arr("STAGE_NJ", [c.num_jacobian for c in t.constraints]),
        _arr("STAGE_JIDX", [first(v) for v in idx.stage_jacobians]),
        _arr("COST_NH", [c.num_hessian for c in t.objective]), _arr("COST_HPTR", cost_hptr),
        _arr("DYN_NH", [d.num_hessian for d in t.dynamics]), _arr("DYN_HPTR", dyn_hptr),
        _arr("STAGE_NH", [c.num_hessian for c in t.constraints]), _arr("STAGE_HPTR", stage_hptr),
        _arr("HIDX", hidx),
    ]
    out.append(_DRIVER)
    return "\n".join(out)


class COracle:
    """ctypes wrapper of a built C twin."""

    def __init__(self, path: str):
        self.path = path
        self.lib = C.CDLL(path)
        self.lib.oracle_eval_batch.restype = C.c_int
        self.lib.oracle_eval_batch.argtypes = [C.c_int, C.c_long, C.c_int] + [C.c_void_p] * 9
        self.lib.oracle_max_threads.restype = C.c_int
        d = (C.c_int * 6)()
        self.lib.oracle_dims(d)
        self.T, self.NZ, self.NC, self.NJ, self.NH, self.NW = list(d)

    def max_threads(self) -> int:
        return int(self.lib.oracle_max_threads())

    def eval(self, what: int, z, lam, sigma, w, nthreads: int = 0):
        B = z.shape[0]
        z = np.ascontiguousarray(z, dtype=np.float64)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        sigma = np.ascontiguousarray(sigma, dtype=np.float64)
        w = np.ascontiguousarray(w if w.size else np.zeros((B, 1)), dtype=np.float64)
        out = dict(f=np.zeros(B), g=np.zeros((B, self.NZ)) if what & 2 else np.zeros(1),
                   c=np.zeros((B, self.NC)) if what & 4 else np.zeros(1),
                   J=np.zeros((B, self.NJ)) if what & 8 else np.zeros(1),
                   H=np.zeros((B, self.NH)) if what & 16 else np.zeros(1))
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        self.lib.oracle_eval_batch(what, B, nthreads, p(z), p(lam), p(sigma), p(w), p(out["f"]), p(out["g"]), p(out["c"]),
                                   p(out["J"]), p(out["H"]))
        return out


def build_c_oracle(solver, name: str, shared_parameters: bool = False, cse: bool = False, opt: str = "-O2",
                   verbose: bool = False) -> COracle:
    src = emit_c(solver, shared_parameters, cse)
    h = hashlib.sha256((src + opt).encode()).hexdigest()[:12]
    fname = f"oracle_{name}_{'cse' if cse else 'nocse'}_{h}"
    if os.path.exists(os.path.join(BUILD_DIR, fname + ".so")):
        return COracle(os.path.join(BUILD_DIR, fname + ".so"))
    # a process that must not write into the source tree (bench.py) points DTO_CACHE_DIR elsewhere
    cache = os.environ.get("DTO_CACHE_DIR") or BUILD_DIR
    os.makedirs(cache, exist_ok=True)
    base = os.path.join(cache, fname)
    if not os.path.exists(base + ".so"):
        with open(base + ".c", "w") as f:
            f.write(src)
        cmd = ["gcc", opt, "-fopenmp", "-shared", "-fPIC", "-o", base + ".so.tmp", base + ".c", "-lm"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("gcc failed:\n" + r.stderr[-3000:])
        os.replace(base + ".so.tmp", base + ".so")
        if verbose:
            print("[oracle cgen] built", base + ".so")
    return COracle(base + ".so")

"""Expression DAG + derivative synthesis for the code generator.

Why this exists: the reference differentiates every output symbolically and `eval`s one
un-shared expression per nonzero (/root/reference/src/dynamics.jl:25-34). For cartpole-RK3
that is ~15 k (Jacobian) + ~138 k (Hessian) operations per knot; tree-level CSE of those
expanded expressions still leaves ~2 k FP64 instructions and ~600 live temporaries (register
spills on the GPU). The chain-rule structure is lost by expansion, so the code generator
does NOT lower the expanded derivatives. It converts the traced RESIDUAL (a ~150-node DAG
that still has the RK-stage nesting) into a hash-consed DAG and synthesises the first and
second derivatives on that DAG by sparse second-order forward propagation: every node
carries a sparse gradient {var: node} and a sparse symmetric Hessian {(v,w): node}; all
derivative nodes are hash-consed, so equal sub-derivatives (e.g. d/dx_i and d/dy_i through a
midpoint 0.5(x+y)) are computed once. The values are the same mathematical functions the
reference evaluates (parity is checked against the oracle at 1e-12).

Node algebra is deliberately small: const, in, add, mul, neg, rcp, powi, unary functions.
Negations and numeric factors are floated outward so that +/- and scaled variants share nodes.
"""
from __future__ import annotations

import math
from typing import Dict, Iterable, List, Optional, Sequence, Tuple

import sympy as sp

UNARY = ("sin", "cos", "tan", "exp", "log", "sqrt", "atan", "sinh", "cosh", "tanh")
CMP = {"lt": "<", "le": "<=", "gt": ">", "ge": ">=", "eq": "==", "ne": "!="}  # boolean nodes (a, b)


class Graph:
    def __init__(self):
        self.op: List[str] = []
        self.args: List[tuple] = []
        self.val: List[object] = []
        self._memo: Dict[tuple, int] = {}
        self.ZERO = self.const(0.0)
        self.ONE = self.const(1.0)

    # ---- raw node creation
    def _mk(self, op: str, args: tuple = (), val=None) -> int:
        key = (op, args, val)
        i = self._memo.get(key)
        if i is None:
            i = len(self.op)
            self.op.append(op)
            self.args.append(args)
            self.val.append(val)
            self._memo[key] = i
        return i

    def const(self, v: float) -> int:
        v = float(v)
        if v == 0.0:
            v = 0.0  # fold -0.0
        return self._mk("const", (), v)

    def inp(self, name: str, idx: int) -> int:
        return self._mk("in", (), (name, idx))

    def is_const(self, a: int) -> bool:
        return self.op[a] == "const"

    def cval(self, a: int) -> float:
        return self.val[a]

    # ---- (coefficient, core) view: a = c * core with core free of numeric factor / negation
    def split(self, a: int) -> Tuple[float, int]:
        op = self.op[a]
        if op == "const":
            return self.val[a], self.ONE
        if op == "neg":
            c, x = self.split(self.args[a][0])
            return -c, x
        if op == "mul" and self.op[self.args[a][0]] == "const":
            c, x = self.split(self.args[a][1])
            return self.val[self.args[a][0]] * c, x
        return 1.0, a

    def scale(self, c: float, x: int) -> int:
        """c * x with x a core (non-const, no leading factor)."""
        if c == 0.0 or (self.is_const(x) and self.val[x] == 0.0):
            return self.ZERO
        if self.is_const(x):
            return self.const(c * self.val[x])
        if c == 1.0:
            return x
        if c == -1.0:
            return self._mk("neg", (x,))
        if c < 0:
            return self._mk("neg", (self._mk("mul", (self.const(-c), x)),))
        return self._mk("mul", (self.const(c), x))

    # ---- smart constructors
    def neg(self, a: int) -> int:
        c, x = self.split(a)
        return self.scale(-c, x)

    def add(self, a: int, b: int) -> int:
        if self.is_const(a) and self.is_const(b):
            return self.const(self.val[a] + self.val[b])
        if self.is_const(a) and self.val[a] == 0.0:
            return b
        if self.is_const(b) and self.val[b] == 0.0:
            return a
        ca, xa = self.split(a)
        cb, xb = self.split(b)
        if xa == xb and not self.is_const(a) and not self.is_const(b):
            return self.scale(ca + cb, xa)  # c1*x + c2*x
        # float a common negation outward: (-p) + (-q) = -(p + q)
        if ca < 0 and cb < 0 and not self.is_const(a) and not self.is_const(b):
            return self.neg(self.add(self.neg(a), self.neg(b)))
        if a > b:
            a, b = b, a
        return self._mk("add", (a, b))

    def sub(self, a: int, b: int) -> int:
        return self.add(a, self.neg(b))

    def mul(self, a: int, b: int) -> int:
        ca, xa = self.split(a)
        cb, xb = self.split(b)
        c = ca * cb
        if c == 0.0:
            return self.ZERO
        if xa == self.ONE:
            return self.scale(c, xb) if xb != self.ONE else self.const(c)
        if xb == self.ONE:
            return self.scale(c, xa)
        if xa == xb:
            core = self.powi(xa, 2)
        else:
            # x * x^k -> x^(k+1)
            if self.op[xa] == "powi" and self.op[xb] == "powi" and self.args[xa][0] == self.args[xb][0]:
                core = self.powi(self.args[xa][0], self.val[xa] + self.val[xb])
            elif self.op[xb] == "powi" and self.args[xb][0] == xa:
                core = self.powi(xa, self.val[xb] + 1)
            elif self.op[xa] == "powi" and self.args[xa][0] == xb:
                core = self.powi(xb, self.val[xa] + 1)
            else:
                if xa > xb:
                    xa, xb = xb, xa
                core = self._mk("mul", (xa, xb))
        c2, core2 = self.split(core)
        return self.scale(c * c2, core2)

    def rcp(self, a: int) -> int:
        c, x = self.split(a)
        if x == self.ONE:
            return self.const(1.0 / c)
        if self.op[x] == "rcp":
            return self.scale(1.0 / c, self.args[x][0])
        return self.scale(1.0 / c, self._mk("rcp", (x,)))

    def div(self, a: int, b: int) -> int:
        return self.mul(a, self.rcp(b))

    def powi(self, a: int, k: int) -> int:
        k = int(k)
        if k == 0:
            return self.ONE
        if k < 0:
            return self.powi(self.rcp(a), -k)
        if k == 1:
            return a
        c, x = self.split(a)
        if x == self.ONE:
            return self.const(c ** k)
        if self.op[x] == "powi":
            core = self._mk("powi", (self.args[x][0],), self.val[x] * k)
        else:
            core = self._mk("powi", (x,), k)
        return self.scale(c ** k, core)

    def func(self, name: str, a: int) -> int:
        if self.is_const(a):
            return self.const(getattr(math, name)(self.val[a]))
        if name == "sqrt":
            return self._mk("sqrt", (a,))
        c, x = self.split(a)
        if c < 0:  # parity: sin(-x) = -sin(x), cos(-x) = cos(x), tan/atan/sinh/tanh odd, cosh even
            if name in ("sin", "tan", "atan", "sinh", "tanh"):
                return self.neg(self._mk(name, (self.neg(a),)))
            if name in ("cos", "cosh"):
                return self._mk(name, (self.neg(a),))
        return self._mk(name, (a,))

    def cmp(self, op: str, a: int, b: int) -> int:
        """boolean node a <op> b (only ever the condition of a `sel`)"""
        return self._mk(op, (a, b))

    def sel(self, c: int, a: int, b: int) -> int:
        """ifelse(c, a, b)"""
        if a == b:
            return a
        return self._mk("sel", (c, a, b))

    def powc(self, a: int, p: float) -> int:
        """a ** p for a non-integer constant exponent."""
        if p == 0.5:
            return self.func("sqrt", a)
        if self.is_const(a):
            return self.const(self.val[a] ** p)
        return self._mk("powc", (a,), float(p))

    def sum(self, xs: Iterable[int]) -> int:
        acc = self.ZERO
        for x in xs:
            acc = self.add(acc, x)
        return acc

    def clone(self) -> "Graph":
        """Independent copy (node ids preserved): the cut search differentiates many trial copies."""
        h = Graph.__new__(Graph)
        h.op, h.args, h.val = list(self.op), list(self.args), list(self.val)
        h._memo = dict(self._memo)
        h.ZERO, h.ONE = self.ZERO, self.ONE
        return h

    def subst(self, n: int, mapping: Dict[int, int], memo: Optional[dict] = None) -> int:
        """Rebuild node n with the nodes in `mapping` replaced (through the smart constructors)."""
        memo = {} if memo is None else memo
        order = [(n, False)]
        while order:
            m, done = order.pop()
            if m in memo:
                continue
            if m in mapping:
                memo[m] = mapping[m]
                continue
            op, a = self.op[m], self.args[m]
            if op in ("const", "in"):
                memo[m] = m
                continue
            if not done:
                order.append((m, True))
                order.extend((x, False) for x in a if x not in memo)
                continue
            b = [memo[x] for x in a]
            if all(x == y for x, y in zip(a, b)):
                r = m
            elif op == "add":
                r = self.add(b[0], b[1])
            elif op == "mul":
                r = self.mul(b[0], b[1])
            elif op == "neg":
                r = self.neg(b[0])
            elif op == "rcp":
                r = self.rcp(b[0])
            elif op == "powi":
                r = self.powi(b[0], self.val[m])
            elif op == "powc":
                r = self.powc(b[0], self.val[m])
            elif op in CMP:
                r = self.cmp(op, b[0], b[1])
            elif op == "sel":
                r = self.sel(b[0], b[1], b[2])
            else:
                r = self.func(op, b[0])
            memo[m] = r
        return memo[n]

    def evaluate(self, nodes: Sequence[int], inputs: Dict[Tuple[str, int], float]) -> List[float]:
        """Numeric value of `nodes` (host-side check of the derivative synthesis; tests only)."""
        need, stack = set(), list(nodes)
        while stack:
            m = stack.pop()
            if m in need:
                continue
            need.add(m)
            stack.extend(self.args[m])
        v: Dict[int, float] = {}
        for m in sorted(need):
            op, a = self.op[m], self.args[m]
            if op == "const":
                v[m] = self.val[m]
            elif op == "in":
                v[m] = float(inputs[self.val[m]])
            elif op == "add":
                v[m] = v[a[0]] + v[a[1]]
            elif op == "mul":
                v[m] = v[a[0]] * v[a[1]]
            elif op == "neg":
                v[m] = -v[a[0]]
            elif op == "rcp":
                v[m] = 1.0 / v[a[0]]
            elif op == "powi":
                v[m] = v[a[0]] ** self.val[m]
            elif op == "powc":
                v[m] = v[a[0]] ** self.val[m]
            elif op in CMP:
                x_, y_ = v[a[0]], v[a[1]]
                v[m] = {"lt": x_ < y_, "le": x_ <= y_, "gt": x_ > y_, "ge": x_ >= y_, "eq": x_ == y_, "ne": x_ != y_}[op]
            elif op == "sel":
                v[m] = v[a[1]] if v[a[0]] else v[a[2]]
            else:
                v[m] = getattr(math, op)(v[a[0]])
        return [v[m] for m in nodes]

    # ---- sympy -> DAG
    def from_sympy(self, e: sp.Expr, sym: Dict[sp.Symbol, int], memo: Optional[dict] = None) -> int:
        memo = {} if memo is None else memo
        return self._conv(sp.sympify(e), sym, memo)

    def _conv(self, e, sym, memo) -> int:
        r = memo.get(e)
        if r is not None:
            return r
        if e.is_Symbol:
            r = sym[e]
        elif e.is_Number or e.is_NumberSymbol:
            r = self.const(float(e))
        elif e.is_Add:
            r = self.ZERO
            for a in e.args:
                r = self.add(r, self._conv(a, sym, memo))
        elif e.is_Mul:
            r = self.ONE
            for a in e.args:
                r = self.mul(r, self._conv(a, sym, memo))
        elif e.is_Pow:
            b, p = e.args
            if p.is_Integer:
                r = self.powi(self._conv(b, sym, memo), int(p))
            elif p.is_Number and float(p) == int(float(p)):
                r = self.powi(self._conv(b, sym, memo), int(float(p)))
            elif p.is_Number:
                r = self.powc(self._conv(b, sym, memo), float(p))
            else:
                # a^b = exp(b log a)
                r = self.func("exp", self.mul(self._conv(p, sym, memo), self.func("log", self._conv(b, sym, memo))))
        elif isinstance(e, sp.Piecewise):
            (val, cond) = e.args[-1]
            if cond is not sp.true:
                raise NotImplementedError("Piecewise without an otherwise branch")
            r = self._conv(val, sym, memo)
            for val, cond in reversed(e.args[:-1]):
                if not cond.is_Relational:
                    raise NotImplementedError(f"no DAG lowering for condition {cond}")
                op = {"<": "lt", "<=": "le", ">": "gt", ">=": "ge", "==": "eq", "!=": "ne"}[cond.rel_op]
                c = self.cmp(op, self._conv(cond.lhs, sym, memo), self._conv(cond.rhs, sym, memo))
                r = self.sel(c, self._conv(val, sym, memo), r)
        elif e.is_Function and len(e.args) == 1 and e.func.__name__ in UNARY:
            r = self.func(e.func.__name__, self._conv(e.args[0], sym, memo))
        else:
            raise NotImplementedError(f"no DAG lowering for {e.func}")
        memo[e] = r
        return r

    # ---- first/second derivative of a unary function at node c = f(a): returns (f', f'')
    def _dfun(self, c: int) -> Tuple[int, int]:
        op, a = self.op[c], self.args[c][0]
        if op == "sin":
            return self.func("cos", a), self.neg(c)
        if op == "cos":
            return self.neg(self.func("sin", a)), self.neg(c)
        if op == "tan":
            d1 = self.add(self.ONE, self.powi(c, 2))
            return d1, self.mul(self.const(2.0), self.mul(c, d1))
        if op == "exp":
            return c, c
        if op == "log":
            r = self.rcp(a)
            return r, self.neg(self.powi(r, 2))
        if op == "sqrt":
            r = self.rcp(c)
            return self.mul(self.const(0.5), r), self.mul(self.const(-0.25), self.powi(r, 3))
        if op == "atan":
            r = self.rcp(self.add(self.ONE, self.powi(a, 2)))
            return r, self.mul(self.const(-2.0), self.mul(a, self.powi(r, 2)))
        if op == "sinh":
            return self.func("cosh", a), c
        if op == "cosh":
            return self.func("sinh", a), c
        if op == "tanh":
            d1 = self.sub(self.ONE, self.powi(c, 2))
            return d1, self.mul(self.const(-2.0), self.mul(c, d1))
        if op == "rcp":
            return self.neg(self.powi(c, 2)), self.mul(self.const(2.0), self.powi(c, 3))
        if op == "powi":
            k = self.val[c]
            return self.mul(self.const(float(k)), self.powi(a, k - 1)), \
                self.mul(self.const(float(k * (k - 1))), self.powi(a, k - 2))
        if op == "powc":
            p = self.val[c]
            d1 = self.mul(self.const(p), self.powc(a, p - 1.0) if (p - 1.0) != int(p - 1.0) else self.powi(a, int(p - 1.0)))
            p2 = p - 2.0
            d2 = self.mul(self.const(p * (p - 1.0)), self.powc(a, p2) if p2 != int(p2) else self.powi(a, int(p2)))
            return d1, d2
        raise NotImplementedError(f"no derivative rule for {op}")


class Derivatives:
    """Sparse second-order forward propagation over a Graph w.r.t. `wrt`: input nodes, or any
    intermediate nodes declared as leaves (the traversal stops there; used by `hierarchical`)."""

    def __init__(self, g: Graph, wrt: Sequence[int], second: bool = True):
        self.g = g
        self.index = {n: i for i, n in enumerate(wrt)}
        self.second = second
        self._grad: Dict[int, Dict[int, int]] = {}
        self._hess: Dict[int, Dict[Tuple[int, int], int]] = {}

    def grad(self, n: int) -> Dict[int, int]:
        r = self._grad.get(n)
        if r is None:
            self._compute(n)
            r = self._grad[n]
        return r

    def hess(self, n: int) -> Dict[Tuple[int, int], int]:
        r = self._hess.get(n)
        if r is None:
            self._compute(n)
            r = self._hess[n]
        return r

    def _compute(self, root: int) -> None:
        g = self.g
        # iterative post-order over not-yet-differentiated ancestors
        stack = [(root, False)]
        while stack:
            n, done = stack.pop()
            if n in self._grad:
                continue
            if n in self.index:  # a leaf of this differentiation (input or cut node)
                self._grad[n] = {self.index[n]: g.ONE}
                self._hess[n] = {}
                continue
            if not done:
                stack.append((n, True))
                for a in g.args[n]:
                    if a not in self._grad:
                        stack.append((a, False))
                continue
            self._node(n)

    def _acc(self, d: dict, k, v: int) -> None:
        g = self.g
        if v == g.ZERO:
            return
        cur = d.get(k)
        d[k] = v if cur is None else g.add(cur, v)
        if d[k] == g.ZERO:
            del d[k]

    def _node(self, n: int) -> None:
        g = self.g
        op = g.op[n]
        G: Dict[int, int] = {}
        H: Dict[Tuple[int, int], int] = {}
        if op == "const":
            pass
        elif op == "in":
            i = self.index.get(n)
            if i is not None:
                G[i] = g.ONE
        elif op == "neg":
            a = g.args[n][0]
            for k, v in self._grad[a].items():
                G[k] = g.neg(v)
            if self.second:
                for k, v in self._hess[a].items():
                    H[k] = g.neg(v)
        elif op == "add":
            a, b = g.args[n]
            for src in (a, b):
                for k, v in self._grad[src].items():
                    self._acc(G, k, v)
            if self.second:
                for src in (a, b):
                    for k, v in self._hess[src].items():
                        self._acc(H, k, v)
        elif op == "mul":
            a, b = g.args[n]
            ga, gb = self._grad[a], self._grad[b]
            for k, v in ga.items():
                self._acc(G, k, g.mul(b, v))
            for k, v in gb.items():
                self._acc(G, k, g.mul(a, v))
            if self.second:
                for k, v in self._hess[a].items():
                    self._acc(H, k, g.mul(b, v))
                for k, v in self._hess[b].items():
                    self._acc(H, k, g.mul(a, v))
                for i, vi in ga.items():
                    for j, vj in gb.items():
                        t = g.mul(vi, vj)
                        if i == j:
                            self._acc(H, (i, i), g.mul(g.const(2.0), t))
                        else:
                            self._acc(H, (i, j) if i < j else (j, i), t)
        elif op in CMP:
            pass  # a condition: piecewise constant, no derivative
        elif op == "sel":
            c, a, b = g.args[n]
            ga, gb = self._grad[a], self._grad[b]
            for k in sorted(set(ga) | set(gb)):
                self._acc(G, k, g.sel(c, ga.get(k, g.ZERO), gb.get(k, g.ZERO)))
            if self.second:
                ha, hb = self._hess[a], self._hess[b]
                for k in sorted(set(ha) | set(hb)):
                    self._acc(H, k, g.sel(c, ha.get(k, g.ZERO), hb.get(k, g.ZERO)))
        else:  # unary function of args[0]
            a = g.args[n][0]
            ga = self._grad[a]
            if ga:
                d1, d2 = g._dfun(n)
                for k, v in ga.items():
                    self._acc(G, k, g.mul(d1, v))
                if self.second:
                    for k, v in self._hess[a].items():
                        self._acc(H, k, g.mul(d1, v))
                    if d2 != g.ZERO:
                        items = sorted(ga.items())
                        # d2 * ga[i] is shared by every pair (i, j)
                        for x, (i, vi) in enumerate(items):
                            d2vi = g.mul(d2, vi)
                            for (j, vj) in items[x:]:
                                self._acc(H, (i, j), g.mul(d2vi, vj))
        self._grad[n] = G
        self._hess[n] = H


# ----------------------------------------------------------------------------- hierarchical derivatives
def _reach(g: Graph, roots: Iterable[int], stop: set) -> set:
    seen, st = set(), list(roots)
    while st:
        n = st.pop()
        if n in seen:
            continue
        seen.add(n)
        if n in stop:
            continue
        st.extend(g.args[n])
    return seen


def hierarchical(g: Graph, outs: Sequence[int], L: Optional[int], wrt: Sequence[int], cuts: Sequence[int] = (),
                 second: bool = True) -> Tuple[List[Dict[int, int]], Dict[Tuple[int, int], int]]:
    """First derivatives of `outs` and the Hessian of the scalar `L` w.r.t. the inputs `wrt`, with the
    intermediate nodes `cuts` used as LOCAL differentiation variables.

    Plain forward propagation carries, at every node, a gradient / Hessian in the GLOBAL variables; after
    an RK stage or a midpoint these are dense (cartpole: 3 + 6 entries per node) although the node
    depends on one or two stage quantities. Here the DAG is split at the cut nodes: a cut node c_k is a
    function phi_k of the inputs and of earlier cuts, and so is L. Per level of cuts:
      * local first/second derivatives of phi_k w.r.t. its own leaves (sparse in those),
      * global tangents by the chain rule,   T(c_k) = sum_leaf dphi_k/dleaf * T(leaf),
      * adjoints by one reverse sweep over the cut nodes,   cbar_k = dL/dc_k,
      * Hessian = sum over levels of  T' M T,  M = local Hessian of  sum_k cbar_k * phi_k  (the adjoints
        enter as placeholders while differentiating and are substituted afterwards), which is the
        second-order chain rule contracted with the adjoint BEFORE the congruence.
    With no cuts this is exactly the plain forward propagation. Returns ([{var index: node}] per output,
    {(i, j), i <= j: node})."""
    cuts = sorted(set(cuts))
    cutset = set(cuts)
    wset = set(wrt)
    level: Dict[int, int] = {}
    for c in cuts:
        anc = _reach(g, g.args[c], cutset)
        level[c] = 1 + max([level[a] for a in anc if a in cutset], default=0)
    nlev = max(level.values(), default=0)
    groups: List[Optional[List[int]]] = [[c for c in cuts if level[c] == lv] for lv in range(1, nlev + 1)]
    gidx = {n: i for i, n in enumerate(wrt)}
    T: Dict[int, Dict[int, int]] = {n: {gidx[n]: g.ONE} for n in wrt}

    def chain(gloc: Dict[int, int], leaves: List[int]) -> Dict[int, int]:
        out: Dict[int, int] = {}
        for li, d in sorted(gloc.items()):
            for i, t in T[leaves[li]].items():
                v = g.mul(d, t)
                out[i] = v if i not in out else g.add(out[i], v)
        return {i: v for i, v in out.items() if v != g.ZERO}

    info = []
    nph = 0
    jac: List[Dict[int, int]] = []
    for grp in groups + [None]:
        roots = list(grp) if grp is not None else list(outs) + ([L] if L is not None else [])
        rr: set = set()
        for c in roots:
            rr |= _reach(g, g.args[c] if grp is not None else [c], cutset)
        leaves = sorted(n for n in rr if n in cutset or n in wset)
        LD = Derivatives(g, leaves, second=second)
        if grp is not None:
            gloc = {c: dict(LD.grad(c)) for c in grp}
            for c in grp:
                T[c] = chain(gloc[c], leaves)
            hloc, ph = {}, []
            if second:
                ph = [g.inp("__adj", nph + k) for k in range(len(grp))]
                nph += len(grp)
                hloc = LD.hess(g.sum(g.mul(p, c) for p, c in zip(ph, grp)))
            info.append((grp, leaves, gloc, hloc, ph))
        else:
            jac = [chain(dict(LD.grad(o)), leaves) for o in outs]
            if second and L is not None:
                info.append((None, leaves, {L: dict(LD.grad(L))}, LD.hess(L), None))
    if not second or L is None:
        return jac, {}
    # adjoints of the cut nodes: reverse sweep over the levels
    cbar: Dict[int, int] = {}
    for grp, leaves, gloc, hloc, ph in reversed(info):
        for c in ([L] if grp is None else grp):
            wgt = g.ONE if grp is None else cbar.get(c, g.ZERO)
            if wgt == g.ZERO:
                continue
            for li, d in sorted(gloc[c].items()):
                leaf = leaves[li]
                if leaf in cutset:
                    v = g.mul(wgt, d)
                    cbar[leaf] = v if leaf not in cbar else g.add(cbar[leaf], v)
    # Hessian: congruence of every level's adjoint-weighted local Hessian with the global tangents
    H: Dict[Tuple[int, int], int] = {}
    for grp, leaves, gloc, hloc, ph in info:
        if grp is not None:
            mp = {p: cbar.get(c, g.ZERO) for p, c in zip(ph, grp)}
            memo: dict = {}
            hloc = {k: g.subst(v, mp, memo) for k, v in hloc.items()}
        N: Dict[int, Dict[int, int]] = {}
        for (a, b), m in sorted(hloc.items()):
            if m == g.ZERO:
                continue
            for p, q in (((a, b),) if a == b else ((a, b), (b, a))):
                row = N.setdefault(p, {})
                for j, t in T[leaves[q]].items():
                    v = g.mul(m, t)
                    row[j] = v if j not in row else g.add(row[j], v)
        for a, row in sorted(N.items()):
            for i, ti in T[leaves[a]].items():
                for j, nj in sorted(row.items()):
                    if i <= j:
                        v = g.mul(ti, nj)
                        H[(i, j)] = v if (i, j) not in H else g.add(H[(i, j)], v)
    return jac, {k: v for k, v in H.items() if v != g.ZERO}


def _total_ops(g: Graph, nodes: Sequence[int]) -> int:
    return sum(count_ops(g, nodes).values())


def choose_cuts(g: Graph, outs: Sequence[int], L: int, wrt: Sequence[int], select, max_evals: int = 4000,
                min_ops: int = 60) -> Tuple[List[int], Dict[str, int]]:
    """Cut nodes for `hierarchical` by local search on the exact operation count of the fused program.
    `select(jac, H, graph)` returns the output nodes whose cost counts. Candidates: intermediate nodes
    that depend on >= 2 differentiation variables. Greedy single additions / removals, then pairs, within
    an evaluation budget (deterministic: the result depends on the model only)."""
    def cost(cc) -> int:
        h = g.clone()
        jac, H = hierarchical(h, outs, L, wrt, sorted(cc))
        return _total_ops(h, select(jac, H, h))

    base = cost(())
    stats = {"plain": base, "evals": 1}
    if base < min_ops:
        stats["ops"] = base
        return [], stats
    wset = set(wrt)
    sup: Dict[int, frozenset] = {}
    for n in sorted(_reach(g, list(outs) + [L], set())):
        if g.op[n] == "in":
            sup[n] = frozenset([n]) if n in wset else frozenset()
        elif g.op[n] == "const":
            sup[n] = frozenset()
        else:
            s_: frozenset = frozenset()
            for a in g.args[n]:
                s_ |= sup[a]
            sup[n] = s_
    cands = [n for n in sorted(sup) if g.op[n] not in ("in", "const", "neg") and g.op[n] not in CMP and len(sup[n]) >= 2
             and n != L and n not in outs]
    cur: set = set()
    best = base
    evals = 1
    pos = {c: i for i, c in enumerate(cands)}
    # pairs, nearest first: related quantities (the components of one stage vector) are created together
    pairs = sorted(((c, d) for x, c in enumerate(cands) for d in cands[x + 1:]), key=lambda cd: (pos[cd[1]] - pos[cd[0]], cd))
    while evals < max_evals:
        improved = False
        for c in cands:  # single additions / removals, first improvement
            trial = (cur - {c}) if c in cur else (cur | {c})
            v = cost(trial)
            evals += 1
            if v < best:
                best, cur, improved = v, trial, True
            if evals >= max_evals:
                break
        if improved:
            continue
        for c, d in pairs:  # no single move helps: first improving pair addition, then singles again
            if c in cur or d in cur:
                continue
            v = cost(cur | {c, d})
            evals += 1
            if v < best:
                best, cur, improved = v, cur | {c, d}, True
                break
            if evals >= max_evals:
                break
        if not improved:
            break
    stats.update(ops=best, evals=evals, cuts=len(cur))
    return sorted(cur), stats


# ----------------------------------------------------------------------------- emission
def _lit(v: float) -> str:
    r = repr(float(v))
    if "e" not in r and "." not in r and "inf" not in r and "nan" not in r:
        r += ".0"
    return r


def count_ops(g: Graph, outputs: Sequence[int]) -> Dict[str, int]:
    seen, stack = set(), list(outputs)
    while stack:
        n = stack.pop()
        if n in seen:
            continue
        seen.add(n)
        stack.extend(g.args[n])
    c: Dict[str, int] = {}
    for n in seen:
        op = g.op[n]
        if op == "powi":
            k = g.val[n]
            c["mul"] = c.get("mul", 0) + (k.bit_length() - 1) + bin(k).count("1") - 1
        elif op not in ("const", "in", "neg"):
            c[op] = c.get(op, 0) + 1
    return c


def _needs_pool(v: float) -> bool:
    """FP64 instructions take a 32-bit immediate = the HIGH word of the double; anything with a
    non-zero low word (0.05, 9.81, 1/6 ...) would be materialised with two UMOVs per use, so it
    goes to the constant bank instead (read as a direct c[bank][ofs] operand)."""
    import struct
    return (struct.unpack("<Q", struct.pack("<d", float(v)))[0] & 0xFFFFFFFF) != 0


def emit(g: Graph, outputs: List[Tuple[str, int]], load: Dict[Tuple[str, int], str], indent: str = "    ",
         prefix: str = "t", cpool: Optional[Dict[float, int]] = None, cname: str = "dto_k", order: int = 0,
         bf: bool = False) -> List[str]:
    """Straight-line C for the nodes reachable from `outputs` [(lhs, node)], DFS post-order in
    output order (keeps live ranges short), or with order=2 register-pressure-aware list scheduling; sin/cos of one
    argument become one sincos().
    bf=True: sin/cos/reciprocal use the branch-free device functions dto_sincos_bf / dto_rcp_bf, which
    OR a flag into the local `dto_bad` when an argument is outside their domain (the caller then
    re-evaluates with the library functions): the whole program becomes ONE basic block, so ptxas can
    overlap the serial Horner / Newton chains with independent work."""
    name: Dict[int, str] = {}
    lines: List[str] = []
    need = set()
    stack = [n for _, n in outputs]
    while stack:
        n = stack.pop()
        if n in need:
            continue
        need.add(n)
        stack.extend(g.args[n])
    # sincos pairing
    sin_of = {g.args[n][0]: n for n in need if g.op[n] == "sin"}
    cos_of = {g.args[n][0]: n for n in need if g.op[n] == "cos"}
    paired = {a for a in sin_of if a in cos_of}

    def ref(n: int) -> str:
        op = g.op[n]
        if op == "const":
            v = g.val[n]
            if cpool is not None and _needs_pool(v):
                k = abs(v)
                idx = cpool.setdefault(k, len(cpool))
                return f"{cname}[{idx}]" if v >= 0 else f"(-{cname}[{idx}])"
            return _lit(v) if v >= 0 else f"({_lit(v)})"
        if op == "neg":
            return f"(-{ref(g.args[n][0])})"
        return name[n]

    def define(n: int) -> None:
        op = g.op[n]
        if op in ("const", "neg") or n in name:
            return
        nm = f"{prefix}{n}"
        a = g.args[n]
        if op == "in":
            name[n] = nm
            lines.append(f"{indent}const double {nm} = {load[g.val[n]]};")
        elif op == "add":
            name[n] = nm
            # print a + (-b) as a - b
            x, y = a
            if g.op[y] == "neg":
                lines.append(f"{indent}const double {nm} = {ref(x)} - {ref(g.args[y][0])};")
            elif g.op[x] == "neg":
                lines.append(f"{indent}const double {nm} = {ref(y)} - {ref(g.args[x][0])};")
            else:
                lines.append(f"{indent}const double {nm} = {ref(x)} + {ref(y)};")
        elif op == "mul":
            name[n] = nm
            lines.append(f"{indent}const double {nm} = {ref(a[0])} * {ref(a[1])};")
        elif op == "rcp":
            name[n] = nm
            if bf:
                lines.append(f"{indent}const double {nm} = dto_rcp_bf({ref(a[0])}, dto_bad);")
            else:
                lines.append(f"{indent}const double {nm} = 1.0 / {ref(a[0])};")
        elif op == "powi":
            name[n] = nm
            lines.append(f"{indent}const double {nm} = dto_powi<{g.val[n]}>({ref(a[0])});")
        elif op == "powc":
            name[n] = nm
            lines.append(f"{indent}const double {nm} = pow({ref(a[0])}, {_lit(g.val[n])});")
        elif op in CMP:
            name[n] = nm
            lines.append(f"{indent}const bool {nm} = {ref(a[0])} {CMP[op]} {ref(a[1])};")
        elif op == "sel":
            name[n] = nm
            lines.append(f"{indent}const double {nm} = {ref(a[0])} ? {ref(a[1])} : {ref(a[2])};")
        elif op in ("sin", "cos") and a[0] in paired:
            s, c = sin_of[a[0]], cos_of[a[0]]
            name[s], name[c] = f"{prefix}{s}", f"{prefix}{c}"
            fnm = "dto_sincos_bf" if bf else "sincos"
            tail = ", dto_bad" if bf else ""
            lines.append(f"{indent}double {name[s]}, {name[c]}; {fnm}({ref(a[0])}, &{name[s]}, &{name[c]}{tail});")
        elif op in ("sin", "cos") and bf:
            name[n] = nm
            other = f"{nm}_o"
            args_ = f"&{nm}, &{other}" if op == "sin" else f"&{other}, &{nm}"
            lines.append(f"{indent}double {nm}, {other}; dto_sincos_bf({ref(a[0])}, {args_}, dto_bad);")
        else:
            name[n] = nm
            lines.append(f"{indent}const double {nm} = {op}({ref(a[0])});")

    if order == 2:
        # register-pressure-aware list scheduling: among the ready nodes pick the one that retires the
        # most live values (last uses) -- ptxas largely keeps source order for long FP64 blocks, so
        # the emitted order decides how many registers the ~1000-instruction knot program needs
        def core(n: int) -> int:
            while g.op[n] == "neg":
                n = g.args[n][0]
            return n

        nodes = [n for n in sorted(need) if g.op[n] not in ("const", "neg")]
        ops_of = {n: [core(a) for a in g.args[n] if g.op[core(a)] != "const"] for n in nodes}
        uses: Dict[int, int] = {n: 0 for n in nodes}
        consumers: Dict[int, List[int]] = {n: [] for n in nodes}
        for n in nodes:
            for a in set(ops_of[n]):
                uses[a] += 1
                consumers[a].append(n)
        outs_of: Dict[int, List[str]] = {}
        for lhs, root in outputs:
            outs_of.setdefault(root, []).append(lhs)
        for lhs, root in outputs:
            c = core(root)
            if g.op[c] != "const":
                uses[c] += 0  # stores are emitted right at definition: they do not extend the live range
        missing = {n: len(set(ops_of[n])) for n in nodes}
        ready = [n for n in nodes if missing[n] == 0]
        done = set()
        last_pick = -1
        order_idx = {n: i for i, n in enumerate(nodes)}
        stored = set()

        def flush_outputs():
            for lhs, root in outputs:
                if lhs in stored:
                    continue
                c = core(root)
                if g.op[c] == "const" or c in done:
                    lines.append(f"{indent}{lhs} = {ref(root)};")
                    stored.add(lhs)

        flush_outputs()
        while ready:
            best, best_key = None, None
            for n in ready:
                frees = sum(1 for a in set(ops_of[n]) if uses[a] == 1)
                creates = 0 if (not consumers[n]) else 1
                # prefer: most net frees, then consumers of the value defined last (chains), then source order
                key = (frees - creates, 1 if last_pick in ops_of[n] else 0, -order_idx[n])
                if best_key is None or key > best_key:
                    best, best_key = n, key
            n = best
            ready.remove(n)
            define(n)
            if g.op[n] in ("sin", "cos") and g.args[n][0] in paired:  # sincos defines both
                for m_ in (sin_of[g.args[n][0]], cos_of[g.args[n][0]]):
                    if m_ not in done and m_ != n:
                        done.add(m_)
                        if m_ in ready:
                            ready.remove(m_)
                        for a in set(ops_of[m_]):
                            uses[a] -= 1
                        for c_ in consumers[m_]:
                            missing[c_] -= 1
                            if missing[c_] == 0 and c_ not in done:
                                ready.append(c_)
            done.add(n)
            last_pick = n
            for a in set(ops_of[n]):
                uses[a] -= 1
            for c_ in consumers[n]:
                missing[c_] -= 1
                if missing[c_] == 0 and c_ not in done and c_ not in ready:
                    ready.append(c_)
            flush_outputs()
        flush_outputs()
        assert len(stored) == len(outputs), "scheduler left outputs unstored"
        return lines
    # iterative DFS post-order
    for lhs, root in outputs:
        stack2 = [(root, False)]
        while stack2:
            n, done = stack2.pop()
            if n in name or g.op[n] == "const":
                continue
            if g.op[n] == "neg":
                stack2.append((g.args[n][0], False))
                continue
            if not done:
                stack2.append((n, True))
                for a in reversed(g.args[n]):
                    stack2.append((a, False))
                continue
            define(n)
        lines.append(f"{indent}{lhs} = {ref(root)};")
    return lines

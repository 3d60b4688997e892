"""Lock-step batched Newton-KKT (SQP) solver on top of the device-resident callbacks and KKT kernels.

Reference anchor: `solve!(solver)` (/root/reference/src/solver.jl:45-47) hands the five MOI callbacks to
Ipopt (src/data.jl:222-255). Ipopt (libipopt) is not in this image, and a CPU solver per problem fed through
PCIe is exactly the bottleneck the KKT consumer of SURVEY 8(f) N3 removes -- so BASELINE config 3 ("acrobot
T=101, batch 4096, full solves with device-resident callbacks") runs on this solver instead: every problem of
the batch advances through the same iteration at the same time, all arrays stay in HBM, and every linear
algebra / callback step is one of this package's CUDA kernels:

    callbacks at (z, lambda, sigma = 1)            dto_kkt_launch(with_callbacks = 1): gradient, constraint,
                                                   fused Jacobian + Hessian-of-Lagrangian kernels
    K = [[H + delta_b I, J'], [J, -delta_c I]]     kkt_band_kernel: per-problem delta_b (inertia control), banded
    K [dz; dlam] = -[g + J'lam; c]                 LDL' without pivoting, negative pivots counted per problem
    trial points z + alpha dz                      objective_kernel + knot_kernel<C> (batched f, c)

What is left to the host language are O(B N) vector updates and per-problem scalars (step acceptance,
regularisation, convergence masks); they are written against an array namespace `xp` -- torch on the device
for the product, numpy for the oracle-driven twin the parity test runs (tests/sqp_oracle.py) -- so both arms
execute literally the same algorithm.

Scope (stated plainly): equality rows, variables free or PINNED by equal lower and upper bounds (end points fixed by stage
constraints as in examples/acrobot, or by Bound(state_lower = x1, state_upper = x1) as in test/solve.jl), and inequalities --
BOUNDS on variables (Bound(action_lower = ..., action_upper = ...)) and inequality ROWS c_i(z) <= 0
(Constraint(...; indices_inequality)) -- in all three arms (`solve` / `solve_bounded` here; dto_sqp_solve with the k_ip_*
kernels). Inequalities are handled as a primal-dual interior point on the same
Newton-KKT step: the barrier terms are a per-problem diagonal the factor kernel adds to K while it gathers a row
(dto_kkt_device_pointer(k, 5): z_L/(x-l) + z_U/(u-x) on bounded variables, -t_i/lam_i on inequality rows whose slacks t
are eliminated), fraction-to-the-boundary steps, monotone barrier updates -- but WITHOUT Ipopt's feasibility-restoration
phase; `solve_bounded` adds a continuation on the bounds (widened tenfold, then tightened with a warm start) for the
problems the direct solve leaves unconverged. Measured on the reference's own examples, each from its own guess:
cartpole (T = 101, |u| <= 3, rollout guess): 4096 of 4096 problems, median 47 iterations, 23 % of the controls AT the
bound; car (T = 51, |u| <= 0.5, pinned ends, obstacle inequality per knot, interpolated guess): 99.7 % of 1024 guesses,
12 % of them through the continuation (tools/ip_cartpole.py, tools/ip_car.py, profiles/ip_*_r02.jsonl); pendulum with
|u| <= 15: device iterates = oracle-twin iterates to 1e-13. What the missing restoration phase costs: cartpole from a guess
whose states are interpolated from x1 to xT (not the example's) settles at ||c||_inf ~ 0.013 with 96 % of the controls
saturated, whatever the options and with the continuation -- a one-swing trajectory that actuator cannot complete.
`Solver.solve()` runs the native arm for all of these (method "native"); "sqp" is this file's torch-glued arm. It is a line-search SQP with an l1 merit function, a second-order correction, Levenberg-Marquardt
damping and Ipopt-style inertia correction of the primal regularisation; it is NOT Ipopt:
iterate-for-iterate parity with the reference's Ipopt runs is unverifiable here and is not claimed.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional


class HessianApproximation(str):
    """"exact", "knot-bfgs" or "partitioned-bfgs": a str whose float() is its dto_sqp_options.hessian_approximation code"""

    CODES = {"exact": 0, "knot-bfgs": 1, "partitioned-bfgs": 2}

    def __float__(self):
        return float(self.CODES[str(self)])


@dataclass
class SQPOptions:
    max_iter: int = 200
    tol_constraint: float = 1.0e-8     # ||c||_inf
    tol_dual: float = 1.0e-6           # ||g + J' lambda||_inf
    dual_reg: float = 1.0e-9           # delta_c: keeps K quasi-definite when J loses rank
    reg_first: float = 1.0e-4          # Ipopt's delta_w^0
    reg_min: float = 1.0e-20
    reg_max: float = 1.0e10
    reg_inc_first: float = 100.0       # kappa_w^+ bar
    reg_inc: float = 8.0               # kappa_w^+
    reg_dec: float = 1.0 / 3.0         # kappa_w^-
    max_refactor: int = 14
    armijo: float = 1.0e-4
    max_backtrack: int = 10            # lock step: the slowest search of the batch sets the pace (25 -> 8: 2.7 -> 1.8 s, same success rate)
    merit_margin: float = 1.1
    merit_rho: float = 0.3
    soc: bool = True
    merit_memory: bool = False
    merit_min: float = 1.0
    lm_first: float = 1.0e-2           # Levenberg-Marquardt damping added to H: first value, growth when the search
    lm_min: float = 1.0e-4             #   accepted less than lm_grow_below of the step, decay after full steps
    lm_grow: float = 4.0
    lm_shrink: float = 0.25
    lm_grow_below: float = 0.3
    lm_zero: float = 1.0e-10
    lam_max: float = 1.0e4             # multiplier estimates beyond this are reset to zero (Ipopt's lambda_max safeguard; 0 = off):
                                       #   config 3 97.1 % -> 99.4 % solved (the failures had |lambda| ~ 1e6..1e8 near rank-deficient Jacobians)
    repack: bool = False               # drop converged problems from the batch once they are half of it (they ride along in
    repack_min: int = 4096             #   lock step otherwise); never below repack_min problems. Off by default: at B = 4096 an
                                       #   iteration is bound by its ~60 launches and the latency of one banded factorisation, not
                                       #   by the batch size, so a smaller batch is no faster (measured 1.80 vs 1.53 s)
    exact_below: float = 1.0           # ||c||_inf under which the exact Hessian of the Lagrangian is used
    # ---- inequality bounds on variables (Bound(action_lower = ..., action_upper = ...), src/bounds.jl): primal-dual
    # interior point on top of the same Newton-KKT step (Ipopt's barrier treatment of the bounds MOI hands it,
    # src/data.jl:240-248): Sigma = z_L/(x - l) + z_U/(u - x) on the diagonal of H, fraction-to-the-boundary steps,
    # monotone barrier updates (Waechter & Biegler 2006, eqs. 7, 11-16)
    mu_init: float = 0.1
    barrier_kappa_eps: float = 10.0    # barrier problem solved to kappa_eps * mu before mu is decreased
    barrier_kappa_mu: float = 0.2
    barrier_theta_mu: float = 1.5
    tau_min: float = 0.99              # fraction to the boundary
    bound_push: float = 1.0e-2         # kappa_1 / kappa_2 of Ipopt's initial point push
    bound_frac: float = 1.0e-2
    kappa_sigma: float = 1.0e10        # z stays within [mu/(kappa s), kappa mu/s]
    tiny_step: float = 1.0e-6          # relative step size under which the full (fraction-to-the-boundary) step is taken untested
    bound_relax: float = 10.0          # fallback of `solve_bounded` for problems the direct solve leaves unconverged: two-sided bounds
                                       #   widened about their midpoint by this factor, solved, then the true bounds warm-started (<= 1: off)
    hessian_approximation: str = HessianApproximation("exact")   # "knot-bfgs": H is one dense block per knot, updated by damped BFGS (`knot_bfgs_update`) --
                                       #   for problems built without Hessians (the reference's default evaluate_hessian = false);
                                       #   the native arm only. exact_below does not apply (H is always the blocks).
                                       #   "partitioned-bfgs": one damped BFGS block per knot element over [x_t; u_t; x_{t+1}]
                                       #   (`knot_elements` states it); no general constraint


class SQPResult:
    def __init__(self, z, lam, iterations, converged, constraint_violation, dual_residual, objective, history, backend=None):
        self.backend = backend                  # the backend in use at the end (a smaller one after re-packing): close it
        self.z, self.lam = z, lam
        self.iterations = iterations            # per problem: iterations until it converged (or max_iter)
        self.converged = converged
        self.constraint_violation = constraint_violation
        self.dual_residual = dual_residual
        self.objective = objective
        self.history = history                  # list of per-iteration dicts (only with record=True)


def solve(be, z0, lam0=None, options: Optional[SQPOptions] = None, record: bool = False) -> SQPResult:
    """`be` is a backend (see DeviceBackend below / tests/sqp_oracle.py):
         be.xp                       array namespace (torch or numpy flavoured shim, see `_XP`)
         be.B, be.N_z, be.N_c
         be.free                     [N_z] 0/1 mask: 0 = variable pinned by equal bounds (its step is zero)
         be.callbacks(z, lam, lamH, delta) -> f [B], g [B,N_z], c [B,N_c]  (leaves J, H(z, lamH) and a first solve with delta ready for `newton`)
         be.newton(delta, mask=None) -> sol [B, N_z+N_c] = K^-1 [g + J'lam; c], nneg [B] negative pivots,
                                        rz [B,N_z] = g + J'lam   with per-problem primal regularisation delta [B];
                                        with a mask only those rows have to be recomputed (the others are ignored)
         be.newton_soc(c_soc, delta, mask) -> sol with the constraint right-hand side c_soc (masked rows)
         be.objective_constraint(z)  -> f [B], c [B,N_c]
    All arrays are [B, ...] and stay wherever `xp` keeps them."""
    o = options or SQPOptions()
    xp = be.xp
    B, N_z, N_c = be.B, be.N_z, be.N_c
    z = xp.copy(z0)
    if getattr(be, "pin", None) is not None:
        z = be.pin(z)
    lam = xp.zeros((B, N_c)) if lam0 is None else xp.copy(lam0)
    free = be.free
    delta_last = xp.zeros((B,))
    nu = xp.ones((B,))
    done = xp.zeros_bool((B,))
    iters = xp.zeros((B,))
    history = []
    f = cv = dr = None
    exact = xp.zeros((B,))
    lm = xp.full((B,), o.lm_first)
    # interior point state (only when the backend reports inequality bounds on variables)
    bnd = getattr(be, "bounds", None)
    ip = bnd is not None
    if ip:
        hasL, hasU, lo, up = bnd["hasL"], bnd["hasU"], bnd["lo"], bnd["up"]          # [N_z] masks (0/1) and finite values (0 where absent)
        z = xp.where((hasL > 0) & (z < lo + bnd["pushL"]), (lo + bnd["pushL"]) + 0.0 * z, z)    # into the interior (Ipopt sec. 3.6)
        z = xp.where((hasU > 0) & (z > up - bnd["pushU"]), (up - bnd["pushU"]) + 0.0 * z, z)
        zL = xp.ones((B, N_z)) * hasL
        zU = xp.ones((B, N_z)) * hasU
        mu = xp.full((B,), o.mu_init)
        # inequality rows c_i(z) <= 0 become c_i(z) + t_i = 0 with slacks t_i > 0; the slacks are eliminated from the Newton
        # system (their row of K gets -t_i/lam_i on the diagonal, lam_i > 0 doubling as the slack's bound multiplier)
        hasI = bnd["hasI"] if int(bnd["hasI"].shape[0]) == N_c else xp.zeros((N_c,))
        any_ineq = bool(xp.any(hasI > 0))
        t = None
        mu_floor = min(o.tol_constraint, o.tol_dual) / 10.0
        big = 1.0e300
    # results in the caller's problem order; `ids` = original problem number of every row of the working batch
    B0 = B
    ids = xp.arange(B0)
    out = dict(z=xp.copy(z), lam=xp.copy(lam), iters=xp.full((B0,), float(o.max_iter)), done=xp.zeros_bool((B0,)),
               cv=xp.zeros((B0,)), dr=xp.zeros((B0,)), f=xp.zeros((B0,)))

    def flush(rows):
        """current values of the working rows `rows` (boolean mask) -> result arrays"""
        sel = ids[rows]
        for key, val in (("z", z), ("lam", lam), ("iters", iters), ("done", done), ("cv", cv), ("dr", dr), ("f", f)):
            out[key][sel] = val[rows]

    for it in range(o.max_iter):
        B = be.B
        # Hessian of the Lagrangian with the multipliers of the problems that are close to feasible; the others
        # use the objective's Hessian only (Gauss-Newton): far from the constraint manifold the multiplier
        # estimates of a swing-up are huge and their curvature term makes H wildly indefinite
        # ---- Newton-KKT step: Levenberg-Marquardt damping lm (grows when the line search had to cut the step,
        # shrinks after full steps) + inertia control on top of it (Ipopt's IC algorithm, per problem)
        delta = xp.copy(lm)
        if ip:
            # barrier problem f - mu sum(log(x - l) + log(u - x)): its gradient replaces g, Sigma joins H's diagonal
            sL = xp.where(hasL > 0, z - lo, xp.ones((B, N_z)))
            sU = xp.where(hasU > 0, up - z, xp.ones((B, N_z)))
            SigL, SigU = hasL * zL / sL, hasU * zU / sU
            gshift = mu[:, None] * (hasU / sU - hasL / sL)
            if any_ineq:
                if t is None:       # first iteration: slacks from the constraint values at the start, multipliers on the central path
                    _, c0 = be.objective_constraint(z)
                    t = hasI * xp.maximum(-c0, xp.full((B, N_c), o.bound_push))
                    lam = xp.where(hasI > 0, mu[:, None] / xp.maximum(t, xp.full((B, N_c), 1.0e-300)), lam)
                tS = xp.where(hasI > 0, t, xp.ones((B, N_c)))
                lamI = xp.where(hasI > 0, lam, xp.ones((B, N_c)))
                diagC = -hasI * tS / lamI                        # (2,2) block: -t_i / lam_i on the inequality rows
                cshift = hasI * (mu[:, None] / lamI)             # their right-hand side: c_i + mu / lam_i
                f, g, c = be.callbacks(z, lam, lam * exact[:, None], delta, diag=xp.hcat(SigL + SigU, diagC), gshift=gshift, cshift=cshift)
                f = f - mu * xp.sum_rows(hasI * xp.log(tS))
                c = c + hasI * t                                 # residual of c(z) + t = 0
            else:
                f, g, c = be.callbacks(z, lam, lam * exact[:, None], delta, diag=SigL + SigU, gshift=gshift)
            f = f - mu * (xp.sum_rows(hasL * xp.log(sL)) + xp.sum_rows(hasU * xp.log(sU)))
        else:
            f, g, c = be.callbacks(z, lam, lam * exact[:, None], delta)
        sol, nneg, rz = be.newton(delta)
        cv = xp.max_abs_rows(c)
        if ip:
            # optimality error of the ORIGINAL problem: g + J'lam - z_L + z_U, and complementarity
            dr = xp.max_abs_rows((rz - gshift - zL + zU) * free)
            compL, compU = hasL * sL * zL, hasU * sU * zU
            comp = xp.maximum(xp.max_abs_rows(compL), xp.max_abs_rows(compU))
            e_mu = xp.maximum(xp.maximum(dr, cv), xp.maximum(xp.max_abs_rows(compL - hasL * mu[:, None]), xp.max_abs_rows(compU - hasU * mu[:, None])))
            if any_ineq:
                compI = hasI * tS * lamI
                comp = xp.maximum(comp, xp.max_abs_rows(compI))
                e_mu = xp.maximum(e_mu, xp.max_abs_rows(compI - hasI * mu[:, None]))
            mu_next = xp.where(e_mu <= o.barrier_kappa_eps * mu,
                               xp.maximum(xp.full((B,), mu_floor), xp.minimum(o.barrier_kappa_mu * mu, mu ** o.barrier_theta_mu)), mu)
            dr = xp.maximum(dr, comp)
        else:
            dr = xp.max_abs_rows(rz * free)
        exact = xp.where(cv <= o.exact_below, xp.ones((B,)), xp.zeros((B,)))
        newly = (~done) & (cv <= o.tol_constraint) & (dr <= o.tol_dual)
        iters = xp.where(newly, xp.full((B,), float(it)), iters)
        done = done | newly
        if record:
            history.append(dict(it=it, z=xp.to_numpy(z), lam=xp.to_numpy(lam), f=xp.to_numpy(f), cv=xp.to_numpy(cv),
                                dr=xp.to_numpy(dr), done=xp.to_numpy(done)))
        n_done = xp.count(done)
        if n_done == B:
            break
        if o.repack and not ip and not record and 2 * n_done >= B and B - n_done >= o.repack_min and getattr(be, "shrink", None) is not None:
            # converged problems leave the batch: their rows go to the result arrays, the rest is re-packed into a
            # smaller batch (problems are independent, every kernel and every row-wise update gives the same bits
            # for a problem wherever it sits in the batch)
            flush(done)
            keep = ~done
            be = be.shrink(keep)
            z, lam, f, g, c, sol, nneg, rz, cv, dr = (v[keep] for v in (z, lam, f, g, c, sol, nneg, rz, cv, dr))
            delta, delta_last, nu, iters, exact, lm, ids = (v[keep] for v in (delta, delta_last, nu, iters, exact, lm, ids))
            B = be.B
            done = xp.zeros_bool((B,))
            be.callbacks(z, lam, lam * exact[:, None], delta)   # same state as before on the smaller batch (J, H, factor):
            be.newton(delta)                                    # deterministic, so g, c, sol ... above stay valid
        bad = ((nneg != N_c) | ~xp.finite_rows(sol)) & ~done
        tries = 0
        first = xp.ones_bool((B,))
        while xp.any(bad) and tries < o.max_refactor:
            start = xp.where(delta_last == 0.0, xp.full((B,), o.reg_first), xp.maximum(xp.full((B,), o.reg_min), o.reg_dec * delta_last))
            grow = xp.where(delta_last == 0.0, xp.full((B,), o.reg_inc_first), xp.full((B,), o.reg_inc))
            nxt = xp.where(first, xp.maximum(start, 2.0 * delta), xp.minimum(xp.full((B,), o.reg_max), grow * delta))
            delta = xp.where(bad, nxt, delta)
            first = first & ~bad
            sol2, nneg2, _ = be.newton(delta, bad)     # only the problems in `bad` need the new factorisation
            sol = xp.where_rows(bad, sol2, sol)
            nneg = xp.where(bad, nneg2, nneg)
            bad = ((nneg != N_c) | ~xp.finite_rows(sol)) & ~done
            tries += 1
        delta_last = xp.where(delta > lm, delta, delta_last)
        dz = -sol[:, :N_z] * free
        dlam = -sol[:, N_z:]
        # ---- l1 merit line search: phi = f + nu ||c||_1. Penalty by the curvature rule (Nocedal & Wright 18.36):
        # nu >= (g'dz + max(dz'(H + delta I)dz, 0)/2) / ((1 - rho) ||c||_1), where the KKT system gives
        # dz'(H + delta I)dz = -g'dz + c'(lambda + dlam) without a product with H. (nu >= ||lambda+||_inf would
        # also give descent, but the multipliers of a swing-up far from the solution are huge and such a nu
        # makes the search follow the curved constraint manifold in tiny steps.)
        c1 = xp.sum_abs_rows(c)
        gd = xp.sum_rows(g * dz)
        curv = xp.maximum(-gd + xp.sum_rows(c * (lam + dlam)), xp.zeros((B,)))
        nu_need = (gd + 0.5 * curv) / ((1.0 - o.merit_rho) * xp.maximum(c1, xp.full((B,), 1.0e-300)))
        if o.merit_memory:
            nu = xp.where((c1 > 0.0) & (nu < nu_need), o.merit_margin * nu_need, nu)
        else:  # the penalty of THIS step only: large multipliers of early iterations do not throttle later ones
            nu = xp.maximum(xp.full((B,), o.merit_min), o.merit_margin * nu_need)
        slope = gd - nu * c1
        phi0 = f + nu * c1
        alpha = xp.ones((B,))
        if ip:
            # bound multiplier steps from the eliminated rows of the primal-dual system; fraction to the boundary
            dzL = hasL * (mu[:, None] / sL - zL - SigL * dz)
            dzU = hasU * (mu[:, None] / sU - zU + SigU * dz)
            tau = xp.maximum(xp.full((B,), o.tau_min), 1.0 - mu)[:, None]
            amax = xp.minimum(xp.min_rows(xp.where((hasL > 0) & (dz < 0.0), -tau * sL / xp.minimum(dz, xp.full((B, N_z), -1.0e-300)), xp.full((B, N_z), big))),
                              xp.min_rows(xp.where((hasU > 0) & (dz > 0.0), tau * sU / xp.maximum(dz, xp.full((B, N_z), 1.0e-300)), xp.full((B, N_z), big))))
            amax = xp.minimum(xp.ones((B,)), amax)
            a_z = xp.minimum(xp.min_rows(xp.where(dzL < 0.0, -tau * zL / xp.minimum(dzL, xp.full((B, N_z), -1.0e-300)), xp.full((B, N_z), big))),
                             xp.min_rows(xp.where(dzU < 0.0, -tau * zU / xp.minimum(dzU, xp.full((B, N_z), -1.0e-300)), xp.full((B, N_z), big))))
            a_z = xp.minimum(xp.ones((B,)), a_z)
            if any_ineq:
                dt = hasI * (mu[:, None] / lamI - tS - (tS / lamI) * dlam)       # from t lam = mu linearised (lam is the slack's multiplier)
                amax = xp.minimum(amax, xp.min_rows(xp.where((hasI > 0) & (dt < 0.0), -tau * tS / xp.minimum(dt, xp.full((B, N_c), -1.0e-300)), xp.full((B, N_c), big))))
                a_z = xp.minimum(a_z, xp.min_rows(xp.where((hasI > 0) & (dlam < 0.0), -tau * lamI / xp.minimum(dlam, xp.full((B, N_c), -1.0e-300)), xp.full((B, N_c), big))))
                # the barrier of the slacks joins the merit function's slope
                gd = gd - xp.sum_rows(hasI * (mu[:, None] / tS) * dt)
                slope = gd - nu * c1
            alpha = amax
        soc_used = xp.zeros_bool((B,))
        accepted = xp.copy_bool(done) | bad     # converged problems and failed factorisations do not move
        for ls in range(o.max_backtrack):
            if ls >= 1 and not ip and getattr(be, "backtrack", None) is not None:
                # the remaining rounds in one call (device: a replayed CUDA graph of exactly the operations below,
                # no host round trip per round; rounds after every problem was accepted change nothing)
                r = be.backtrack(z, lam, dz, dlam, nu, phi0, slope, alpha, accepted, o.armijo, o.max_backtrack - ls)
                if r is not None:
                    z, lam, alpha, accepted = r
                    break
            zt = z + alpha[:, None] * dz
            ft, ct = be.objective_constraint(zt)
            if ip:      # barrier terms of the trial point (strictly inside by the fraction-to-the-boundary rule)
                stL = xp.where(hasL > 0, xp.maximum(zt - lo, xp.full((B, N_z), 1.0e-300)), xp.ones((B, N_z)))
                stU = xp.where(hasU > 0, xp.maximum(up - zt, xp.full((B, N_z), 1.0e-300)), xp.ones((B, N_z)))
                ft = ft - mu * (xp.sum_rows(hasL * xp.log(stL)) + xp.sum_rows(hasU * xp.log(stU)))
                if any_ineq:
                    tt = xp.where(hasI > 0, xp.maximum(t + alpha[:, None] * dt, xp.full((B, N_c), 1.0e-300)), xp.ones((B, N_c)))
                    ft = ft - mu * xp.sum_rows(hasI * xp.log(tt))
                    ct = ct + hasI * tt
            phit = ft + nu * xp.sum_abs_rows(ct)
            # (interior point: Ipopt's relaxation of the test by 10 eps |phi| -- with mu -> 0 the predicted decrease of a
            # converging problem drops below the rounding error of phi itself)
            ok = (phit <= phi0 + o.armijo * alpha * slope + (2.2e-15 * abs(phi0) if ip else 0.0)) & ~accepted
            if ip and ls == 0:
                # tiny steps are taken without the test (Ipopt's tiny_step_tol idea, wider): right after mu was decreased the
                # step mostly re-centres z_L, z_U (dz ~ 1e-7), need not be a descent direction of the NEW barrier function,
                # and rejecting it would also reject the multiplier step it carries
                ok = ok | ((xp.max_abs_rows(dz) <= o.tiny_step * (1.0 + xp.max_abs_rows(z))) & ~accepted)
            z = xp.where_rows(ok, zt, z)
            if ip and any_ineq:      # inequality multipliers move with the dual step length (they must stay positive)
                lam = xp.where_rows(ok, lam + xp.where(hasI > 0, a_z[:, None] * dlam, alpha[:, None] * dlam), lam)
                t = xp.where_rows(ok, hasI * tt, t)
            else:
                lam = xp.where_rows(ok, lam + alpha[:, None] * dlam, lam)
            if ip:
                zL = xp.where_rows(ok, zL + a_z[:, None] * dzL, zL)
                zU = xp.where_rows(ok, zU + a_z[:, None] * dzU, zU)
            accepted = accepted | ok
            if xp.all(accepted):
                break
            if ls == 0 and o.soc and not ip:
                # second-order correction (Maratos effect: near the constraint manifold a long tangential step is
                # rejected because c grows quadratically along it): re-solve the same K with the constraint
                # right-hand side c(z) + c(z + dz) and try that step once before backtracking
                need = ~accepted & (xp.sum_abs_rows(ct) >= c1)
                if xp.any(need):
                    sol_s = be.newton_soc(c + ct, delta, need)
                    dzs = -sol_s[:, :N_z] * free
                    zs = z + dzs
                    fs, cs = be.objective_constraint(zs)
                    oks = (fs + nu * xp.sum_abs_rows(cs) <= phi0 + o.armijo * slope) & need & xp.finite_rows(sol_s)
                    z = xp.where_rows(oks, zs, z)
                    lam = xp.where_rows(oks, lam - sol_s[:, N_z:], lam)
                    accepted = accepted | oks
                    soc_used = soc_used | oks
                    if xp.all(accepted):
                        break
            alpha = xp.where(accepted, alpha, 0.5 * alpha)
        if o.lam_max > 0.0:
            # runaway multiplier estimates (damped steps near a rank-deficient Jacobian): start them again from zero, the
            # next Hessian of such a problem is then the objective's alone
            if ip and any_ineq:
                lam = xp.where_rows(xp.max_abs_rows(lam * (1.0 - hasI)) > o.lam_max, lam * hasI, lam)      # equality rows only
            else:
                lam = xp.where_rows(xp.max_abs_rows(lam) > o.lam_max, xp.zeros((B, N_c)), lam)
        # a problem whose search failed keeps its point; more regularisation next time shortens the step
        stuck = ~accepted
        moved = ~done & ~bad
        if ip:
            # keep z_L, z_U within [mu / (kappa s), kappa mu / s] of the new slacks (Waechter & Biegler eq. 16), then the next mu
            sLn = xp.where(hasL > 0, z - lo, xp.ones((B, N_z)))
            sUn = xp.where(hasU > 0, up - z, xp.ones((B, N_z)))
            zL = hasL * xp.maximum(xp.minimum(zL, o.kappa_sigma * mu[:, None] / sLn), mu[:, None] / (o.kappa_sigma * sLn))
            zU = hasU * xp.maximum(xp.minimum(zU, o.kappa_sigma * mu[:, None] / sUn), mu[:, None] / (o.kappa_sigma * sUn))
            if any_ineq:
                tSn = xp.where(hasI > 0, t, xp.ones((B, N_c)))
                lam = xp.where(hasI > 0, xp.maximum(xp.minimum(lam, o.kappa_sigma * mu[:, None] / tSn), mu[:, None] / (o.kappa_sigma * tSn)), lam)
            mu = xp.where(done, mu, mu_next)
            alpha = alpha / amax            # the damping rules below look at the fraction of the allowed step that was taken
        lm = xp.where(moved & (alpha < o.lm_grow_below), xp.maximum(xp.full((B,), o.lm_min), o.lm_grow * xp.maximum(lm, delta)), lm)
        lm = xp.where(moved & accepted & (alpha >= 1.0), o.lm_shrink * lm, lm)
        lm = xp.where(lm < o.lm_zero, xp.zeros((B,)), lm)
        if record:
            history[-1].update(alpha=xp.to_numpy(alpha), delta=xp.to_numpy(delta), nu=xp.to_numpy(nu), stuck=xp.to_numpy(stuck),
                               slope=xp.to_numpy(slope), soc=xp.to_numpy(soc_used))
        delta_last = xp.where(stuck | bad, xp.maximum(xp.full((B,), o.reg_first), o.reg_inc * xp.maximum(delta_last, delta)), delta_last)
    iters = xp.where(done, iters, xp.full((be.B,), float(o.max_iter)))
    flush(xp.ones_bool((be.B,)))
    return SQPResult(out["z"], out["lam"], out["iters"], out["done"], out["cv"], out["dr"], out["f"], history, backend=be)


def knot_bfgs_update(xp, blocks, s, y, free, first):
    """One damped BFGS update (Nocedal & Wright, Procedure 18.2) of M dense symmetric n x n blocks -- the knot blocks of the
    "knot-bfgs" Hessian approximation, one per (problem, knot); dto_sqp.cu `k_qn_update` is its native form.
    blocks [M, n, n]; s = z - z_prev and y = (g + J'lam) - (g_prev + J_prev'lam) (the same multipliers in both terms; bound
    multipliers left out) over the block's variables, [M, n]; free [n] or [M, n]: 0 masks pinned variables out of s and y;
    first [M] bool: the block has taken no update yet. Returns (blocks, first).
      skipped (block unchanged) when s's = 0 to 1e-30 (a problem that did not move), a quantity is not finite, or s'Bs or
      s'r is not positive; on a block's first update with s'y > 0, B is first scaled to (y'y / s'y) I;
      theta = 1 if s'y >= 0.2 s'Bs else 0.8 s'Bs / (s'Bs - s'y),  r = theta y + (1 - theta) Bs,
      B <- B - (Bs)(Bs)'/s'Bs + r r'/s'r   (so B+ s = r, and B stays symmetric positive definite)."""
    s = s * free
    y = y * free
    ss, sy, yy = xp.sum_rows(s * s), xp.sum_rows(s * y), xp.sum_rows(y * y)
    fin = lambda v: xp.finite_rows(v[:, None])  # noqa: E731
    ok = (ss > 1.0e-30) & fin(ss) & fin(sy) & fin(yy)
    M, n = int(s.shape[0]), int(s.shape[1])
    scale = ok & first & (sy > 0.0)
    sc = yy / xp.where(scale, sy, xp.ones((M,)))
    eye = xp.eye(n)
    B0 = xp.where(scale[:, None, None], sc[:, None, None] * eye[None, :, :], blocks)
    Bs = xp.sum_rows3(B0 * s[:, :, None])             # (B s)_i = sum_j B(j, i) s_j
    sBs = xp.sum_rows(s * Bs)
    low = sy < 0.2 * sBs
    theta = xp.where(low, 0.8 * sBs / xp.where(low, sBs - sy, xp.ones((M,))), xp.ones((M,)))
    r = theta[:, None] * y + (1.0 - theta)[:, None] * Bs
    sr = xp.sum_rows(s * r)
    ok = ok & fin(sBs) & fin(sr) & (sBs > 0.0) & (sr > 0.0)
    one = xp.ones((M,))
    dBs, dsr = xp.where(ok, sBs, one), xp.where(ok, sr, one)
    Bn = B0 - (Bs[:, :, None] * Bs[:, None, :]) / dBs[:, None, None] + (r[:, :, None] * r[:, None, :]) / dsr[:, None, None]
    return xp.where(ok[:, None, None], Bn, blocks), first & ~ok


def knot_elements(nlp):
    """The partitioned damped BFGS approximation ("partitioned-bfgs", dto_sqp_options.hessian_approximation = 2). Stated here
    once; dto_sqp.cu `k_pqn_update` / `k_pqn_assemble`, the KKT layer's knot chain (DTO_KKT_HESSIAN_KNOT_CHAIN) and the tests'
    twin follow it.

    The Lagrangian L = sigma f + lam'c splits into one element per knot t = 0..T-1 (0-based; sigma, lam as the solver holds them):
      t < T-1:  E_t(x_t, u_t, x_{t+1}) = sigma cost_t(x_t, u_t) + lam_{S,t}' stage_t(x_t, u_t) + lam_{D,t}' d_t(x_{t+1}, x_t, u_t)
      t = T-1:  E_t(x_T) = sigma cost_T(x_T) + lam_{S,T}' stage_T(x_T)
    Element t's variables v_t = [x_t; u_t; x_{t+1}] are one contiguous range z[v0_t, v0_t + m_t), m_t = n_t + nx_{t+1}
    (n_t = nx_t + nu_t; the last knot: m = n = nx_T). Without a general constraint sum_t E_t = L, so the Hessian of L is
    sum_t P_t' (Hessian of E_t) P_t. Each element keeps a dense symmetric m_t x m_t block B_t (the identity at the start of
    every solve and continuation stage); after the callbacks of every iteration (where "knot-bfgs" updates its blocks)
      s_t = P_t (z - z_prev), pinned variables masked;
      y_t = grad_{v_t} E_t(z) - grad_{v_t} E_t(z_prev), both with the multipliers as they stand (bound multipliers left out):
            on [x_t; u_t] g (only cost_t touches them in the objective) + the J'lam terms of the rows of d_t and stage_t,
            on x_{t+1} the J'lam terms of the rows of d_t only (`element_gradients`);
    and B_t takes exactly the update `knot_bfgs_update` states (first update scaled, Powell damping, the same skips).
    H of K is sum_t P_t' B_t P_t, kept as the knot chain: row block t = B_t[0:n_t, :] plus, on its x_t x x_t corner, the
    x_t x x_t tail of B_{t-1}, added in that order (`chain_from_elements`).

    Returns [(v0, n, m, rows)] per knot: 0-based first variable, n_t, m_t, and the constraint rows of d_t and stage_t (0-based,
    ascending; the rows of J that element t owns). A shape with a general constraint has none: ValueError."""
    import numpy as np
    if getattr(nlp, "use_general", False):
        raise ValueError("partitioned BFGS: a general constraint couples distant knots; no knot element owns its curvature")
    xs, nx, _, nu = nlp.knot_layout()
    T = int(nlp.T)
    jr, jc = (np.asarray(v) - 1 for v in nlp.jacobian_structure_arrays())
    n_dyn = int(sum(int(nx[t + 1]) for t in range(T - 1)))      # d_t has nx_{t+1} rows; all dynamics rows come first
    out, r0 = [], 0
    for t in range(T):
        v0, n = int(xs[t]) - 1, int(nx[t] + nu[t])
        m = n + (int(nx[t + 1]) if t + 1 < T else 0)
        dyn = list(range(r0, r0 + (m - n)))
        r0 += m - n
        stage = np.unique(jr[(jr >= n_dyn) & (jc >= v0) & (jc < v0 + n)]).tolist()
        out.append((v0, n, m, np.array(dyn + stage, dtype=np.int64)))
    return out


def element_gradients(elements, g, Jd, lam):
    """numpy: grad_{v_t} E_t of every element (`knot_elements`), [B, m_t] each, from g [B, N_z], the dense Jacobian Jd
    [B, N_c, N_z] and lam [B, N_c]"""
    import numpy as np
    out = []
    for v0, n, m, rows in elements:
        gr = np.einsum("brj,br->bj", Jd[:, rows, v0:v0 + m], lam[:, rows])
        gr[:, :n] += g[:, v0:v0 + n]
        out.append(gr)
    return out


def chain_from_elements(elements, blocks):
    """numpy: the knot chain [B, nnz_chain] (nlp.hessian_chain_structure() order) from the element blocks [B, m_t, m_t]"""
    import numpy as np
    rows = []
    for t, (v0, n, m, _) in enumerate(elements):
        top = blocks[t][:, :n, :].copy()
        if t > 0:
            npv = elements[t - 1][1]                        # B_{t-1}'s tail: its x_t x x_t corner
            k = elements[t - 1][2] - npv
            top[:, :k, :k] = top[:, :k, :k] + blocks[t - 1][:, npv:, npv:]
        rows.append(top.reshape(top.shape[0], -1))
    return np.concatenate(rows, axis=1)


def bound_arrays(lo, up, options: Optional[SQPOptions] = None, clo=None, cup=None, scale: float = 1.0):
    """numpy: primal_bounds (src/data.jl:123-133) -> what `solve` needs. Returns (fixed, bounds): `fixed` = variables pinned
    by lo == up; `bounds` = None when no other finite bound exists, else dict(hasL, hasU, lo, up, pushL, pushU) with 0/1
    masks, finite values (0 where absent) and the distances the starting point is pushed inside (Ipopt's bound_push/frac).
    lo, up may be [N_z] (every problem) or [B, N_z] (row b = problem b's values): `fixed`, hasL and hasU are then still [N_z]
    -- one bound pattern per batch, checked to be common to all rows (ValueError otherwise) -- and lo, up, pushL, pushU are
    [B, N_z], each row computed by the same elementwise operations as the [N_z] case (the same values, bit for bit)."""
    import numpy as np
    o = options or SQPOptions()
    lo, up = np.asarray(lo, float), np.asarray(up, float)
    rows = lo.ndim == 2
    if rows:
        bad = np.isnan(lo) | np.isnan(up) | (np.isfinite(lo) & np.isfinite(up) & (lo > up))
        if bad.any():
            p, i = (int(v[0]) for v in np.nonzero(bad))
            raise ValueError(f"problem {p}, variable index {i}: bounds [{lo[p, i]}, {up[p, i]}]")
        fx = np.isfinite(lo) & (lo == up)
        for name, pat in (("pinned", fx), ("lower-bounded", np.isfinite(lo) & ~fx), ("upper-bounded", np.isfinite(up) & ~fx)):
            diff = pat != pat[:1]
            if diff.any():
                p, i = (int(v[0]) for v in np.nonzero(diff))
                raise ValueError(f"problem {p}, variable index {i}: bounds [{lo[p, i]}, {up[p, i]}] differ from problem 0's "
                                 f"[{lo[0, i]}, {up[0, i]}] in which variables are {name}: a batch has one bound pattern")
    fixed = np.isfinite(lo) & (lo == up)
    if scale != 1.0:        # continuation stage: two-sided bounds widened about their midpoint (one-sided and pinned ones stay)
        two = np.isfinite(lo) & np.isfinite(up) & ~fixed
        l2, u2 = np.where(two, lo, 0.0), np.where(two, up, 0.0)
        mid, half = 0.5 * (l2 + u2), 0.5 * (u2 - l2)
        lo = np.where(two, mid - scale * half, lo)
        up = np.where(two, mid + scale * half, up)
    hasL = np.isfinite(lo) & ~fixed
    hasU = np.isfinite(up) & ~fixed
    # inequality rows c_i(z) <= 0: constraint_bounds (src/data.jl:135-148) gives them (-Inf, 0], equalities [0, 0]
    hasI = np.zeros(0, dtype=bool) if clo is None else (np.asarray(clo, float) != np.asarray(cup, float))
    if hasI.any() and not (np.all(np.isneginf(np.asarray(clo, float)[hasI])) and np.all(np.asarray(cup, float)[hasI] == 0.0)):
        raise NotImplementedError("sqp: inequality rows other than c(z) <= 0 are outside this solver's scope")
    if not (hasL.any() or hasU.any() or hasI.any()):
        return (fixed[0] if rows else fixed), None
    if np.any((hasL & hasU) & (lo >= up)):
        raise ValueError("a variable's lower bound exceeds its upper bound")
    l0, u0 = np.where(hasL, lo, 0.0), np.where(hasU, up, 0.0)
    width = np.where(hasL & hasU, u0 - l0, np.inf)
    pushL = np.where(hasL, np.minimum(o.bound_push * np.maximum(1.0, np.abs(l0)), o.bound_frac * width), 0.0)
    pushU = np.where(hasU, np.minimum(o.bound_push * np.maximum(1.0, np.abs(u0)), o.bound_frac * width), 0.0)
    if rows:        # the pattern is the batch's (checked above): one mask per variable
        fixed, hasL, hasU = fixed[0], hasL[0], hasU[0]
    return fixed, dict(hasL=hasL.astype(np.float64), hasU=hasU.astype(np.float64), lo=l0, up=u0, pushL=pushL, pushU=pushU,
                       hasI=hasI.astype(np.float64))


def solve_bounded(be, z0, lam0=None, options: Optional[SQPOptions] = None, record: bool = False) -> SQPResult:
    """`solve`, plus a fallback for problems with inequality bounds that the direct solve leaves unconverged (no restoration
    phase: an iterate can run into its bounds while the constraints are still violated): the two-sided bounds are widened
    about their midpoint by options.bound_relax, the problem is solved from the ORIGINAL guess, and then the true bounds are
    solved warm-started from there. A problem
    keeps its direct result when that converged; otherwise it takes the staged one. Problems stay independent: what a
    problem gets depends only on its own guess and the fixed stage list. The backend must offer set_bound_scale(scale)."""
    o = options or SQPOptions()
    xp = be.xp
    res = solve(be, z0, lam0, o, record)
    if getattr(be, "bounds", None) is None or getattr(be, "set_bound_scale", None) is None or o.bound_relax <= 1.0 or xp.all(res.converged):
        return res
    z, lam, its = z0, lam0, None
    stages = (float(o.bound_relax), 1.0)      # the last stage is the true problem
    try:
        for scale in stages:
            be.set_bound_scale(float(scale))
            stage = solve(be, z, lam, o, False)
            z, lam = stage.z, stage.lam
            its = stage.iterations if its is None else its + stage.iterations
    finally:
        be.set_bound_scale(1.0)
    take = stage.converged & ~res.converged
    res.z = xp.where_rows(take, stage.z, res.z)
    res.lam = xp.where_rows(take, stage.lam, res.lam)
    for name in ("constraint_violation", "dual_residual", "objective"):
        setattr(res, name, xp.where(take, getattr(stage, name), getattr(res, name)))
    res.iterations = xp.where(take, res.iterations + its, res.iterations)      # direct attempt + all stages
    res.converged = res.converged | take
    res.staged = take
    return res


# --------------------------------------------------------------------------------------- array namespaces
class _XP:
    """The handful of batched array operations the algorithm uses, for torch (device) and numpy."""

    def __init__(self, mod, device=None):
        self.m = mod
        self.device = device
        self.is_torch = mod.__name__ == "torch"

    def _kw(self):
        return dict(dtype=self.m.float64, device=self.device) if self.is_torch else dict(dtype=self.m.float64)

    def zeros(self, shape):
        return self.m.zeros(shape, **self._kw())

    def ones(self, shape):
        return self.m.ones(shape, **self._kw())

    def full(self, shape, v):
        return self.m.full(shape, float(v), **self._kw())

    def zeros_bool(self, shape):
        return self.m.zeros(shape, dtype=self.m.bool, device=self.device) if self.is_torch else self.m.zeros(shape, dtype=bool)

    def ones_bool(self, shape):
        return ~self.zeros_bool(shape)

    def copy(self, a):
        return a.clone() if self.is_torch else a.copy()

    copy_bool = copy

    def where(self, c, a, b):
        return self.m.where(c, a, b)

    def where_rows(self, c, a, b):
        return self.m.where(c[:, None], a, b)

    def maximum(self, a, b):
        return self.m.maximum(a, b)

    def minimum(self, a, b):
        return self.m.minimum(a, b)

    def max_abs_rows(self, a):
        if a.shape[1] == 0:
            return self.zeros((a.shape[0],))
        return a.abs().amax(dim=1) if self.is_torch else self.m.abs(a).max(axis=1)

    def sum_abs_rows(self, a):
        return a.abs().sum(dim=1) if self.is_torch else self.m.abs(a).sum(axis=1)

    def sum_rows(self, a):
        return a.sum(dim=1) if self.is_torch else a.sum(axis=1)

    def hcat(self, a, b):
        return self.m.cat([a, b], dim=1) if self.is_torch else self.m.concatenate([a, b], axis=1)

    def min_rows(self, a):
        return a.amin(dim=1) if self.is_torch else a.min(axis=1)

    def log(self, a):
        return self.m.log(a)

    def finite_rows(self, a):
        return self.m.isfinite(a).all(dim=1) if self.is_torch else self.m.isfinite(a).all(axis=1)

    def arange(self, n):
        return self.m.arange(n, device=self.device) if self.is_torch else self.m.arange(n)

    def count(self, a):
        return int(a.sum())

    def all(self, a):
        return bool(a.all())

    def any(self, a):
        return bool(a.any())

    def to_numpy(self, a):
        return a.detach().cpu().numpy().copy() if self.is_torch else self.m.array(a, copy=True)

    def eye(self, n):
        return self.m.eye(n, **self._kw())

    def sum_rows3(self, a):
        """[M, j, i] -> [M, i]: sum over j"""
        return a.sum(dim=1) if self.is_torch else a.sum(axis=1)


# --------------------------------------------------------------------------------------- device backend
class _CudaArray:
    """zero-copy view of a device buffer of libdto.so for torch (CUDA array interface)"""

    def __init__(self, ptr: int, shape, typestr="<f8"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}


class DeviceBackend:
    """The product arm: callbacks and KKT solves are this package's CUDA kernels on the batch's device arrays;
    torch provides the views of those arrays and the O(B N) vector glue. One shard (one device) per backend:
    multi-GPU runs use one backend per rank / per shard, problems are independent."""

    def __init__(self, nlp, dual_reg: float = 1.0e-9, options: Optional[SQPOptions] = None):
        import torch

        from . import _lib
        from .evaluator import A_C, A_F, A_G, A_LAMBDA, A_SIGMA, A_Z, K_CONSTRAINT, K_OBJECTIVE
        from .kkt import KKTSystem
        if nlp.num_shards != 1:
            raise ValueError("DeviceBackend drives one shard; create one batch per device")
        if options is not None and options.hessian_approximation != "exact":
            raise ValueError(f"hessian_approximation={options.hessian_approximation!r} is a mode of the native solver (method='native')")
        self.nlp = nlp
        self.torch = torch
        dev = torch.device("cuda", nlp.shard_device(0))
        self.xp = _XP(torch, dev)
        self.B, self.N_z, self.N_c = nlp.batch, nlp.num_variables, nlp.num_constraint
        lo, up = nlp.batch_variable_bounds       # [N_z] each, or [B, N_z]: every problem's values (one pattern)
        import numpy as np
        clo, cup = nlp.constraint_bounds
        # Bound(state_lower = x1, state_upper = x1): pinned variables; any other finite bound: interior point in `solve`
        fixed, bounds = bound_arrays(lo, up, options, clo, cup)       # (inequality rows c(z) <= 0: slacks in `solve`)
        self._bound_args = (lo, up, options, clo, cup)
        self.bounds = None if bounds is None else {k: torch.as_tensor(v, device=dev) for k, v in bounds.items()}
        self.free = torch.as_tensor((~fixed).astype(np.float64), device=dev)
        self.pinned_value = torch.as_tensor(np.where(fixed, lo, 0.0), device=dev)
        self._fixed = fixed
        self._dual_reg = dual_reg
        self._owned_nlp = None      # a batch created by shrink() (closed with this backend)
        self._launches_before = 0
        self.kkt = KKTSystem(nlp, 0.0, dual_reg)
        if fixed.any():
            self.kkt.set_fixed(fixed)                   # identity rows/columns in K, zero right-hand side: their step is 0
        self._K = (K_OBJECTIVE, K_CONSTRAINT)
        view = lambda arr, shape: torch.as_tensor(_CudaArray(nlp.device_pointer(arr, 0), shape), device=dev)  # noqa: E731
        B = self.B
        self.d_z = view(A_Z, (B, self.N_z))
        self.d_lam = view(A_LAMBDA, (B, self.N_c))
        self.d_sigma = view(A_SIGMA, (B,))
        self.d_f = view(A_F, (B,))
        self.d_g = view(A_G, (B, self.N_z))
        self.d_c = view(A_C, (B, self.N_c))
        kview = lambda which, shape, ts="<f8": torch.as_tensor(_CudaArray(self.kkt.device_pointer(which, 0), shape, ts), device=dev)  # noqa: E731
        self.d_rhs = kview(0, (B, self.kkt.dim))
        self.d_sol = kview(1, (B, self.kkt.dim))
        self.d_reg = kview(3, (B,))
        self.d_nneg = kview(4, (B,), "<i4")
        self.d_diag = kview(5, (B, self.kkt.dim)) if self.bounds is not None else None   # barrier diagonal added to K
        self.d_sigma.fill_(1.0)
        # ONE stream for the kernels of libdto.so and torch's glue operations: the batch launches on torch's
        # current stream of the device, so every copy / update is ordered with the kernels without events
        self.stream = torch.cuda.current_stream(dev)
        nlp.set_stream(self.stream.cuda_stream, 0)
        self.launches0 = nlp.launch_count()
        self._graph = None          # (CUDAGraph, static buffers, armijo) of one backtracking round; False = capture unavailable

    def set_bound_scale(self, scale: float):
        """continuation stage of `solve_bounded`: two-sided bounds widened about their midpoint by `scale` (1 = the true ones)"""
        if self.bounds is not None:
            _, bounds = bound_arrays(*self._bound_args, scale=scale)
            self.bounds = {k: self.torch.as_tensor(v, device=self.xp.device) for k, v in bounds.items()}

    def close(self):
        self.kkt.close()
        if self._owned_nlp is not None:
            self._owned_nlp.close()
            self._owned_nlp = None

    def total_launches(self) -> int:
        return self._launches_before + self.nlp.launch_count() - self.launches0

    def shrink(self, keep):
        """A backend over the problems of the boolean mask `keep` only: a new, smaller batch of the same shape (static
        tables and model library are shared), per-problem parameters copied device to device."""
        from .evaluator import A_W
        t = self.torch
        idx = keep.nonzero().flatten()
        n = int(idx.numel())
        nlp2 = self.nlp.new_batch(batch=n)
        rows = self.nlp._bounds_host
        if rows is not None:
            sel = idx.cpu().numpy()
            nlp2.set_variable_bounds(rows[0][sel], rows[1][sel])
        dev = self.xp.device
        if self.nlp.num_parameter:
            nw = self.nlp.num_parameter
            src = t.as_tensor(_CudaArray(self.nlp.device_pointer(A_W, 0), (self.B, nw)), device=dev)
            dst = t.as_tensor(_CudaArray(nlp2.device_pointer(A_W, 0), (n, nw)), device=dev)
            dst.copy_(src[idx])
            t.cuda.current_stream(dev).synchronize()
        be2 = DeviceBackend(nlp2, dual_reg=self._dual_reg)
        be2._owned_nlp = nlp2
        be2._launches_before = self.total_launches()
        self.close()
        return be2

    def callbacks(self, z, lam, lam_hess, delta, diag=None, gshift=None, cshift=None):
        """f, g, c at z; J and H(z, lam_hess) stay on the device; first KKT solve with the damping `delta` and the
        right-hand side of the TRUE multipliers `lam` (the Hessian may use others: Gauss-Newton for far-away problems).
        Interior point: `diag` [B, N_z] joins the diagonal of H inside the factor kernel, `gshift` is added to g (the
        barrier's gradient) before the right-hand side is formed; the g returned includes it."""
        t = self.torch
        with t.cuda.stream(self.stream):
            self.d_z.copy_(z)
            self.d_lam.copy_(lam_hess)
            self.d_reg.copy_(delta)
            self.nlp.launch(self._K[0])                 # f
            self.kkt.launch(2)                          # g, c, J, H(z, lam_hess)
            c_raw = None
            if diag is not None:
                if diag.shape[1] == self.N_z:                       # bounds on variables only: the constraint rows keep -dual_reg
                    self.d_diag[:, :self.N_z].copy_(diag)
                else:
                    self.d_diag.copy_(diag)
                self.d_g.add_(gshift)
                if cshift is not None:                              # inequality rows: right-hand side c + mu / lam
                    c_raw = self.d_c.clone()
                    self.d_c.add_(cshift)
            self.d_lam.copy_(lam)
            self.kkt.launch(0)                          # h = [g + J'lam; c], K = L D L', sol
            self._fresh = True
            return self.d_f.clone(), self.d_g.clone(), (self.d_c.clone() if c_raw is None else c_raw)

    def _solution(self):
        t = self.torch
        return self.d_sol.clone(), self.d_nneg.to(t.float64), self.d_rhs[:, :self.N_z].clone()

    def pin(self, z):
        """pinned variables take their bound value (Ipopt: fixed variables are removed from the problem)"""
        return z * self.free + self.pinned_value

    def _relaunch(self, mask):
        """linear algebra again: for every problem, or (lock step would otherwise make one bad problem re-factor the
        whole batch) only for the problems of `mask` -- dto_kkt_launch_subset; the others keep their solution"""
        if mask is None:
            self.kkt.launch(0)
            return
        self._idx = mask.nonzero().flatten().to(self.torch.int32)      # (kept alive until the next launch)
        n = int(self._idx.numel())
        if n * 2 >= self.B:
            self.kkt.launch(0)
        elif n > 0:
            self.kkt.launch_subset(self._idx.data_ptr(), n)

    def newton(self, delta, mask=None):
        with self.torch.cuda.stream(self.stream):
            if not self._fresh:                         # re-factor with the new per-problem regularisation
                self.d_reg.copy_(delta)
                self._relaunch(mask)
            self._fresh = False
            return self._solution()

    def newton_soc(self, c_soc, delta, mask=None):
        """second-order correction: same K, constraint right-hand side c_soc (the device c is overwritten: the
        iteration's own copy lives in the solver). K is already factorised: dto_kkt_resolve runs the forward and
        backward solves only (bit-identical to factorising again)"""
        with self.torch.cuda.stream(self.stream):
            self.d_c.copy_(c_soc)
            if mask is None:
                self.kkt.resolve()
            else:
                self._idx = mask.nonzero().flatten().to(self.torch.int32)
                n = int(self._idx.numel())
                if n * 2 >= self.B:
                    self.kkt.resolve()
                elif n > 0:
                    self.kkt.resolve(self._idx.data_ptr(), n)
            self._fresh = False
            return self.d_sol.clone()

    def objective_constraint(self, z):
        t = self.torch
        with t.cuda.stream(self.stream):
            self.d_z.copy_(z)
            self.nlp.launch(self._K[0])
            self.nlp.launch(self._K[1])
            return self.d_f.clone(), self.d_c.clone()

    # ---- backtracking rounds as one replayed CUDA graph -------------------------------------------------------
    def _round(self, S, armijo):
        """One backtracking round on the static buffers S: the very statements of the loop in `solve`."""
        t = self.torch
        t.add(S["z"], S["alpha"][:, None] * S["dz"], out=self.d_z)       # zt = z + alpha dz, straight into the device z
        self.nlp.launch(self._K[0])
        self.nlp.launch(self._K[1])
        phit = self.d_f + S["nu"] * self.d_c.abs().sum(dim=1)
        ok = (phit <= S["phi0"] + armijo * S["alpha"] * S["slope"]) & ~S["accepted"]
        S["z"].copy_(t.where(ok[:, None], self.d_z, S["z"]))
        S["lam"].copy_(t.where(ok[:, None], S["lam"] + S["alpha"][:, None] * S["dlam"], S["lam"]))
        S["accepted"].logical_or_(ok)
        S["alpha"].copy_(t.where(S["accepted"], S["alpha"], 0.5 * S["alpha"]))

    def _capture(self, armijo):
        t = self.torch
        dev = self.xp.device
        f64 = dict(dtype=t.float64, device=dev)
        S = {"z": t.zeros((self.B, self.N_z), **f64), "dz": t.zeros((self.B, self.N_z), **f64), "lam": t.zeros((self.B, self.N_c), **f64),
             "dlam": t.zeros((self.B, self.N_c), **f64), "nu": t.ones((self.B,), **f64), "phi0": t.zeros((self.B,), **f64),
             "slope": t.zeros((self.B,), **f64), "alpha": t.ones((self.B,), **f64), "accepted": t.ones((self.B,), dtype=t.bool, device=dev)}
        side = t.cuda.Stream(device=dev)
        side.wait_stream(self.stream)
        self.nlp.set_stream(side.cuda_stream, 0)
        try:
            with t.cuda.stream(side):
                for _ in range(2):                       # warm-up outside the capture (lazy allocations, plan tables)
                    self._round(S, armijo)
            side.synchronize()
            g = t.cuda.CUDAGraph()
            with t.cuda.graph(g, stream=side):
                self._round(S, armijo)
        finally:
            self.nlp.set_stream(self.stream.cuda_stream, 0)
        self.stream.wait_stream(side)
        return g, S

    def backtrack(self, z, lam, dz, dlam, nu, phi0, slope, alpha, accepted, armijo, rounds):
        if self._graph is False:
            return None
        try:
            if self._graph is None or self._graph[2] != armijo:
                g, S = self._capture(armijo)
                self._graph = (g, S, armijo)
        except Exception as e:  # noqa: BLE001 - e.g. a driver that cannot capture: the eager loop of `solve` runs instead
            import warnings
            warnings.warn(f"sqp: CUDA-graph capture of the backtracking round failed ({e}); using the eager loop")
            self._graph = False
            self.backtrack = None
            return None
        g, S, _ = self._graph
        for k, v in (("z", z), ("lam", lam), ("dz", dz), ("dlam", dlam), ("nu", nu), ("phi0", phi0), ("slope", slope), ("alpha", alpha),
                     ("accepted", accepted)):
            S[k].copy_(v)
        for _ in range(rounds):
            g.replay()
        return S["z"].clone(), S["lam"].clone(), S["alpha"].clone(), S["accepted"].clone()


# --------------------------------------------------------------------------------------- native arm
def solve_native(nlp, z0, lam0=None, options: Optional[SQPOptions] = None) -> SQPResult:
    """The same algorithm as `solve`, run by libdto.so itself (dto_sqp_solve, csrc/dto_sqp_host.inc + dto_sqp.cu): the
    vector glue that `solve` leaves to torch is a handful of warp-per-problem kernels, and the host reads back eight
    counters per decision instead of launching ~100 small torch operations per iteration. This is what a Julia caller
    reaches through `ccall` (julia/DTOB200.jl `solve!`); no torch is involved. numpy in, numpy out."""
    import ctypes as C

    import numpy as np

    from . import _lib
    o = options or SQPOptions()
    if o.merit_memory:
        raise NotImplementedError("solve_native: merit_memory is an experiment of the python arm only")
    L = _lib.lib()
    co = _lib.SqpOptions()
    L.dto_sqp_default_options(C.byref(co))
    if o.hessian_approximation not in HessianApproximation.CODES:
        raise ValueError(f"hessian_approximation={o.hessian_approximation!r}: expected one of {sorted(HessianApproximation.CODES)}")
    for name, _ in _lib.SqpOptions._fields_:
        v = HessianApproximation.CODES[o.hessian_approximation] if name == "hessian_approximation" else getattr(o, name)
        setattr(co, name, type(getattr(co, name))(v))
    B, N_z, N_c = nlp.batch, nlp.num_variables, nlp.num_constraint
    z0 = np.ascontiguousarray(z0, dtype=np.float64)
    if z0.shape != (B, N_z):
        raise ValueError(f"z0 has shape {z0.shape}, expected {(B, N_z)}")
    if lam0 is not None:
        lam0 = np.ascontiguousarray(lam0, dtype=np.float64)
        if lam0.shape != (B, N_c):
            raise ValueError(f"lam0 has shape {lam0.shape}, expected {(B, N_c)}")
    lo, up = (np.ascontiguousarray(v, dtype=np.float64) for v in nlp.batch_variable_bounds)
    stride = N_z if lo.ndim == 2 else 0         # [B, N_z]: one row per problem (dto_sqp_solve_ex); [N_z]: shared by all
    z, lam = np.empty((B, N_z)), np.empty((B, N_c))
    iters, done = np.empty(B, np.int32), np.empty(B, np.uint8)
    cv, dr, f = np.empty(B), np.empty(B), np.empty(B)
    stats = np.zeros(16, np.int64)
    ptr = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    _lib.check(L.dto_sqp_solve_ex(nlp.handle, C.byref(co), ptr(z0), ptr(lam0), ptr(lo), ptr(up), stride, ptr(z), ptr(lam), ptr(iters),
                                  ptr(done), ptr(cv), ptr(dr), ptr(f), ptr(stats)))
    res = SQPResult(z, lam, iters.astype(np.float64), done.astype(bool), cv, dr, f, [])
    res.staged = done == 2          # converged by the bound continuation (see solve_bounded)
    res.stats = dict(iterations=int(stats[0]), launches=int(stats[1]), factorisations=int(stats[2]), syncs=int(stats[3]),
                     refactorisations=int(stats[4]), corrections=int(stats[5]), search_rounds=int(stats[6]), multi_trial_passes=int(stats[7]),
                     phase_ms=dict(callbacks_first_factor=stats[8] / 1e3, inertia_correction=stats[9] / 1e3, line_search=stats[10] / 1e3,
                                   of_which_corrections=stats[11] / 1e3, setup=stats[12] / 1e3, loop=stats[13] / 1e3,
                                   results=stats[14] / 1e3))
    return res


def solve_native_sharded(nlp, z0, lam0=None, options: Optional[SQPOptions] = None) -> SQPResult:
    """`solve_native` for a batch spread over several devices (row (e): problems are independent, contiguous shards, no
    collective): dto_sqp_solve drives ONE device, so every shard gets its own one-device batch of the same shape (model library
    and static tables shared, its slice of the per-problem parameters and bounds), the solves run side by side from one host thread each
    (ctypes releases the GIL for the duration of the C call), and the results are put back in the caller's order; the final
    iterate also becomes the resident z of the original batch (get_trajectory)."""
    import threading

    import numpy as np
    B = nlp.batch
    z0 = np.ascontiguousarray(z0, dtype=np.float64)
    parts = [(nlp.shard_device(i),) + tuple(int(v) for v in nlp.shard_range(i)) for i in range(nlp.num_shards)]
    w = getattr(nlp, "_w_host", None)
    if nlp.num_parameter and w is None:
        raise RuntimeError("solve_native_sharded: the per-problem parameters were not set through set_parameters")
    rows = getattr(nlp, "_bounds_host", None)
    results, errors = [None] * len(parts), []

    def work(k, device, begin, size):
        sub = None
        try:
            if size == 0:
                return
            sub = nlp.new_batch(batch=size, devices=[device])
            if nlp.num_parameter:
                sub.set_parameters(w[begin:begin + size])
            if rows is not None:
                sub.set_variable_bounds(rows[0][begin:begin + size], rows[1][begin:begin + size])
            results[k] = solve_native(sub, z0[begin:begin + size], None if lam0 is None else lam0[begin:begin + size], options)
        except Exception as e:  # noqa: BLE001 - re-raised in the caller's thread
            errors.append(e)
        finally:
            if sub is not None:
                sub.close()

    threads = [threading.Thread(target=work, args=(k,) + p) for k, p in enumerate(parts)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    done = [r for r in results if r is not None]
    cat = lambda name: np.concatenate([getattr(r, name) for r in done])  # noqa: E731
    res = SQPResult(cat("z"), cat("lam"), cat("iterations"), cat("converged"), cat("constraint_violation"), cat("dual_residual"), cat("objective"), [])
    res.staged = cat("staged")
    res.stats = {k: (max if k == "iterations" else sum)(r.stats[k] for r in done) for k in done[0].stats if k != "phase_ms"}
    res.stats["devices"] = [p[0] for p in parts]
    assert res.z.shape[0] == B
    nlp.set_x(res.z)
    return res

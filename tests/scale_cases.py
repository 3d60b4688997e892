"""TEST INFRASTRUCTURE: the native solver's walks through the oracle twin at the sizes it ships at (tests/test_sqp_scale_gpu.py),
and the branches each walk claims to reach, checked on the twin alone (tests/test_sqp_scale_cpu.py).

Every case builds the product batch (host side only until it is solved), its starting point and the twin: `sqp.solve` driven
by the oracle's C twin (per-problem parameters where the model has them) and the banded LDL' of the product's ordering
vectorised over the batch (`linear="band-batched"`). Rows pass 128 entries in every case, so the warp-per-problem kernels of
dto_sqp.cu take a second and later trip over N_z and N_c.

  a  pendulum T = 101, exact Hessian, B = 37 (ten CTAs of four problems, the last one partial); the even problems (19) start
     at a converged solution, so from the first check fewer than half are open: the first factorisation runs over `alist`
     and converged problems sit between open ones inside CTAs
  b  band model (15, 2, 14, False) at T = 10, B = 21: 32-lane KKT rows (half bandwidth 30), an indefinite reduced Hessian,
     inertia corrections with the full ladder of four candidates per problem
  c  cartpole T = 41 with per-problem parameters w = [x1; xT] and no control bounds (equality mode), B = 33: second-order
     corrections and one-pass searches over trial slots, whose objective and constraints see each problem's own w
  d  interior point over long rows: pendulum T = 101 with |u| <= 15 (bounds only) and car T = 41 with an obstacle row per knot
  e  knot-block and partitioned BFGS on the pendulum T = 101 built without Hessians, B = 9
  f  acrobot T = 101, the shipped shape, B = 8, for 15 iterations: far from the solution the swing-up's KKT matrices are badly
     conditioned, and the native iterate leaves the twin's gradually (1e-10 relative after one iteration, 8e-9 after 14, 2e-7
     after 15, measured on a B200) with every decision the same: a flipped step length or regularisation would move z by
     alpha |dz|, orders of magnitude more. The walk stops where the shared tolerance of 1e-7 still holds.
"""
from __future__ import annotations

import numpy as np

import dto_b200 as D
from dto_b200 import kkt as PK
from dto_b200 import sqp
from examples import models as M
from oracle import api as O
from oracle import cgen

from band_models import band_kwargs, build_band
from sqp_oracle import OracleBackend
from test_sqp_pqn_cpu import PQNOracleBackend
from test_sqp_qn_cpu import QNOracleBackend

DUAL_REG = 1.0e-6

# name: (builder, kwargs, B, twin max_iter, Hessian mode)
CASES = {
    "a_pendulum_alist": ("pendulum", dict(T=101), 37, 40, "exact"),
    "b_band_ladder": ("band", dict(band_kwargs((15, 2, 14, False), T=10)), 21, 30, "exact"),
    "c_cartpole_w": ("cartpole", dict(T=41, u_bnd=None), 33, 40, "exact"),
    "d_pendulum_bounds": ("pendulum", dict(T=101, u_bnd=15.0), 9, 40, "exact"),
    "d_car_obstacle": ("car", dict(T=41, obstacle="stage"), 9, 30, "exact"),
    "e_pendulum_knot_bfgs": ("pendulum", dict(T=101, evaluate_hessian=False), 9, 30, "knot-bfgs"),
    "e_pendulum_partitioned_bfgs": ("pendulum", dict(T=101, evaluate_hessian=False), 9, 30, "partitioned-bfgs"),
    "f_acrobot": ("acrobot", dict(T=101), 8, 15, "exact"),
}
# iterations the twin runs in each case (len(history)): pinned, so that no case can shrink without notice
ITERATIONS = {"a_pendulum_alist": 37, "b_band_ladder": 20, "c_cartpole_w": 16, "d_pendulum_bounds": 40, "d_car_obstacle": 30,
              "e_pendulum_knot_bfgs": 30, "e_pendulum_partitioned_bfgs": 30, "f_acrobot": 15}


def _models(name, kw):
    if name == "band":
        return build_band(O, **kw), build_band(D, **kw)
    return M.BUILDERS[name](O, **kw), M.BUILDERS[name](D, **kw)


def _guess(model, B, seed, state_noise=0.0, ends=None):
    """states interpolated between the end points (each problem's own with `ends` = (x1 [B, n], xT [B, n])), random controls"""
    T, n, m = model["T"], model["n"], model["m"]
    rng = np.random.default_rng(seed)
    x1 = np.tile(model["x1"], (B, 1)) if ends is None else ends[0]
    xT = np.tile(model["xT"], (B, 1)) if ends is None else ends[1]
    z = np.zeros((B, T * n + (T - 1) * m))
    for t in range(T):
        o = t * (n + m)
        z[:, o:o + n] = x1 + (xT - x1) * t / (T - 1) + state_noise * rng.normal(size=(B, n))
        if t < T - 1:
            z[:, o + n:o + n + m] = rng.normal(size=(B, m))
    return z


class Case:
    """one walk: the product batch `pn` (parameters set), the start (z0, lam0), the twin's backend `be` and result `ref`
    (history recorded), and `native(k)`: the options that stop dto_sqp_solve after k iterations"""

    def __init__(self, key):
        name, kw, B, iters, mode = CASES[key]
        self.key, self.B, self.mode = key, B, mode
        mo, mp = _models(name, kw)
        osolver = O.solver_from(mo)
        self.pn = pn = D.solver_from(mp, batch=B).nlp
        self.N_z, self.N_c = pn.num_variables, pn.num_constraint
        self.opts = sqp.SQPOptions(max_iter=iters, dual_reg=DUAL_REG)
        w = None
        self.lam0 = None
        self._params_set = False
        if name == "cartpole":
            # w = [x1; xT] per problem around the swing-up's end points (as tests/util.make_inputs draws them)
            rng = np.random.default_rng(31)
            w = np.zeros((B, 8))
            w[:, 0:4] = rng.normal(0.0, 0.1, (B, 4))
            w[:, 4:8] = mp["xT"] + rng.normal(0.0, 0.1, (B, 4))
            osolver.set_parameters([np.zeros(8) for _ in range(mp["T"])] + [np.zeros(0)])
            self.z0 = _guess(mp, B, 32, ends=(w[:, 0:4], w[:, 4:8]))
        elif name == "band":
            self.z0 = _guess(mp, B, 5, state_noise=0.3)
        elif name == "car":
            self.z0 = _guess(mp, B, 8) * 0.05
            n, m, T = mp["n"], mp["m"], mp["T"]
            for t in range(T):
                self.z0[:, t * (n + m): t * (n + m) + n] = mp["x1"] + (mp["xT"] - mp["x1"]) * t / (T - 1)
        else:
            self.z0 = _guess(mp, B, 5)
        co = cgen.build_c_oracle(osolver, f"scale_{key}", shared_parameters=bool(mp.get("shared_parameters")), cse=True)
        hess = {"exact": None, "knot-bfgs": "knot-blocks", "partitioned-bfgs": "knot-chain"}[mode]
        perm, bw = PK.analyze(pn) if hess is None else PK.analyze(pn, hessian=hess)
        kw_be = dict(dual_reg=DUAL_REG, perm=perm - 1, bw=bw, linear="band-batched", options=self.opts, c_twin=co, w=w)
        if mode == "knot-bfgs":
            self.be = QNOracleBackend(osolver, pn, B, **kw_be)
        elif mode == "partitioned-bfgs":
            self.be = PQNOracleBackend(osolver, pn, B, **kw_be)
        else:
            self.be = OracleBackend(osolver, B, **kw_be)
        self.w, self.bw = w, bw
        if key.startswith("a_"):
            self._start_half_converged(osolver, co, perm, bw)
        self.ref = sqp.solve(self.be, self.z0, self.lam0, options=self.opts, record=True)
        self.iterations = len(self.ref.history)

    def _start_half_converged(self, osolver, co, perm, bw):
        """the even problems start at a solution the twin converged to well inside the tolerances, with its multipliers"""
        tight = sqp.SQPOptions(max_iter=200, dual_reg=DUAL_REG, tol_constraint=1.0e-11, tol_dual=1.0e-9)
        one = OracleBackend(osolver, 1, dual_reg=DUAL_REG, perm=perm - 1, bw=bw, linear="band-batched", c_twin=co)
        sol = sqp.solve(one, self.z0[1:2], options=tight)
        assert sol.converged.all()
        self.lam0 = np.zeros((self.B, self.N_c))
        self.z0[::2], self.lam0[::2] = sol.z[0], sol.lam[0]

    def native(self, k):
        return sqp.SQPOptions(max_iter=k, dual_reg=DUAL_REG, bound_relax=1.0, hessian_approximation=self.mode)

    def solve_native(self, k):
        """dto_sqp_solve stopped after k iterations (the per-problem parameters go to the device first: needs a GPU)"""
        if self.w is not None and not self._params_set:
            self.pn.set_parameters(self.w)
            self._params_set = True
        return sqp.solve_native(self.pn, self.z0, self.lam0, options=self.native(k))

    # ---- what the twin's history says about the branches the native solver takes (dto_sqp_host.inc)
    def open_after_check(self):
        """problems not converged after each iteration's check"""
        return [int((~h["done"]).sum()) for h in self.ref.history]

    def open_after_first_round(self):
        """per iteration, the problems whose search went past its first round and its second-order correction"""
        return [int((h["alpha"] < 1.0).sum()) for h in self.ref.history if "alpha" in h]

    def one_pass_search_after_first_round(self):
        """some iteration leaves 1 <= n open problems after the first round with n * R <= 4 B, R = max_backtrack - 1 remaining
        step lengths: the native solver then evaluates them in one pass over its trial slots (a sufficient condition)"""
        R = self.opts.max_backtrack - 1
        return any(1 <= n and n * R <= 4 * self.B for n in self.open_after_first_round())

    def close(self):
        self.pn.close()

// dto_sqp.cu -- per-problem bookkeeping kernels of the native lock-step Newton-KKT solver (dto_sqp_solve).
//
// Reference anchor: solve!(solver) (/root/reference/src/solver.jl:45-47) hands the MOI callbacks to Ipopt; Ipopt is
// absent here and a CPU solver per problem would put PCIe back between the callbacks and their consumer, so the
// caller of the callback path is this batched solver (DESIGN section 10). The algorithm is stated once, in
// directtrajectoryoptimization.jl_b200/sqp.py (`solve`); this file and dto_sqp_host.inc are its native form: the same
// statements in the same order, one warp per problem for everything that reduces over a problem's row, so that the
// python twin driven by the CPU oracle (tests/sqp_oracle.py) checks it iterate by iterate.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "dto_sqp_dev.h"

namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ double wsum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}
// Row helpers: one warp walks a problem's row with stride 32. A single warp per row means few loads in flight unless
// they are issued in batches, so every helper loads four strided elements before it uses the first (out-of-range
// slots read nothing and contribute a neutral value); sums keep the order i = lane, lane + 32, ... of a plain loop.
#define ROW4(n, lane, i) for (int i = (lane); i < (n); i += 128)
__device__ __forceinline__ void ld4(const double* p, int i, int n, double (&v)[4], double fill)
{
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = (i + 32 * u < n) ? p[i + 32 * u] : fill;
}
__device__ __forceinline__ void st4(double* p, int i, int n, const double (&v)[4])
{
#pragma unroll
    for (int u = 0; u < 4; ++u)
        if (i + 32 * u < n) p[i + 32 * u] = v[u];
}
__device__ __forceinline__ void row_copy(double* __restrict__ dst, const double* __restrict__ src, int n, int lane)
{
    ROW4(n, lane, i) {
        double v[4];
        ld4(src, i, n, v, 0.0);
        st4(dst, i, n, v);
    }
}
// dst = x + alpha * y. dst may be x or y (in-place updates): the four loads of a batch precede its stores in program order,
// nothing is restrict here. The equality-mode callers pass 1, -1 or a power of two, where the product is exact, fused or not;
// k_ip_ls_round passes amax * 2^-k, where a contraction to an FMA rounds once and a separate multiply and add round twice, so
// its trial point may differ from the twin's z + alpha * dz in the last bit
__device__ __forceinline__ void row_axpy(double* dst, const double* x, double alpha, const double* y, int n, int lane)
{
    ROW4(n, lane, i) {
        double vx[4], vy[4];
        ld4(x, i, n, vx, 0.0);
        ld4(y, i, n, vy, 0.0);
#pragma unroll
        for (int u = 0; u < 4; ++u) vx[u] = vx[u] + alpha * vy[u];
        st4(dst, i, n, vx);
    }
}
__device__ __forceinline__ double row_sum_abs(const double* __restrict__ p, int n, int lane)
{
    double acc = 0.0;
    ROW4(n, lane, i) {
        double v[4];
        ld4(p, i, n, v, 0.0);
#pragma unroll
        for (int u = 0; u < 4; ++u) acc += fabs(v[u]);
    }
    return wsum(acc);
}
// max |x|; a NaN, once seen, is kept (torch's amax propagates NaN): a row with a NaN never passes a tolerance test
__device__ __forceinline__ double absmax_row(const double* __restrict__ r, int n, int lane, const double* __restrict__ mask = nullptr)
{
    double m = 0.0;
    ROW4(n, lane, i) {
        double v[4], k[4];
        ld4(r, i, n, v, 0.0);
        if (mask) ld4(mask, i, n, k, 0.0);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const double x = fabs(mask ? v[u] * k[u] : v[u]);
            m = (x > m || x != x) ? x : m;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double w = __shfl_xor_sync(FULL, m, o);
        m = (w > m || w != w) ? w : m;
    }
    return m;
}
__device__ __forceinline__ bool finite_row(const double* __restrict__ r, int n, int lane)
{
    bool ok = true;
    ROW4(n, lane, i) {
        double v[4];
        ld4(r, i, n, v, 0.0);
#pragma unroll
        for (int u = 0; u < 4; ++u) ok = ok && isfinite(v[u]);
    }
    return __all_sync(FULL, ok);
}

#define WARP_PROBLEM()                                                        \
    const int lane = threadIdx.x & 31;                                        \
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); \
    if (b >= a.B) return;

// ---- delta = lm; the callbacks see z and lam * exact (Hessian multipliers), the factor kernel sees delta
__global__ void k_begin(const dto_sqp_args a)
{
    WARP_PROBLEM();
    const double ex = a.exact[b];
    row_copy(a.bz + b * a.N_z, a.z + b * a.N_z, a.N_z, lane);
    {
        const double* __restrict__ src = a.lam + b * a.N_c;
        double* __restrict__ dst = a.blam + b * a.N_c;
        ROW4(a.N_c, lane, i) {
            double v[4];
            ld4(src, i, a.N_c, v, 0.0);
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] *= ex;
            st4(dst, i, a.N_c, v);
        }
    }
    if (lane == 0) {
        const double d = a.lm[b];
        a.delta[b] = d;
        a.preg[b] = d;
    }
}

__global__ void k_set_lam(const dto_sqp_args a)
{
    WARP_PROBLEM();
    row_copy(a.blam + b * a.N_c, a.lam + b * a.N_c, a.N_c, lane);
}

// ---- after the callbacks and the first factorisation of the iteration
__global__ void k_after_first(const dto_sqp_args a)
{
    WARP_PROBLEM();
    const double* c = a.bc + b * a.N_c;
    const double dr = absmax_row(a.rhs + b * a.dim, a.N_z, lane, a.free);   // ||(g + J'lam) * free||_inf
    const double cv = absmax_row(c, a.N_c, lane);
    row_copy(a.ckeep + b * a.N_c, c, a.N_c, lane);
    const bool fin = finite_row(a.sol + b * a.dim, a.dim, lane);
    if (lane == 0) {
        a.cv[b] = cv;
        a.dr[b] = dr;
        a.fcur[b] = a.bf[b];
        a.exact[b] = cv <= a.p.exact_below ? 1.0 : 0.0;
        bool done = a.done[b] != 0;
        const bool newly = !done && cv <= a.p.tol_constraint && dr <= a.p.tol_dual;
        if (newly) a.iters[b] = a.it;
        done = done || newly;
        a.done[b] = done ? 1 : 0;
        const bool bad = (a.nneg[b] != a.N_c || !fin) && !done;
        a.bad[b] = bad ? 1 : 0;
        a.first[b] = 1;
        a.tries[b] = 0;
        if (done) atomicAdd(a.counters + DTO_SQP_N_DONE, 1);
        if (!done) a.alist[atomicAdd(a.counters + DTO_SQP_N_ACTIVE, 1)] = (int32_t)b;   // the next first factorisation skips the others
        if (bad) {
            atomicAdd(a.counters + DTO_SQP_N_BAD, 1);
            if (a.p.max_refactor > 0) atomicAdd(a.counters + DTO_SQP_N_RETRY, 1);
        }
    }
}

// ---- inertia control (Ipopt's IC rule per problem): next regularisation of the problems whose pivot count was wrong
__global__ void k_reg_next(const dto_sqp_args a)
{
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B || !a.bad[b] || a.tries[b] >= a.p.max_refactor) return;
    const double dl = a.delta_last[b], d = a.delta[b];
    const double start = dl == 0.0 ? a.p.reg_first : fmax(a.p.reg_min, a.p.reg_dec * dl);
    const double grow = dl == 0.0 ? a.p.reg_inc_first : a.p.reg_inc;
    const double nxt = a.first[b] ? fmax(start, 2.0 * d) : fmin(a.p.reg_max, grow * d);
    a.delta[b] = nxt;
    a.preg[b] = nxt;
    a.first[b] = 0;
    a.tries[b] += 1;
    a.idx[atomicAdd(a.counters + DTO_SQP_N_IDX, 1)] = (int32_t)b;
}

__global__ void k_recheck(const dto_sqp_args a, int32_t count)
{
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= count) return;
    const int64_t b = a.idx[k];
    const bool fin = finite_row(a.sol + b * a.dim, a.dim, lane);
    if (lane == 0) {
        const bool bad = a.nneg[b] != a.N_c || !fin;   // (these problems are not done)
        a.bad[b] = bad ? 1 : 0;
        if (bad) atomicAdd(a.counters + DTO_SQP_N_BAD, 1);
        if (bad && a.tries[b] < a.p.max_refactor) atomicAdd(a.counters + DTO_SQP_N_RETRY, 1);
    }
}

// ---- step, l1-merit quantities (curvature rule for the penalty), first trial point
__global__ void k_direction(const dto_sqp_args a)
{
    WARP_PROBLEM();
    const double* sol = a.sol + b * a.dim;
    const double* g = a.bg + b * a.N_z;
    const double* ck = a.ckeep + b * a.N_c;
    double gd = 0.0, c1 = 0.0, cl = 0.0;
    {
        const double* __restrict__ fr = a.free;
        const double* __restrict__ zc = a.z + b * a.N_z;
        double* __restrict__ dz = a.dz + b * a.N_z;
        double* __restrict__ bz = a.bz + b * a.N_z;
        ROW4(a.N_z, lane, i) {
            double vs[4], vf[4], vg[4], vz[4];
            ld4(sol, i, a.N_z, vs, 0.0);
            ld4(fr, i, a.N_z, vf, 0.0);
            ld4(g, i, a.N_z, vg, 0.0);
            ld4(zc, i, a.N_z, vz, 0.0);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const double d = -vs[u] * vf[u];
                vs[u] = d;
                if (i + 32 * u < a.N_z) gd += vg[u] * d;      // (guarded: 0 * inf of a padded slot would be NaN)
                vz[u] = vz[u] + 1.0 * d;                      // first trial: alpha = 1
            }
            st4(dz, i, a.N_z, vs);
            st4(bz, i, a.N_z, vz);
        }
        const double* __restrict__ sl = sol + a.N_z;
        const double* __restrict__ lam = a.lam + b * a.N_c;
        double* __restrict__ dlam = a.dlam + b * a.N_c;
        ROW4(a.N_c, lane, i) {
            double vs[4], vc[4], vl[4];
            ld4(sl, i, a.N_c, vs, 0.0);
            ld4(ck, i, a.N_c, vc, 0.0);
            ld4(lam, i, a.N_c, vl, 0.0);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const double dl = -vs[u];
                vs[u] = dl;
                if (i + 32 * u < a.N_c) {
                    c1 += fabs(vc[u]);
                    cl += vc[u] * (vl[u] + dl);
                }
            }
            st4(dlam, i, a.N_c, vs);
        }
    }
    gd = wsum(gd);
    c1 = wsum(c1);
    cl = wsum(cl);
    if (lane == 0) {
        const double delta = a.delta[b], lm = a.lm[b];
        if (delta > lm) a.delta_last[b] = delta;
        const double curv = fmax(-gd + cl, 0.0);
        const double nu_need = (gd + 0.5 * curv) / ((1.0 - a.p.merit_rho) * fmax(c1, 1.0e-300));
        const double nu = fmax(a.p.merit_min, a.p.merit_margin * nu_need);
        a.nu[b] = nu;
        a.c1[b] = c1;
        a.slope[b] = gd - nu * c1;
        a.phi0[b] = a.fcur[b] + nu * c1;
        a.alpha[b] = 1.0;
        a.accepted[b] = (a.done[b] || a.bad[b]) ? 1 : 0;   // converged problems and failed factorisations do not move
    }
}

// ---- one backtracking round: bz holds the trial point, bf / bc its objective and constraint values
__global__ void k_ls_round(const dto_sqp_args a, int32_t round)
{
    WARP_PROBLEM();
    const double* ct = a.bc + b * a.N_c;
    const double ct1 = row_sum_abs(ct, a.N_c, lane);
    bool accepted = a.accepted[b] != 0;
    double alpha = a.alpha[b];
    const double nu = a.nu[b];
    const double phit = a.bf[b] + nu * ct1;
    const bool ok = (phit <= a.phi0[b] + a.p.armijo * alpha * a.slope[b]) && !accepted;
    if (ok) {
        row_copy(a.z + b * a.N_z, a.bz + b * a.N_z, a.N_z, lane);
        row_axpy(a.lam + b * a.N_c, a.lam + b * a.N_c, alpha, a.dlam + b * a.N_c, a.N_c, lane);
    }
    accepted = accepted || ok;
    if (round == 0 && a.p.soc) {
        // second-order correction candidates: rejected full steps that did not even reduce the constraint violation
        const bool need = !accepted && ct1 >= a.c1[b];
        // c(z) + c(z + dz), straight into the constraint part of the right-hand side [g + J'lam ; c] (the rest of it stays)
        if (need) row_axpy(a.rhs + b * a.dim + a.N_z, a.ckeep + b * a.N_c, 1.0, ct, a.N_c, lane);
        if (lane == 0) {
            a.need[b] = need ? 1 : 0;
            if (need) a.idx[atomicAdd(a.counters + DTO_SQP_N_NEED, 1)] = (int32_t)b;
        }
    }
    if (!accepted) alpha = 0.5 * alpha;
    __syncwarp();
    row_axpy(a.bz + b * a.N_z, a.z + b * a.N_z, alpha, a.dz + b * a.N_z, a.N_z, lane);   // next trial
    if (lane == 0) {
        a.accepted[b] = accepted ? 1 : 0;
        a.alpha[b] = alpha;
        if (!accepted) a.oidx[atomicAdd(a.counters + DTO_SQP_N_OPEN, 1)] = (int32_t)b;   // the host stops the search when no problem is open
    }
}

__global__ void k_soc_trial(const dto_sqp_args a, int32_t count)
{
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= count) return;
    const int64_t b = a.idx[k];
    const double* sol = a.sol + b * a.dim;
    const double* __restrict__ zc = a.z + b * a.N_z;
    const double* __restrict__ fr = a.free;
    double* __restrict__ bz = a.bz + b * a.N_z;
    ROW4(a.N_z, lane, i) {
        double vs[4], vf[4], vz[4];
        ld4(sol, i, a.N_z, vs, 0.0);
        ld4(fr, i, a.N_z, vf, 0.0);
        ld4(zc, i, a.N_z, vz, 0.0);
#pragma unroll
        for (int u = 0; u < 4; ++u) vz[u] = vz[u] + (-vs[u] * vf[u]);
        st4(bz, i, a.N_z, vz);
    }
}

__global__ void k_soc_accept(const dto_sqp_args a, int32_t count)
{
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= count) return;
    const int64_t b = a.idx[k];
    const double* cs = a.bc + b * a.N_c;
    const double* sol = a.sol + b * a.dim;
    const double cs1 = row_sum_abs(cs, a.N_c, lane);
    const bool fin = finite_row(sol, a.dim, lane);
    const bool oks = (a.bf[b] + a.nu[b] * cs1 <= a.phi0[b] + a.p.armijo * a.slope[b]) && fin;
    double alpha = a.alpha[b];
    if (oks) {
        row_copy(a.z + b * a.N_z, a.bz + b * a.N_z, a.N_z, lane);
        row_axpy(a.lam + b * a.N_c, a.lam + b * a.N_c, -1.0, sol + a.N_z, a.N_c, lane);   // lam - sol_lambda
        alpha = 1.0;   // the full (corrected) step was taken: round 0 had already halved alpha for this problem
    }
    __syncwarp();
    row_axpy(a.bz + b * a.N_z, a.z + b * a.N_z, alpha, a.dz + b * a.N_z, a.N_z, lane);   // trial of round 1
    if (lane == 0) {
        if (oks) {
            a.accepted[b] = 1;
            atomicAdd(a.counters + DTO_SQP_N_SOC_OK, 1);
        }
        a.alpha[b] = alpha;
    }
}

// ---- end of the iteration: multiplier safeguard, Levenberg-Marquardt damping, regularisation memory
__global__ void k_end(const dto_sqp_args a)
{
    WARP_PROBLEM();
    if (a.p.lam_max > 0.0) {
        const double m = absmax_row(a.lam + b * a.N_c, a.N_c, lane);
        if (m > a.p.lam_max)
            for (int i = lane; i < a.N_c; i += 32) a.lam[b * a.N_c + i] = 0.0;   // (stores only)
    }
    if (lane == 0) {
        const bool accepted = a.accepted[b] != 0, done = a.done[b] != 0, bad = a.bad[b] != 0;
        const bool moved = !done && !bad;
        const double alpha = a.alpha[b], delta = a.delta[b];
        double lm = a.lm[b];
        if (moved && alpha < a.p.lm_grow_below) lm = fmax(a.p.lm_min, a.p.lm_grow * fmax(lm, delta));
        if (moved && accepted && alpha >= 1.0) lm = a.p.lm_shrink * lm;
        if (lm < a.p.lm_zero) lm = 0.0;
        a.lm[b] = lm;
        if (!accepted || bad) a.delta_last[b] = fmax(a.p.reg_first, a.p.reg_inc * fmax(a.delta_last[b], delta));
    }
}

// ---- the remaining backtracking rounds of the open problems in one pass: R sequential rounds would try
// alpha, alpha/2, .., alpha/2^(R-1) one after the other and take the first that passes; here every such trial point
// gets a slot of the trial arrays, the objective and constraint kernels run once over the slots, and k_multi_pick
// takes the first passing one in the same order (same trial points, same kernels, same test: same result)
__global__ void k_multi_trial(const dto_sqp_args a, int32_t count, int32_t R)
{
    const int lane = threadIdx.x & 31;
    const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (s >= (int64_t)count * R) return;
    const int64_t k = s / R;
    const int j = (int)(s - k * R);
    const int64_t b = a.oidx[k];
    double alpha = a.alpha[b];
    for (int q = 0; q < j; ++q) alpha = 0.5 * alpha;
    row_axpy(a.tz + s * a.N_z, a.z + b * a.N_z, alpha, a.dz + b * a.N_z, a.N_z, lane);
    if (a.N_w > 0) row_copy(a.tw + s * a.N_w, a.w + b * a.N_w, a.N_w, lane);
}

__global__ void k_multi_pick(const dto_sqp_args a, int32_t count, int32_t R)
{
    const int lane = threadIdx.x & 31;
    const int64_t k = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (k >= count) return;
    const int64_t b = a.oidx[k];
    if (a.accepted[b]) return;            // taken by the second-order correction after the list was written
    double alpha = a.alpha[b];
    const double nu = a.nu[b], phi0 = a.phi0[b], slope = a.slope[b];
    bool taken = false;
    for (int j = 0; j < R && !taken; ++j) {
        const int64_t s = k * R + j;
        const double* ct = a.tc + s * a.N_c;
        const double ct1 = row_sum_abs(ct, a.N_c, lane);
        const double phit = a.tf[s] + nu * ct1;
        if (phit <= phi0 + a.p.armijo * alpha * slope) {
            row_copy(a.z + b * a.N_z, a.tz + s * a.N_z, a.N_z, lane);
            row_axpy(a.lam + b * a.N_c, a.lam + b * a.N_c, alpha, a.dlam + b * a.N_c, a.N_c, lane);
            taken = true;
        } else {
            alpha = 0.5 * alpha;
        }
    }
    if (lane == 0) {
        a.alpha[b] = alpha;
        if (taken) a.accepted[b] = 1;
    }
}

// ---- inertia correction, m tries at once: sequential tries would factorise a bad problem with nxt_1, look at the
// pivot count, then with nxt_2 = grow * nxt_1, ... Each try costs the full latency of a banded factorisation however
// few problems take part, so the next m values of the ladder are factorised side by side in candidate slots and the
// first one that works is kept: the same regularisation, factor and step the sequential tries end with.
// the next values of problem b's ladder from (d, first): what m sequential tries would use; entries past the problem's
// remaining tries repeat the last value (a duplicate factorisation nobody prefers)
__device__ __forceinline__ void ladder_values(const dto_sqp_args& a, int64_t b, double d, bool first, int32_t m, int32_t left, int64_t k,
                                              double* __restrict__ vreg, int32_t* __restrict__ vidx)
{
    const double dl = a.delta_last[b];
    const double start = dl == 0.0 ? a.p.reg_first : fmax(a.p.reg_min, a.p.reg_dec * dl);
    const double grow = dl == 0.0 ? a.p.reg_inc_first : a.p.reg_inc;
    for (int j = 0; j < m; ++j) {
        if (j < left) d = first ? fmax(start, 2.0 * d) : fmin(a.p.reg_max, grow * d);
        first = false;
        vreg[k * m + j] = d;
        vidx[k * m + j] = (int32_t)b;
    }
}

__global__ void k_reg_ladder(const dto_sqp_args a, int32_t m)
{
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= a.B || !a.bad[b]) return;
    const int32_t left = a.p.max_refactor - a.tries[b];
    if (left <= 0) return;
    const int64_t k = atomicAdd(a.counters + DTO_SQP_N_IDX, 1);
    a.idx[k] = (int32_t)b;
    ladder_values(a, b, a.delta[b], a.first[b] != 0, m, left, k, a.vreg, a.vidx);
    a.first[b] = 0;
    a.tries[b] += left < m ? left : m;
}

// block per listed problem: the first candidate with N_c negative pivots and a finite solution is kept
__global__ void __launch_bounds__(256) k_pick(const dto_sqp_args a, int32_t count, int32_t m)
{
    __shared__ int s_pick, s_good;
    const int64_t k = blockIdx.x;
    const int64_t b = a.idx[k];
    const double* __restrict__ vreg = a.vreg;
    const double* __restrict__ vsol = a.vsol;
    const int32_t* __restrict__ vnneg = a.vnneg;
    const double* __restrict__ vL = a.vL;
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        int pick = m - 1, good = 0;
        for (int j = 0; j < m; ++j) {
            const int64_t v = k * m + j;
            const bool fin = finite_row(vsol + v * a.dim, a.dim, lane);
            if (vnneg[v] == a.N_c && fin) {
                pick = j;
                good = 1;
                break;
            }
        }
        if (lane == 0) {
            s_pick = pick;
            s_good = good;
            const int64_t v = k * m + pick;
            a.delta[b] = vreg[v];      // a failed ladder leaves the last value tried, as sequential tries do
            a.preg[b] = vreg[v];
            a.nneg_w[b] = vnneg[v];
            a.bad[b] = good ? 0 : 1;
            if (!good) atomicAdd(a.counters + DTO_SQP_N_BAD, 1);
            if (!good && a.tries[b] < a.p.max_refactor) atomicAdd(a.counters + DTO_SQP_N_RETRY, 1);
        }
    }
    __syncthreads();
    const int64_t v = k * m + s_pick;
    for (int i = threadIdx.x; i < a.dim; i += blockDim.x) a.sol_w[b * a.dim + i] = vsol[v * a.dim + i];
    if (s_good) {   // the factor is read again by a second-order correction
        const double2* __restrict__ src = reinterpret_cast<const double2*>(vL + (size_t)v * a.factor_stride);
        double2* __restrict__ dst = reinterpret_cast<double2*>(a.L + (size_t)b * a.factor_stride);
        const int64_t n2 = a.factor_stride / 2, step = blockDim.x;
        for (int64_t i = threadIdx.x; i < n2; i += 4 * step) {
            double2 v4[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i + u * step < n2) v4[u] = src[i + u * step];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (i + u * step < n2) dst[i + u * step] = v4[u];
        }
    }
}

// =====================================================================================================================
// Interior-point mode (sqp.py `solve`, the `ip` branches): inequality bounds on variables and inequality rows c_i(z) <= 0.
// Barrier terms enter the SAME Newton-KKT step as a per-problem diagonal of K (Sigma = z_L/(x-l) + z_U/(u-x) on bounded
// variables, -t_i/lam_i on inequality rows whose slacks t are eliminated), a shifted gradient and a shifted constraint
// right-hand side. Separate kernels: the equality-only kernels above are what the parity tests pinned and stay untouched.
// =====================================================================================================================
__device__ __forceinline__ double wmin(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(FULL, v, o));
    return v;
}
__device__ __forceinline__ double wmaxnan(double m)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double w = __shfl_xor_sync(FULL, m, o);
        m = (w > m || w != w) ? w : m;
    }
    return m;
}
#define KEEPMAX(m, x)                     \
    do {                                  \
        const double x__ = fabs(x);       \
        m = (x__ > m || x__ != x__) ? x__ : m; \
    } while (0)

// The five k_ip_* kernels read the bound values of problem b at lo + b * bstride, up + b * bstride. PP (per-problem bound
// values, bstride = N_z) is a template flag so that the shared-bounds instantiation (bstride = 0) is the code without a stride.

// after the callbacks (g, c, J, H at z): diagonal of K, barrier gradient into g, shifted constraint right-hand side,
// residual of c(z) + t = 0 into ckeep, barrier value; first iteration: slacks and their multipliers
template <bool PP>
__global__ void k_ip_prepare(const dto_sqp_args a)
{
    WARP_PROBLEM();
    const double mu = a.mu[b];
    double accB = 0.0, accI = 0.0;
    const double* z = a.z + b * a.N_z;
    const double *lo = PP ? a.lo + b * a.bstride : a.lo, *up = PP ? a.up + b * a.bstride : a.up;
    for (int i = lane; i < a.N_z; i += 32) {
        const double hl = a.hasL[i], hu = a.hasU[i];
        const double sL = hl > 0.0 ? z[i] - lo[i] : 1.0, sU = hu > 0.0 ? up[i] - z[i] : 1.0;
        a.diag[b * a.dim + i] = hl * a.zL[b * a.N_z + i] / sL + hu * a.zU[b * a.N_z + i] / sU;
        a.bg_w[b * a.N_z + i] += mu * (hu / sU - hl / sL);
        accB += hl * log(sL) + hu * log(sU);
    }
    for (int j = lane; j < a.N_c; j += 32) {
        const double c = a.bc[b * a.N_c + j];
        if (a.p.any_ineq) {
            const double hi = a.hasI[j];
            double t = a.t[b * a.N_c + j], lam = a.lam[b * a.N_c + j];
            if (a.it == 0) {   // slacks from the constraint values at the start, multipliers on the central path
                t = hi * fmax(-c, a.p.bound_push);
                if (hi > 0.0) lam = mu / fmax(t, 1.0e-300);
                a.t[b * a.N_c + j] = t;
                a.lam[b * a.N_c + j] = lam;
            }
            const double tS = hi > 0.0 ? t : 1.0, lamI = hi > 0.0 ? lam : 1.0;
            a.diag[b * a.dim + a.N_z + j] = -hi * tS / lamI;
            a.ckeep[b * a.N_c + j] = c + hi * t;                // residual of c(z) + t = 0
            a.bc[b * a.N_c + j] = c + hi * (mu / lamI);         // right-hand side of the row
            accI += hi * log(tS);
        } else {
            a.ckeep[b * a.N_c + j] = c;
        }
    }
    accB = wsum(accB);
    accI = wsum(accI);
    if (lane == 0) a.fbar[b] = -mu * accI - mu * accB;
}

template <bool PP>
__global__ void k_ip_after_first(const dto_sqp_args a)
{
    WARP_PROBLEM();
    const double mu = a.mu[b];
    const double* z = a.z + b * a.N_z;
    const double* rz = a.rhs + b * a.dim;
    const double *lo = PP ? a.lo + b * a.bstride : a.lo, *up = PP ? a.up + b * a.bstride : a.up;
    double dr = 0.0, comp = 0.0, emu = 0.0;
    for (int i = lane; i < a.N_z; i += 32) {
        const double hl = a.hasL[i], hu = a.hasU[i];
        const double sL = hl > 0.0 ? z[i] - lo[i] : 1.0, sU = hu > 0.0 ? up[i] - z[i] : 1.0;
        const double zL = a.zL[b * a.N_z + i], zU = a.zU[b * a.N_z + i];
        const double gshift = mu * (hu / sU - hl / sL);
        KEEPMAX(dr, (rz[i] - gshift - zL + zU) * a.free[i]);     // g + J'lam - z_L + z_U of the ORIGINAL problem
        const double cL = hl * sL * zL, cU = hu * sU * zU;
        KEEPMAX(comp, cL);
        KEEPMAX(comp, cU);
        KEEPMAX(emu, cL - hl * mu);
        KEEPMAX(emu, cU - hu * mu);
    }
    if (a.p.any_ineq)
        for (int j = lane; j < a.N_c; j += 32) {
            const double hi = a.hasI[j];
            const double cI = hi * (hi > 0.0 ? a.t[b * a.N_c + j] * a.lam[b * a.N_c + j] : 1.0);
            KEEPMAX(comp, cI);
            KEEPMAX(emu, cI - hi * mu);
        }
    dr = wmaxnan(dr);
    comp = wmaxnan(comp);
    emu = wmaxnan(emu);
    const double cv = absmax_row(a.ckeep + b * a.N_c, a.N_c, lane);
    const bool fin = finite_row(a.sol + b * a.dim, a.dim, lane);
    if (lane == 0) {
        double e = dr > cv ? dr : cv;
        e = (emu > e || emu != emu) ? emu : e;
        const double lower = fmin(a.p.kappa_mu * mu, pow(mu, a.p.theta_mu));
        a.mu_next[b] = (e <= a.p.kappa_eps * mu) ? fmax(a.p.mu_floor, lower) : mu;
        const double drc = (comp > dr || comp != comp) ? comp : dr;
        a.cv[b] = cv;
        a.dr[b] = drc;
        a.fcur[b] = a.bf[b] + a.fbar[b];
        a.exact[b] = cv <= a.p.exact_below ? 1.0 : 0.0;
        bool done = a.done[b] != 0;
        const bool newly = !done && cv <= a.p.tol_constraint && drc <= a.p.tol_dual;
        if (newly) a.iters[b] = a.it;
        done = done || newly;
        a.done[b] = done ? 1 : 0;
        const bool bad = (a.nneg[b] != a.N_c || !fin) && !done;
        a.bad[b] = bad ? 1 : 0;
        a.first[b] = 1;
        a.tries[b] = 0;
        if (done) atomicAdd(a.counters + DTO_SQP_N_DONE, 1);
        if (!done) a.alist[atomicAdd(a.counters + DTO_SQP_N_ACTIVE, 1)] = (int32_t)b;
        if (bad) {
            atomicAdd(a.counters + DTO_SQP_N_BAD, 1);
            if (a.p.max_refactor > 0) atomicAdd(a.counters + DTO_SQP_N_RETRY, 1);
        }
    }
}

template <bool PP>
__global__ void k_ip_direction(const dto_sqp_args a)
{
    WARP_PROBLEM();
    const double mu = a.mu[b];
    const double tau = fmax(a.p.tau_min, 1.0 - mu);
    const double* sol = a.sol + b * a.dim;
    const double* z = a.z + b * a.N_z;
    const double *lo = PP ? a.lo + b * a.bstride : a.lo, *up = PP ? a.up + b * a.bstride : a.up;
    const double big = 1.0e300;
    double gd = 0.0, c1 = 0.0, cl = 0.0, gdt = 0.0, amax = big, az = big;
    for (int i = lane; i < a.N_z; i += 32) {
        const double d = -sol[i] * a.free[i];
        a.dz[b * a.N_z + i] = d;
        gd += a.bg[b * a.N_z + i] * d;
        const double hl = a.hasL[i], hu = a.hasU[i];
        const double sL = hl > 0.0 ? z[i] - lo[i] : 1.0, sU = hu > 0.0 ? up[i] - z[i] : 1.0;
        const double zL = a.zL[b * a.N_z + i], zU = a.zU[b * a.N_z + i];
        const double dzL = hl * (mu / sL - zL - (hl * zL / sL) * d);
        const double dzU = hu * (mu / sU - zU + (hu * zU / sU) * d);
        a.dzL[b * a.N_z + i] = dzL;
        a.dzU[b * a.N_z + i] = dzU;
        if (hl > 0.0 && d < 0.0) amax = fmin(amax, -tau * sL / fmin(d, -1.0e-300));
        if (hu > 0.0 && d > 0.0) amax = fmin(amax, tau * sU / fmax(d, 1.0e-300));
        if (dzL < 0.0) az = fmin(az, -tau * zL / fmin(dzL, -1.0e-300));
        if (dzU < 0.0) az = fmin(az, -tau * zU / fmin(dzU, -1.0e-300));
    }
    for (int j = lane; j < a.N_c; j += 32) {
        const double dl = -sol[a.N_z + j];
        a.dlam[b * a.N_c + j] = dl;
        const double ck = a.ckeep[b * a.N_c + j], lam = a.lam[b * a.N_c + j];
        c1 += fabs(ck);
        cl += ck * (lam + dl);
        if (a.p.any_ineq) {
            const double hi = a.hasI[j];
            const double tS = hi > 0.0 ? a.t[b * a.N_c + j] : 1.0, lamI = hi > 0.0 ? lam : 1.0;
            const double dt = hi * (mu / lamI - tS - (tS / lamI) * dl);      // from t lam = mu, linearised
            a.dt[b * a.N_c + j] = dt;
            if (hi > 0.0 && dt < 0.0) amax = fmin(amax, -tau * tS / fmin(dt, -1.0e-300));
            if (hi > 0.0 && dl < 0.0) az = fmin(az, -tau * lamI / fmin(dl, -1.0e-300));
            gdt += hi * (mu / tS) * dt;
        }
    }
    gd = wsum(gd);
    c1 = wsum(c1);
    cl = wsum(cl);
    gdt = wsum(gdt);
    amax = fmin(1.0, wmin(amax));
    az = fmin(1.0, wmin(az));
    {
        double* bz = a.bz + b * a.N_z;
        for (int i = lane; i < a.N_z; i += 32) bz[i] = z[i] + amax * a.dz[b * a.N_z + i];      // first trial: the longest allowed step
    }
    if (lane == 0) {
        const double delta = a.delta[b], lm = a.lm[b];
        if (delta > lm) a.delta_last[b] = delta;
        const double curv = fmax(-gd + cl, 0.0);
        const double nu_need = (gd + 0.5 * curv) / ((1.0 - a.p.merit_rho) * fmax(c1, 1.0e-300));
        const double nu = fmax(a.p.merit_min, a.p.merit_margin * nu_need);
        gd -= gdt;                                   // the barrier of the slacks joins the slope
        a.nu[b] = nu;
        a.c1[b] = c1;
        a.slope[b] = gd - nu * c1;
        a.phi0[b] = a.fcur[b] + nu * c1;
        a.alpha[b] = amax;
        a.amax[b] = amax;
        a.a_z[b] = az;
        a.accepted[b] = (a.done[b] || a.bad[b]) ? 1 : 0;
    }
}

template <bool PP>
__global__ void k_ip_ls_round(const dto_sqp_args a, int32_t round)
{
    WARP_PROBLEM();
    const double mu = a.mu[b];
    double alpha = a.alpha[b];
    const double az = a.a_z[b];
    const double* bz = a.bz + b * a.N_z;
    const double *lo = PP ? a.lo + b * a.bstride : a.lo, *up = PP ? a.up + b * a.bstride : a.up;
    double barB = 0.0, barI = 0.0, ct1 = 0.0, mdz = 0.0, mz = 0.0;
    for (int i = lane; i < a.N_z; i += 32) {
        const double hl = a.hasL[i], hu = a.hasU[i];
        const double sL = hl > 0.0 ? fmax(bz[i] - lo[i], 1.0e-300) : 1.0, sU = hu > 0.0 ? fmax(up[i] - bz[i], 1.0e-300) : 1.0;
        barB += hl * log(sL) + hu * log(sU);
        KEEPMAX(mdz, a.dz[b * a.N_z + i]);
        KEEPMAX(mz, a.z[b * a.N_z + i]);
    }
    for (int j = lane; j < a.N_c; j += 32) {
        double r = a.bc[b * a.N_c + j];
        if (a.p.any_ineq) {
            const double hi = a.hasI[j];
            const double tt = hi > 0.0 ? fmax(a.t[b * a.N_c + j] + alpha * a.dt[b * a.N_c + j], 1.0e-300) : 1.0;
            barI += hi * log(tt);
            r += hi * tt;
        }
        ct1 += fabs(r);
    }
    barB = wsum(barB);
    barI = wsum(barI);
    ct1 = wsum(ct1);
    mdz = wmaxnan(mdz);
    mz = wmaxnan(mz);
    bool accepted = a.accepted[b] != 0;
    const double phi0 = a.phi0[b];
    double ft = a.bf[b] - mu * barB;
    ft = ft - mu * barI;
    const double phit = ft + a.nu[b] * ct1;
    bool ok = (phit <= phi0 + a.p.armijo * alpha * a.slope[b] + 2.2e-15 * fabs(phi0)) && !accepted;
    if (round == 0) ok = ok || ((mdz <= a.p.tiny_step * (1.0 + mz)) && !accepted);      // tiny steps are taken untested
    if (ok) {
        for (int i = lane; i < a.N_z; i += 32) {
            a.z[b * a.N_z + i] = bz[i];
            a.zL[b * a.N_z + i] += az * a.dzL[b * a.N_z + i];
            a.zU[b * a.N_z + i] += az * a.dzU[b * a.N_z + i];
        }
        for (int j = lane; j < a.N_c; j += 32) {
            const double hi = a.p.any_ineq ? a.hasI[j] : 0.0;
            a.lam[b * a.N_c + j] += (hi > 0.0 ? az : alpha) * a.dlam[b * a.N_c + j];
            if (a.p.any_ineq) a.t[b * a.N_c + j] = hi * (hi > 0.0 ? fmax(a.t[b * a.N_c + j] + alpha * a.dt[b * a.N_c + j], 1.0e-300) : 1.0);
        }
    }
    accepted = accepted || ok;
    if (!accepted) alpha = 0.5 * alpha;
    __syncwarp();
    row_axpy(a.bz + b * a.N_z, a.z + b * a.N_z, alpha, a.dz + b * a.N_z, a.N_z, lane);   // next trial
    if (lane == 0) {
        a.accepted[b] = accepted ? 1 : 0;
        a.alpha[b] = alpha;
        if (!accepted) a.oidx[atomicAdd(a.counters + DTO_SQP_N_OPEN, 1)] = (int32_t)b;
    }
}

template <bool PP>
__global__ void k_ip_end(const dto_sqp_args a)
{
    WARP_PROBLEM();
    const double mu = a.mu[b];
    if (a.p.lam_max > 0.0) {      // runaway multiplier estimates start again from zero -- equality rows only (lam_I > 0 is a barrier quantity)
        double m = 0.0;
        for (int j = lane; j < a.N_c; j += 32) KEEPMAX(m, a.lam[b * a.N_c + j] * (a.p.any_ineq ? 1.0 - a.hasI[j] : 1.0));
        m = wmaxnan(m);
        if (m > a.p.lam_max)
            for (int j = lane; j < a.N_c; j += 32) a.lam[b * a.N_c + j] *= (a.p.any_ineq ? a.hasI[j] : 0.0);
    }
    const double ks = a.p.kappa_sigma;
    const double *lo = PP ? a.lo + b * a.bstride : a.lo, *up = PP ? a.up + b * a.bstride : a.up;
    for (int i = lane; i < a.N_z; i += 32) {      // z_L, z_U within [mu / (kappa s), kappa mu / s] of the new slacks
        const double hl = a.hasL[i], hu = a.hasU[i];
        const double zi = a.z[b * a.N_z + i];
        const double sL = hl > 0.0 ? zi - lo[i] : 1.0, sU = hu > 0.0 ? up[i] - zi : 1.0;
        a.zL[b * a.N_z + i] = hl * fmax(fmin(a.zL[b * a.N_z + i], ks * mu / sL), mu / (ks * sL));
        a.zU[b * a.N_z + i] = hu * fmax(fmin(a.zU[b * a.N_z + i], ks * mu / sU), mu / (ks * sU));
    }
    if (a.p.any_ineq)
        for (int j = lane; j < a.N_c; j += 32)
            if (a.hasI[j] > 0.0) {
                const double t = a.t[b * a.N_c + j];
                a.lam[b * a.N_c + j] = fmax(fmin(a.lam[b * a.N_c + j], ks * mu / t), mu / (ks * t));
            }
    if (lane == 0) {
        const bool accepted = a.accepted[b] != 0, done = a.done[b] != 0, bad = a.bad[b] != 0;
        if (!done) a.mu[b] = a.mu_next[b];
        const bool moved = !done && !bad;
        const double alpha = a.alpha[b] / a.amax[b], delta = a.delta[b];     // fraction of the allowed step that was taken
        double lm = a.lm[b];
        if (moved && alpha < a.p.lm_grow_below) lm = fmax(a.p.lm_min, a.p.lm_grow * fmax(lm, delta));
        if (moved && accepted && alpha >= 1.0) lm = a.p.lm_shrink * lm;
        if (lm < a.p.lm_zero) lm = 0.0;
        a.lm[b] = lm;
        if (!accepted || bad) a.delta_last[b] = fmax(a.p.reg_first, a.p.reg_inc * fmax(a.delta_last[b], delta));
    }
}


// =====================================================================================================================
// Knot-block damped BFGS (hessian_approximation = 1; sqp.py `knot_bfgs_update` states it): H of K is one dense symmetric
// block per knot over that knot's variables, updated once per iteration right after the callbacks (Nocedal & Wright,
// Procedure 18.2). A group of W lanes owns one (problem, knot) block, lane i row (and, by symmetry, column) i; W = 16 puts
// two blocks in a warp. Column i of a block is read and written by lane i, so consecutive lanes touch consecutive doubles.
// =====================================================================================================================
template <int W>
__device__ __forceinline__ double gsum(double v)
{
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o, W);
    return v;
}

// One damped BFGS update of a dense symmetric n x n block (n <= W) held by a group of W lanes, lane i with s_i and y_i of
// the block's variable i; `upd` is the block's first-update flag. Both quasi-Newton modes call it: k_qn_update on knot
// blocks, k_pqn_update on element blocks. A lane with i >= n, or a group with `live` false, only takes part in the shuffles.
template <int W>
__device__ __forceinline__ void qn_block_update(double* __restrict__ blk, int n, int i, bool live, double s, double y, uint8_t* upd)
{
    const bool own = i < n;
    const double ss = gsum<W>(s * s), sy = gsum<W>(s * y), yy = gsum<W>(y * y);
    bool ok = live && ss > 1.0e-30 && isfinite(ss) && isfinite(sy) && isfinite(yy);
    // the block's first update starts from (y'y / s'y) I instead of the identity
    const bool scale = ok && !*upd && sy > 0.0;
    const double sc = yy / sy;
    const int nmax = (int)__reduce_max_sync(FULL, (unsigned)n);
    double bs = 0.0;   // (B s)_i = sum_j B(j, i) s_j, j ascending
    for (int j0 = 0; j0 < nmax; j0 += 4) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = (own && j0 + u < n && !scale) ? blk[(j0 + u) * n + i] : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = j0 + u;
            const double sj = __shfl_sync(FULL, s, j & (W - 1), W);
            if (own && j < n) bs += (scale ? (j == i ? sc : 0.0) : v[u]) * sj;
        }
    }
    const double sBs = gsum<W>(s * bs);
    const double th = sy >= 0.2 * sBs ? 1.0 : 0.8 * sBs / (sBs - sy);
    const double r = th * y + (1.0 - th) * bs;
    const double sr = gsum<W>(s * r);
    ok = ok && isfinite(sBs) && isfinite(sr) && sBs > 0.0 && sr > 0.0;
    // B <- B - (Bs)(Bs)'/s'Bs + r r'/s'r: lane i writes column i (bitwise symmetric: both triangles form the same products)
    for (int j0 = 0; j0 < nmax; j0 += 4) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = (ok && own && j0 + u < n && !scale) ? blk[(j0 + u) * n + i] : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = j0 + u;
            const double bsj = __shfl_sync(FULL, bs, j & (W - 1), W), rj = __shfl_sync(FULL, r, j & (W - 1), W);
            if (ok && own && j < n) {
                const double old = scale ? (j == i ? sc : 0.0) : v[u];
                blk[j * n + i] = old - (bsj * bs) / sBs + (rj * r) / sr;
            }
        }
    }
    if (ok && i == 0) *upd = 1;
}

template <int W>
__global__ void __launch_bounds__(128) k_qn_update(const dto_sqp_args a)
{
    const int i = threadIdx.x & (W - 1);
    const int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / W;   // (problem, knot) of this group
    const bool live = gid < a.B * a.T;
    const int64_t b = live ? gid / a.T : 0;
    const int t = live ? (int)(gid - b * a.T) : 0;
    const int n = live ? a.kdim[t] : 0;
    const bool own = i < n;
    const int zc = a.kofs[t] + i;                                  // variable of row i
    // s_i and y_i = (g + J'lam)_i - (gp + Jp'lam)_i (pinned variables masked out); z, g and J become the previous ones
    double s = 0.0, y = 0.0;
    if (own) {
        const int64_t zi = b * a.N_z + zc;
        const double f = a.free[zc];
        const double zn = a.z[zi], zo = a.zp[zi], gn = a.bg[zi], go = a.gp[zi];
        const double* __restrict__ lam = a.lam + b * a.N_c;
        const double* __restrict__ Jn = a.bJ + b * a.nnz_J;
        double* __restrict__ Jo = a.Jp + b * a.nnz_J;
        double jl = 0.0, jlp = 0.0;
        const int q1 = a.colptr[zc + 1];
        for (int q0 = a.colptr[zc]; q0 < q1; q0 += 4) {
            int sl[4];
            double vl[4], vn[4], vo[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool in = q0 + u < q1;
                sl[u] = in ? a.colslot[q0 + u] : 0;
                vl[u] = in ? lam[a.colrow[q0 + u]] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                vn[u] = q0 + u < q1 ? Jn[sl[u]] : 0.0;
                vo[u] = q0 + u < q1 ? Jo[sl[u]] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (q0 + u < q1) {
                    jl += vn[u] * vl[u];
                    jlp += vo[u] * vl[u];
                    Jo[sl[u]] = vn[u];
                }
        }
        s = (zn - zo) * f;
        y = ((gn + jl) - (go + jlp)) * f;
        a.zp[zi] = zn;
        a.gp[zi] = gn;
    }
    if (a.it == 0) return;   // (uniform over the launch) the previous point is the one just stored
    qn_block_update<W>(a.blocks + b * a.nnz_blk + (live ? a.boff[t] : 0), n, i, live, s, y, a.qn_updated + b * a.T + t);
}


// =====================================================================================================================
// Partitioned damped BFGS (hessian_approximation = 2; sqp.py `PARTITIONED_BFGS` states it): one dense symmetric block B_t
// per knot element E_t over v_t = [x_t; u_t; x_{t+1}] (the last knot: x_T), a contiguous range of z. A group of W lanes
// owns one (problem, element), lane i variable i of v_t. s_t = P_t (z - z_prev); y_t = the change of the element's gradient:
// g + the J'lam terms of the rows of d_t and stage_t on [x_t; u_t], the J'lam terms of d_t's rows on x_{t+1}. The J'lam
// terms go over the element's own column table (ecolptr/ecolslot/ecolrow, rows ascending), so every J slot has one owning
// lane, which refreshes J_prev in place as k_qn_update does.
// The previous point: element t reads z_prev on x_{t+1}, which element t+1 owns and would rewrite in the same launch. So z
// alternates between two buffers by iteration parity: iteration `it` stores z into buffer it & 1 (owner lanes, i < n_t, only)
// and reads z_prev from the other one, which no lane writes in this launch. g_prev is read and written on [x_t; u_t] only,
// by the owner lane.
// =====================================================================================================================
template <int W>
__global__ void __launch_bounds__(128) k_pqn_update(const dto_sqp_args a)
{
    const int i = threadIdx.x & (W - 1);
    const int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / W;   // (problem, element) of this group
    const bool live = gid < a.B * a.T;
    const int64_t b = live ? gid / a.T : 0;
    const int t = live ? (int)(gid - b * a.T) : 0;
    const int m = live ? a.edim[t] : 0, n = live ? a.kdim[t] : 0;
    const bool own = i < m;
    const int zc = a.kofs[t] + i;                                  // variable i of v_t
    double* __restrict__ blk = a.eblocks + b * a.nnz_el + (live ? a.eoff[t] : 0);
    double* __restrict__ zcur = (a.it & 1) ? a.zp2 : a.zp;
    const double* __restrict__ zprev = (a.it & 1) ? a.zp : a.zp2;
    double s = 0.0, y = 0.0;
    if (own) {
        const int64_t zi = b * a.N_z + zc;
        const double f = a.free[zc];
        const double zn = a.z[zi], zo = zprev[zi];
        const double* __restrict__ lam = a.lam + b * a.N_c;
        const double* __restrict__ Jn = a.bJ + b * a.nnz_J;
        double* __restrict__ Jo = a.Jp + b * a.nnz_J;
        double jl = 0.0, jlp = 0.0;
        const int e = a.evar[t] + i;
        const int q1 = a.ecolptr[e + 1];
        for (int q0 = a.ecolptr[e]; q0 < q1; q0 += 4) {
            int sl[4];
            double vl[4], vn[4], vo[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const bool in = q0 + u < q1;
                sl[u] = in ? a.ecolslot[q0 + u] : 0;
                vl[u] = in ? lam[a.ecolrow[q0 + u]] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                vn[u] = q0 + u < q1 ? Jn[sl[u]] : 0.0;
                vo[u] = q0 + u < q1 ? Jo[sl[u]] : 0.0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (q0 + u < q1) {
                    jl += vn[u] * vl[u];
                    jlp += vo[u] * vl[u];
                    Jo[sl[u]] = vn[u];
                }
        }
        s = (zn - zo) * f;
        if (i < n) {   // [x_t; u_t]: the cost's gradient too; these lanes own z_prev and g_prev of their variable
            const double gn = a.bg[zi], go = a.gp[zi];
            y = ((gn + jl) - (go + jlp)) * f;
            zcur[zi] = zn;
            a.gp[zi] = gn;
        } else {
            y = (jl - jlp) * f;
        }
    }
    if (a.it == 0) {   // (uniform over the launch) every solve and continuation stage starts from identity element blocks
        if (own)
            for (int j = 0; j < m; ++j) blk[j * m + i] = j == i ? 1.0 : 0.0;
        return;
    }
    qn_block_update<W>(blk, m, i, live, s, y, a.qn_updated + b * a.T + t);
}

// H of K from the element blocks: chain row block t (rows [x_t; u_t], columns [x_t; u_t; x_{t+1}], dense row-major) is
// B_t[0:n_t, :], plus the x_t x x_t tail of B_{t-1} on its x_t x x_t corner (in that order: sqp.py sums the same way).
// Lane j writes column j; no two groups write the same entry.
template <int W>
__global__ void __launch_bounds__(128) k_pqn_assemble(const dto_sqp_args a)
{
    const int j = threadIdx.x & (W - 1);
    const int64_t gid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / W;
    if (gid >= a.B * a.T) return;
    const int64_t b = gid / a.T;
    const int t = (int)(gid - b * a.T);
    const int m = a.edim[t], n = a.kdim[t];
    if (j >= m) return;
    const double* __restrict__ E = a.eblocks + b * a.nnz_el + a.eoff[t];
    double* __restrict__ C = a.blocks + b * a.nnz_blk + a.boff[t];
    const int mp = t > 0 ? a.edim[t - 1] : 0, np = t > 0 ? a.kdim[t - 1] : 0;
    const int nx = mp - np;                                        // x_t: the tail of element t - 1
    const double* __restrict__ P = a.eblocks + b * a.nnz_el + (t > 0 ? a.eoff[t - 1] + np * mp + np : 0);
    for (int r = 0; r < n; ++r) {
        double v = E[r * m + j];
        if (r < nx && j < nx) v += P[r * mp + j];
        C[r * m + j] = v;
    }
}

template <class K, class... Args>
int launch_warp_per(K kernel, int64_t n, void* stream, Args... args)
{
    if (n <= 0) return 0;
    kernel<<<(unsigned)((n + 3) / 4), 128, 0, (cudaStream_t)stream>>>(args...);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : -(int)e;
}

}  // namespace

extern "C" int dto_sqp_k_begin(const dto_sqp_args* a, void* s) { return launch_warp_per(k_begin, a->B, s, *a); }
extern "C" int dto_sqp_k_set_lam(const dto_sqp_args* a, void* s) { return launch_warp_per(k_set_lam, a->B, s, *a); }
extern "C" int dto_sqp_k_after_first(const dto_sqp_args* a, void* s) { return launch_warp_per(k_after_first, a->B, s, *a); }
extern "C" int dto_sqp_k_reg_next(const dto_sqp_args* a, void* s)
{
    if (a->B <= 0) return 0;
    k_reg_next<<<(unsigned)((a->B + 127) / 128), 128, 0, (cudaStream_t)s>>>(*a);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : -(int)e;
}
extern "C" int dto_sqp_k_recheck(const dto_sqp_args* a, int32_t count, void* s) { return launch_warp_per(k_recheck, count, s, *a, count); }
extern "C" int dto_sqp_k_direction(const dto_sqp_args* a, void* s) { return launch_warp_per(k_direction, a->B, s, *a); }
extern "C" int dto_sqp_k_ls_round(const dto_sqp_args* a, int32_t round, void* s) { return launch_warp_per(k_ls_round, a->B, s, *a, round); }
extern "C" int dto_sqp_k_soc_trial(const dto_sqp_args* a, int32_t count, void* s) { return launch_warp_per(k_soc_trial, count, s, *a, count); }
extern "C" int dto_sqp_k_soc_accept(const dto_sqp_args* a, int32_t count, void* s) { return launch_warp_per(k_soc_accept, count, s, *a, count); }
extern "C" int dto_sqp_k_end(const dto_sqp_args* a, void* s) { return launch_warp_per(k_end, a->B, s, *a); }
extern "C" int dto_sqp_k_multi_trial(const dto_sqp_args* a, int32_t count, int32_t R, void* s)
{
    return launch_warp_per(k_multi_trial, (int64_t)count * R, s, *a, count, R);
}
extern "C" int dto_sqp_k_multi_pick(const dto_sqp_args* a, int32_t count, int32_t R, void* s) { return launch_warp_per(k_multi_pick, count, s, *a, count, R); }
extern "C" int dto_sqp_k_reg_ladder(const dto_sqp_args* a, int32_t m, void* s)
{
    if (a->B <= 0) return 0;
    k_reg_ladder<<<(unsigned)((a->B + 127) / 128), 128, 0, (cudaStream_t)s>>>(*a, m);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : -(int)e;
}
extern "C" int dto_sqp_k_reg_pick(const dto_sqp_args* a, int32_t count, int32_t m, void* s)
{
    if (count <= 0) return 0;
    k_pick<<<(unsigned)count, 256, 0, (cudaStream_t)s>>>(*a, count, m);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : -(int)e;
}
extern "C" int dto_sqp_k_ip_prepare(const dto_sqp_args* a, void* s) { return launch_warp_per(a->bstride ? k_ip_prepare<true> : k_ip_prepare<false>, a->B, s, *a); }
extern "C" int dto_sqp_k_ip_after_first(const dto_sqp_args* a, void* s) { return launch_warp_per(a->bstride ? k_ip_after_first<true> : k_ip_after_first<false>, a->B, s, *a); }
extern "C" int dto_sqp_k_ip_direction(const dto_sqp_args* a, void* s) { return launch_warp_per(a->bstride ? k_ip_direction<true> : k_ip_direction<false>, a->B, s, *a); }
extern "C" int dto_sqp_k_ip_ls_round(const dto_sqp_args* a, int32_t round, void* s)
{
    return launch_warp_per(a->bstride ? k_ip_ls_round<true> : k_ip_ls_round<false>, a->B, s, *a, round);
}
extern "C" int dto_sqp_k_ip_end(const dto_sqp_args* a, void* s) { return launch_warp_per(a->bstride ? k_ip_end<true> : k_ip_end<false>, a->B, s, *a); }
extern "C" int dto_sqp_k_qn_update(const dto_sqp_args* a, void* s)
{
    const int64_t threads = a->B * a->T * a->qn_W;
    if (threads <= 0) return 0;
    const unsigned grid = (unsigned)((threads + 127) / 128);
    if (a->qn_W == 16)
        k_qn_update<16><<<grid, 128, 0, (cudaStream_t)s>>>(*a);
    else
        k_qn_update<32><<<grid, 128, 0, (cudaStream_t)s>>>(*a);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : -(int)e;
}
extern "C" int dto_sqp_k_pqn_update(const dto_sqp_args* a, void* s)
{
    const int64_t threads = a->B * a->T * a->qn_W;
    if (threads <= 0) return 0;
    const unsigned grid = (unsigned)((threads + 127) / 128);
    if (a->qn_W == 16)
        k_pqn_update<16><<<grid, 128, 0, (cudaStream_t)s>>>(*a);
    else
        k_pqn_update<32><<<grid, 128, 0, (cudaStream_t)s>>>(*a);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : -(int)e;
}
extern "C" int dto_sqp_k_pqn_assemble(const dto_sqp_args* a, void* s)
{
    const int64_t threads = a->B * a->T * a->qn_W;
    if (threads <= 0) return 0;
    const unsigned grid = (unsigned)((threads + 127) / 128);
    if (a->qn_W == 16)
        k_pqn_assemble<16><<<grid, 128, 0, (cudaStream_t)s>>>(*a);
    else
        k_pqn_assemble<32><<<grid, 128, 0, (cudaStream_t)s>>>(*a);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 0 : -(int)e;
}

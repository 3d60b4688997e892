/* dto_sqp_dev.h -- launch interface between the host runtime (dto_runtime.cpp, g++) and the per-problem bookkeeping
 * kernels of the native lock-step Newton-KKT solver (dto_sqp.cu, nvcc). Plain C. The heavy work of an iteration is
 * done by the callback kernels (model library) and the KKT kernels (dto_kkt.cu); the kernels here are the O(B N)
 * glue between them: row reductions, step / merit bookkeeping, masks, trial points. */
#ifndef DTO_SQP_DEV_H
#define DTO_SQP_DEV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dto_sqp_params {   /* SQPOptions of sqp.py, same meaning */
    double tol_constraint, tol_dual;
    double reg_first, reg_min, reg_max, reg_inc_first, reg_inc, reg_dec;
    double armijo, merit_margin, merit_rho, merit_min;
    double lm_first, lm_min, lm_grow, lm_shrink, lm_grow_below, lm_zero;
    double exact_below, lam_max;
    int32_t soc;
    int32_t max_refactor;   /* inertia-correction tries per problem and iteration */
    /* interior-point mode (inequality bounds on variables, inequality rows c_i(z) <= 0) */
    int32_t ip, any_ineq;
    double mu_floor, kappa_eps, kappa_mu, theta_mu, tau_min, kappa_sigma, tiny_step, bound_push;
} dto_sqp_params;

enum { DTO_SQP_N_DONE = 0, DTO_SQP_N_BAD = 1, DTO_SQP_N_IDX = 2, DTO_SQP_N_NEED = 3, DTO_SQP_N_OPEN = 4, DTO_SQP_N_SOC_OK = 5,
       DTO_SQP_N_RETRY = 6 /* bad problems that still have tries left */, DTO_SQP_N_ACTIVE = 7 /* not converged */,
       DTO_SQP_N_COUNTERS = 8 };

typedef struct dto_sqp_args {
    int64_t B;
    int32_t N_z, N_c, dim, it;
    dto_sqp_params p;
    /* arrays of the batch and of its KKT handle (device) */
    double* bz;           /* [B][N_z]  the z the callback kernels read                          */
    double* blam;         /* [B][N_c]  the lambda the Hessian / right-hand-side kernels read   */
    const double* bf;     /* [B]       objective                                               */
    const double* bg;     /* [B][N_z]  gradient                                                */
    double* bc;           /* [B][N_c]  constraint values (overwritten by trial evaluations)    */
    double* rhs;          /* [B][dim]  [g + J'lam ; c] (a second-order correction rewrites its c part) */
    const double* sol;    /* [B][dim]  K^-1 rhs                                                */
    double* preg;         /* [B]       per-problem primal regularisation read by the factor kernel */
    const int32_t* nneg;  /* [B]       negative pivots of the last factorisation              */
    /* solver state (device) */
    double *z, *lam, *dz, *dlam, *ckeep;
    double *delta, *delta_last, *nu, *lm, *exact, *alpha, *phi0, *slope, *c1, *fcur, *cv, *dr;
    int32_t* iters;
    uint8_t *done, *bad, *accepted, *first, *need;
    const double* free;   /* [N_z] 1 = free variable, 0 = pinned by equal bounds               */
    int32_t* counters;    /* [DTO_SQP_N_COUNTERS]                                              */
    int32_t* idx;         /* [B] problem list of a subset launch                               */
    int32_t* oidx;        /* [B] problems whose line search is still open after a round        */
    /* trial slots: the remaining step lengths of the open problems evaluated in one pass */
    int32_t N_w;
    const double* w;      /* [B][N_w] per-problem parameters of the batch                      */
    double *tz, *tw, *tf, *tc;   /* [cap][N_z], [cap][N_w], [cap], [cap][N_c]                  */
    /* candidate slots of the inertia correction: several regularisations of a problem factorised at once */
    int32_t* vidx;        /* [V] problem of candidate slot v                                   */
    double* vreg;         /* [V] its regularisation                                            */
    double* vsol;         /* [V][dim]                                                          */
    int32_t* vnneg;       /* [V]                                                               */
    double* vL;           /* [V][factor_stride]                                                */
    double* L;            /* [B][factor_stride] the batch's factors (the chosen candidate's is copied here) */
    double* sol_w;        /* = sol, writable                                                   */
    int32_t* nneg_w;      /* = nneg, writable                                                  */
    int64_t factor_stride;
    int32_t* tries;       /* [B] inertia-correction tries used by the problem in this iteration */
    int32_t* alist;       /* [B] problems that have not converged (written by the first check, for the next iteration) */
    /* interior-point mode */
    const double *hasL, *hasU;             /* [N_z] 0/1 masks (one bound pattern per batch)                     */
    const double *lo, *up;                 /* finite bound values (0 where absent): problem b's at lo + b * bstride */
    int64_t bstride;                       /* 0: one [N_z] pair for every problem; N_z: [B][N_z]                  */
    const double* hasI;                    /* [N_c] 1 = inequality row c_i(z) <= 0                              */
    double *zL, *zU, *dzL, *dzU;           /* [B][N_z] bound multipliers and their steps                        */
    double *t, *dt;                        /* [B][N_c] slacks of the inequality rows and their steps            */
    double *mu, *mu_next, *amax, *a_z, *fbar;   /* [B] barrier parameter, step limits, barrier value at z      */
    double* diag;                          /* [B][dim] the diagonal the factor kernel adds to K                 */
    double* bg_w;                          /* = bg, writable (the barrier gradient is added to g)               */
    /* knot-block damped BFGS (hessian_approximation = 1): block t of a problem covers z[kofs[t], kofs[t] + kdim[t]) and is a
     * dense row-major kdim[t]^2 matrix at offset boff[t] of the problem's nnz_blk block values */
    int32_t T, qn_W;                       /* knots; lanes per block (16: two blocks per warp, or 32)           */
    int32_t nnz_blk, nnz_J;
    const int32_t *kofs, *kdim, *boff;     /* [T]                                                               */
    double* blocks;                        /* [B][nnz_blk] the KKT handle's blocks (H of K)                     */
    const double* bJ;                      /* [B][nnz_J] Jacobian of the callbacks                              */
    const int32_t *colptr, *colslot, *colrow;   /* the KKT handle's Jacobian-by-column tables (J'lam, rows ascending) */
    double *zp, *gp, *Jp;                  /* z, g, J of the previous iteration                                */
    uint8_t* qn_updated;                   /* [B][T] 1 once a block has taken an update (the first one is scaled) */
    /* partitioned damped BFGS (hessian_approximation = 2): element t covers z[kofs[t], kofs[t] + edim[t]) = [x_t; u_t; x_{t+1}]
     * (the last knot: x_T) and is a dense row-major edim[t]^2 matrix at offset eoff[t] of the problem's nnz_el element values;
     * T, qn_W, kofs, kdim (= n_t), bJ, Jp, gp and qn_updated (one flag per element) as above; blocks / nnz_blk / boff: the KKT
     * handle's chain array, row block t (kdim[t] x edim[t]) at offset boff[t] */
    const int32_t *edim, *eoff, *evar;     /* [T]; evar[t] = sum_{s<t} edim[s]: element t's first entry of ecolptr         */
    int32_t nnz_el;
    double* eblocks;                       /* [B][nnz_el]                                                       */
    const int32_t *ecolptr, *ecolslot, *ecolrow;   /* [sum_t edim[t] + 1], [nnz_J], [nnz_J]: J entries of the rows of d_t and
                                                      stage_t by variable of v_t, rows ascending                     */
    double* zp2;                           /* [B][N_z] z_prev of odd iterations (zp: even ones)                 */
} dto_sqp_args;

/* each returns 0 or -(cudaError_t) */
int dto_sqp_k_begin(const dto_sqp_args* a, void* stream);        /* bz = z, blam = lam * exact, preg = delta = lm            */
int dto_sqp_k_set_lam(const dto_sqp_args* a, void* stream);      /* blam = lam                                              */
int dto_sqp_k_after_first(const dto_sqp_args* a, void* stream);  /* cv, dr, exact, done, bad, ckeep, counters              */
int dto_sqp_k_reg_next(const dto_sqp_args* a, void* stream);     /* next regularisation of the bad problems + their index list */
int dto_sqp_k_recheck(const dto_sqp_args* a, int32_t count, void* stream);  /* bad again? for the idx list                    */
int dto_sqp_k_direction(const dto_sqp_args* a, void* stream);    /* dz, dlam, merit quantities, first trial point          */
int dto_sqp_k_ls_round(const dto_sqp_args* a, int32_t round, void* stream);
int dto_sqp_k_soc_trial(const dto_sqp_args* a, int32_t count, void* stream);
int dto_sqp_k_soc_accept(const dto_sqp_args* a, int32_t count, void* stream);
int dto_sqp_k_end(const dto_sqp_args* a, void* stream);
/* the next m regularisations of every bad problem (the values m sequential tries would use) into candidate slots k*m + j */
int dto_sqp_k_reg_ladder(const dto_sqp_args* a, int32_t m, void* stream);
/* per bad problem: the first candidate with the right inertia and a finite solution is kept (factor and solution copied) */
int dto_sqp_k_reg_pick(const dto_sqp_args* a, int32_t count, int32_t m, void* stream);
/* interior-point mode: the same iteration with barrier terms (separate kernels: the equality-only path above stays as it is) */
int dto_sqp_k_ip_prepare(const dto_sqp_args* a, void* stream);      /* after the callbacks: diag, g += barrier gradient, c shifted, residual, barrier value */
int dto_sqp_k_ip_after_first(const dto_sqp_args* a, void* stream);
int dto_sqp_k_ip_direction(const dto_sqp_args* a, void* stream);
int dto_sqp_k_ip_ls_round(const dto_sqp_args* a, int32_t round, void* stream);
int dto_sqp_k_ip_end(const dto_sqp_args* a, void* stream);
/* knot-block damped BFGS: update every block from s = z - zp, y = (g + J'lam) - (gp + Jp'lam), then zp, gp, Jp = z, g, J */
int dto_sqp_k_qn_update(const dto_sqp_args* a, void* stream);
/* partitioned damped BFGS: update every element block from its s_t, y_t (identity element blocks at it = 0), then z, g, J
 * become the previous ones */
int dto_sqp_k_pqn_update(const dto_sqp_args* a, void* stream);
/* chain row blocks (H of K) from the element blocks */
int dto_sqp_k_pqn_assemble(const dto_sqp_args* a, void* stream);
/* slot k * R + j (k-th entry of oidx, j < R) <- z + alpha 2^-j dz and the problem's parameters */
int dto_sqp_k_multi_trial(const dto_sqp_args* a, int32_t count, int32_t R, void* stream);
/* per open problem: the first j whose trial passes the Armijo test is taken, as R sequential rounds would */
int dto_sqp_k_multi_pick(const dto_sqp_args* a, int32_t count, int32_t R, void* stream);

#ifdef __cplusplus
}
#endif
#endif

/* dto_kkt_dev.h -- launch interface between the host runtime (dto_runtime.cpp, g++) and the KKT
 * kernels (dto_kkt.cu, nvcc). Plain C. */
#ifndef DTO_KKT_DEV_H
#define DTO_KKT_DEV_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dto_kkt_args {
    int64_t B;           /* problems of this shard                                            */
    int32_t dim;         /* N_z + N_c                                                          */
    int32_t N_z, N_c;
    int32_t nnz_J, nnz_H;
    int32_t W;           /* band entries kept per row = rows per block = lanes per problem (16 or 32) */
    int32_t bw;          /* half bandwidth of the ordered matrix (<= W - 1)                    */
    int32_t nblk;        /* ceil(dim / W) row blocks                                           */
    int64_t factor_stride; /* doubles of factor storage per problem: nblk*W*LW + nblk*W, LW = dto_kkt_col_width */
    /* callback outputs / inputs of the shard (problem-major) */
    const double* H;     /* [B][nnz_H]  */
    const double* J;     /* [B][nnz_J]  */
    const double* g;     /* [B][N_z]    */
    const double* c;     /* [B][N_c]    */
    const double* y;     /* [B][N_c] multipliers (lambda)                                      */
    /* static tables, shared by all problems */
    const int32_t* src;    /* [nblk][W][W] value source of band slot (row block, column mod W, row in block):
                              < nnz_H -> H, else J, -1 structural zero                               */
    const double* dreg;    /* [nblk*W] diagonal shift: +primal_reg, -dual_reg, 1.0 on padding rows   */
    const int32_t* iperm;  /* [nblk*W] original (0-based) index of permuted row, -1 on padding       */
    const int32_t* colptr; /* [N_z+1] Jacobian by column ...                                         */
    const int32_t* colslot;/* [nnz_J] ... slot in J, rows ascending                                  */
    const int32_t* colrow; /* [nnz_J] ... constraint row (0-based)                                   */
    /* work / outputs */
    double* rhs;         /* [B][dim] h = [grad f + J'y ; c], natural order                     */
    double* L;           /* [B][factor_stride]: per problem [nblk*W][LW] columns of L (slot 0 = pivot d_j,
                            slot q = L(j+q, j)) followed by [nblk*W] D^-1 L^-1 h                 */
    double* sol;         /* [B][dim] K^-1 h, natural order                                     */
    /* per-problem primal regularisation (inertia control of a solver driving the batch): when non-NULL the
     * diagonal shift of the VARIABLE rows of problem b is preg[b] instead of the scalar primal_reg          */
    const double* preg;  /* [B] or NULL                                                        */
    int32_t* nneg;       /* [B] or NULL: number of negative pivots of D (inertia; N_c when K is quasi-definite) */
    /* subset launch (a solver re-factorising only the problems whose inertia was wrong): when non-NULL, slot s of
     * the launch works on problem pidx[s] and B is the number of slots; every array above stays indexed by problem */
    const int32_t* pidx; /* [B] or NULL                                                        */
    /* candidate launch (several regularisations of the same problem tried at once): with virt = 1 and pidx given, slot s
     * READS problem pidx[s] (H, J, rhs) but its regularisation preg[s], factor L[s], solution sol[s] and pivot count
     * nneg[s] are indexed by the SLOT: the caller passes scratch arrays there and keeps the candidate it wants */
    int32_t virt;
    double primal_reg, dual_reg;   /* the scalars behind the dreg table (+primal_reg on variable rows, -dual_reg on constraint rows) */
    /* per-problem diagonal added to K, natural order [variables; constraint rows] (an interior-point solver's barrier terms:
     * Sigma = z_L / (x - l) + z_U / (u - x) on the variables, -t_i / lambda_i on inequality rows): K(i, i) += diag[b][i];
     * NULL = none */
    const double* diag;  /* [B][dim] or NULL                                                   */
    /* variables pinned by equal lower/upper bounds (Bound(state_lower = x1, state_upper = x1), test/solve.jl): their
     * rows and columns of K are replaced by the identity (the gather table carries structural zeros there) and their
     * right-hand-side entries by 0, so their step is exactly 0 and the others get the reduced Newton step */
    const uint8_t* fixed;    /* [N_z] or NULL: 1 = pinned variable                             */
    const uint8_t* rowfixed; /* [nblk*W] or NULL: 1 = permuted row belongs to a pinned variable (diagonal shift 1.0)  */
} dto_kkt_args;

/* The factor kernel is instantiated for a few bounds BW on the half bandwidth; a column of L is stored
 * as LW = BW + 1 doubles rounded up to even (pivot, then L(j+1..j+BW, j)), so both sides must agree: */
static inline int dto_kkt_bw_bound(int W, int bw)
{
    if (W == 16) return bw <= 6 ? 6 : bw <= 9 ? 9 : bw <= 12 ? 12 : 15;
    return bw <= 20 ? 20 : 31;
}
static inline int dto_kkt_col_width(int W, int bw) { return (dto_kkt_bw_bound(W, bw) + 2) & ~1; }

/* each returns the number of kernels enqueued (>= 0) or -(cudaError_t) */
int dto_kkt_launch_rhs(const dto_kkt_args* a, void* stream);
int dto_kkt_launch_band(const dto_kkt_args* a, void* stream);
int dto_kkt_launch_resolve(const dto_kkt_args* a, void* stream);   /* solve again with the stored factor */
int dto_kkt_launch_assemble(const dto_kkt_args* a, int64_t problem, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif

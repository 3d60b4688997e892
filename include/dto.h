/* dto.h -- C ABI of the B200-native batched NLP-callback engine (libdto.so).
 *
 * Drop-in boundary for the ONE hot path of thowell/DirectTrajectoryOptimization.jl: the five
 * MathOptInterface evaluator callbacks of /root/reference/src/moi.jl and the two structure
 * queries, evaluated for a batch of B independent problems of one shape on one or more B200s.
 * Plain C: opaque handles, pointers and sizes only. Every entry point names the reference
 * interface it replaces. Julia binds these with `ccall` (see INTEGRATION.md).
 *
 * Conventions
 *   - all values are IEEE double; all indices handed OUT are int64 and 1-based (Julia Int),
 *     in exactly the reference's order; indices handed IN (knot kinds) are 0-based ints.
 *   - batched arrays are problem-major and dense: z[B][num_variables], lambda[B][num_constraint],
 *     J[B][num_jacobian], H[B][num_hessian] ... problem b of a batch lives on device b / ceil(B/ndev).
 *   - every function returns 0 on success or a negative dto_status; the message is available
 *     from dto_last_error() (thread-local). Nothing aborts or throws across this boundary;
 *     NaN/Inf values pass through unchanged, like the reference.
 *   - the caller owns every host pointer; calls taking host pointers return after the copy
 *     has completed. The library owns all device memory. A dto_batch may be used from one
 *     host thread at a time; distinct batches are independent.
 *   - there is NO CPU fallback: without a CUDA device dto_batch_create fails with
 *     DTO_ERR_CUDA. Shape/structure queries are host-only and work without a GPU.
 */
#ifndef DTO_H
#define DTO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTO_ABI_VERSION 1

typedef enum dto_status {
    DTO_OK = 0,
    DTO_ERR_BAD_ARG = -1,      /* null pointer, size mismatch, inconsistent shape description */
    DTO_ERR_CUDA = -2,         /* CUDA runtime error (message carries cudaGetErrorString)      */
    DTO_ERR_OOM = -3,          /* host or device allocation failed                             */
    DTO_ERR_MODEL = -4,        /* model library missing / wrong ABI / not compiled             */
    DTO_ERR_NO_HESSIAN = -5,   /* Hessian requested but a Cost was built without evaluate_hessian
                                  (the reference throws here: src/costs.jl:68, SURVEY Q9)      */
    DTO_ERR_STATE = -6,        /* e.g. evaluation requested before dto_set_x                   */
    DTO_ERR_UNSUPPORTED = -7   /* the shape is outside what a kernel covers (e.g. KKT bandwidth) */
} dto_status;

typedef struct dto_model dto_model; /* a loaded generated model library (element device code)   */
typedef struct dto_shape dto_shape; /* static tables of one problem shape (reference: NLPData's
                                       indices/sparsity fields, src/data.jl:106-121)            */
typedef struct dto_batch dto_batch; /* B problems of one shape resident on 1..n devices         */
typedef struct dto_kkt dto_kkt;     /* device-resident KKT systems of a batch (consumer of J, H)  */

/* Description of one problem shape in terms of the model library's element kinds.
 * Mirrors the arguments of Solver(dynamics, objective, constraints, bounds; general_constraint,
 * parameters) (/root/reference/src/solver.jl:6-10): which Dynamics/Cost/Constraint object sits at
 * which knot. */
typedef struct dto_shape_desc {
    int32_t T;                    /* horizon: number of knots (length(objective))                  */
    const int32_t* dynamics_kind; /* [T-1] kind of dynamics[t]                                     */
    const int32_t* cost_kind;     /* [T]   kind of objective[t]                                    */
    const int32_t* stage_kind;    /* [T]   kind of constraints[t]; -1 = empty Constraint()         */
    int32_t use_general;          /* 1: attach the model's GeneralConstraint block                 */
    /* Per-knot parameter vectors w_t are slices [parameter_offset[t], +nw_t) of each problem's
     * flat parameter vector of length num_parameter. NULL = the reference's layout
     * vcat(parameters...) (src/data.jl:218): offsets are prefix sums of parameter_dim. Overlapping
     * slices let all knots of a problem share one small vector (e.g. w = [x1; xT]). */
    const int32_t* parameter_dim;    /* [T] length of w_t (NULL = all zero)                        */
    const int32_t* parameter_offset; /* [T] or NULL                                                */
    int32_t num_parameter;           /* per-problem flat parameter length (ignored when
                                        parameter_offset is NULL: then it is sum(parameter_dim))   */
} dto_shape_desc;

/* ---- library ---- */
int dto_abi_version(void);
const char* dto_last_error(void);
const char* dto_status_string(int status);
/* number of CUDA devices visible (0 without a GPU / driver; never fails) */
int dto_device_count(void);

/* ---- model library: generated element code (replaces the eval'd closures in the ::Any fields
 * of Dynamics/Cost/Constraint/GeneralConstraint, src/dynamics.jl:2-4 etc.) ---- */
int dto_model_load(const char* path, dto_model** out);
void dto_model_destroy(dto_model* m);
const char* dto_model_name(const dto_model* m);
const char* dto_model_hash(const dto_model* m);
/* role: 0 dynamics, 1 cost, 2 stage constraint */
int dto_model_num_kinds(const dto_model* m, int role);
/* dims[0..5] = n_out (num_next_state | 1 | num_constraint), num_state, num_action, num_parameter,
 * num_jacobian (cost: num_gradient), num_hessian */
int dto_model_kind_dims(const dto_model* m, int role, int kind, int32_t dims[6]);
int dto_model_has_general(const dto_model* m);

/* ---- shape: replaces NLPData(trajopt; ...) assembly, src/data.jl:150-220, in O(nnz log nnz) ---- */
int dto_shape_create(dto_model* m, const dto_shape_desc* desc, dto_shape** out);
void dto_shape_destroy(dto_shape* s);
int64_t dto_num_variables(const dto_shape* s);          /* nlp.num_variables      src/data.jl:155   */
int64_t dto_num_constraint(const dto_shape* s);         /* nlp.num_constraint     src/data.jl:158-161 */
int64_t dto_num_jacobian(const dto_shape* s);           /* nlp.num_jacobian       src/data.jl:164-167 */
int64_t dto_num_hessian(const dto_shape* s);            /* length(nlp.hessian_lagrangian_sparsity), src/data.jl:184 */
int64_t dto_num_hessian_nonunique(const dto_shape* s);  /* nlp.num_hessian_lagrangian src/data.jl:187 (Q4) */
int64_t dto_num_parameter(const dto_shape* s);          /* per-problem flat parameter length          */
int dto_hessian_available(const dto_shape* s);          /* every Cost kind carries a Hessian (Q9)     */
/* MOI.jacobian_structure (src/moi.jl:124): rows/cols[num_jacobian], 1-based, reference order */
int dto_jacobian_structure(const dto_shape* s, int64_t* rows, int64_t* cols);
/* MOI.hessian_lagrangian_structure (src/moi.jl:125): sorted unique (row, col), both triangles */
int dto_hessian_lagrangian_structure(const dto_shape* s, int64_t* rows, int64_t* cols);
/* constraint_bounds (src/data.jl:135-148): lower/upper[num_constraint]; inequality rows (-Inf, 0] */
int dto_constraint_bounds(const dto_shape* s, double* lower, double* upper);
/* z-layout (src/dynamics.jl:188-195): 1-based index of x_t[1] / u_t[1] and the dims, t = 0..T-1 */
int dto_knot_layout(const dto_shape* s, int64_t* state_start, int32_t* num_state, int64_t* action_start,
                    int32_t* num_action);

/* ---- batch ---- */
/* devices == NULL && ndev == 0: current device only. The batch is split into contiguous chunks of
 * ceil(B/ndev) problems per device (no collective on the hot path). A device may be listed more
 * than once (logical shards on one GPU). */
int dto_batch_create(dto_shape* s, int64_t B, const int* devices, int ndev, dto_batch** out);
void dto_batch_destroy(dto_batch* b);
int64_t dto_batch_size(const dto_batch* b);
int dto_batch_num_shards(const dto_batch* b);

/* inputs (host -> device). Replaces trajectory!/duals! (src/data.jl:258-278): x, lambda, sigma stay
 * device-resident between callbacks. */
int dto_set_parameters(dto_batch* b, const double* w /* [B][num_parameter] */);
int dto_set_x(dto_batch* b, const double* z /* [B][num_variables] */);
int dto_set_duals(dto_batch* b, const double* sigma /* [B] */, const double* lambda /* [B][num_constraint] */);

/* the five callbacks at the resident (z, lambda, sigma, w); results copied to host arrays */
int dto_eval_objective(dto_batch* b, double* f /* [B] */);                      /* src/moi.jl:1-13   */
int dto_eval_objective_gradient(dto_batch* b, double* g /* [B][num_variables] */);   /* src/moi.jl:15-30  */
int dto_eval_constraint(dto_batch* b, double* c /* [B][num_constraint] */);          /* src/moi.jl:32-50  */
int dto_eval_constraint_jacobian(dto_batch* b, double* J /* [B][num_jacobian] */);   /* src/moi.jl:52-70  */
int dto_eval_hessian_lagrangian(dto_batch* b, double* H /* [B][num_hessian] */);     /* src/moi.jl:72-120 */
/* Jacobian + Hessian of the Lagrangian in ONE pass over the knots (shares the element's
 * common subexpressions; the benchmark unit). Either output may be NULL to skip its copy. */
int dto_eval_jacobian_hessian(dto_batch* b, double* J, double* H);

/* The same fused pass as ONE host call: z, sigma, lambda in -- J, H out. Each shard is cut into
 * `nchunks` (<= 0: library default) contiguous sub-batches that are pipelined over several CUDA
 * streams (copy-in of chunk k+1 and copy-out of chunk k-1 overlap the kernel of chunk k, and the
 * two PCIe directions overlap each other). Host buffers should be page-locked for the overlap
 * to happen; pageable memory still works. z/sigma/lambda stay resident afterwards. */
int dto_eval_jacobian_hessian_host(dto_batch* b, const double* z, const double* sigma, const double* lambda, double* J,
                                   double* H, int nchunks);

/* one-Ipopt-per-problem drivers: copy one problem's slice of the last results (device -> host) */
typedef enum dto_array {
    DTO_ARRAY_Z = 0, DTO_ARRAY_LAMBDA = 1, DTO_ARRAY_SIGMA = 2, DTO_ARRAY_W = 3, DTO_ARRAY_F = 4,
    DTO_ARRAY_G = 5, DTO_ARRAY_C = 6, DTO_ARRAY_J = 7, DTO_ARRAY_H = 8
} dto_array;
int dto_get_problem(dto_batch* b, int array, int64_t problem, double* out);
/* host mirror of the last z handed to dto_set_x (get_trajectory semantics, src/solver.jl:41-43) */
int dto_get_last_x(const dto_batch* b, int64_t problem, double* z /* [num_variables] */);

/* ---- device-resident interface (no host copies; for device-side consumers and benchmarks) ---- */
/* device pointer of an array of shard `shard`; the shard holds problems
 * [dto_shard_begin, dto_shard_begin + dto_shard_size) */
void* dto_device_pointer(dto_batch* b, int array, int shard);
int64_t dto_shard_begin(const dto_batch* b, int shard);
int64_t dto_shard_size(const dto_batch* b, int shard);
int dto_shard_device(const dto_batch* b, int shard);
/* cudaStream_t of a shard; dto_set_stream substitutes a caller-owned stream (e.g. torch's) */
void* dto_get_stream(dto_batch* b, int shard);
int dto_set_stream(dto_batch* b, int shard, void* cuda_stream);
/* enqueue callback `kernel_id` (0 objective, 1 gradient, 2 constraint, 3 jacobian, 4 hessian,
 * 5 jacobian+hessian) on every shard's stream and return without synchronising */
int dto_launch(dto_batch* b, int kernel_id);
int dto_sync(dto_batch* b);
/* number of CUDA kernels enqueued by this batch so far (evidence counter) */
int64_t dto_launch_count(const dto_batch* b);
/* algorithmic bytes of one fused Jacobian+Hessian call per problem:
 * 8*(N_z + N_c + N_w + nnz_J + nnz_H) + 8 (SURVEY 8d) */
int64_t dto_algorithmic_bytes_per_problem(const dto_shape* s);
/* 1 if every knot of the shape matched a compiled Hessian-gather class of the model library
 * (straight-line gather, no table loads); 0 = the generic table-driven gather is used */
int dto_shape_compiled_gather(const dto_shape* s);
/* dynamic shared memory per CTA of the knot kernel for `kernel_id` */
int64_t dto_kernel_smem_bytes(const dto_shape* s, int kernel_id);

/* ---- device-side consumer of the callbacks: batched KKT assembly + LDL' (SURVEY 8f, N3) ----
 * Replaces the reference's own sketch of what is done with the callback outputs,
 * /root/reference/examples/pendulum/pendulum.jl:138-211: for every problem of the batch
 *     K = [ H + primal_reg*I   J' ; J   -dual_reg*I ],   h = [ grad f + J' lambda ; c ],
 * K = L D L' (quasi-definite: no pivoting; the example uses QDLDL), sol = K \ h -- computed from the
 * device-resident g, c, J, H, so only `sol` (N_z + N_c doubles per problem) crosses PCIe instead of
 * J and H. All problems share one bandwidth-reducing ordering computed once on the host. */
/* host-only symbolic analysis (works without a GPU): perm[p] = 1-based original index (variables
 * 1..N_z, constraint rows N_z+1..N_z+N_c) placed at position p; *bandwidth = half bandwidth of
 * the permuted matrix. Either output may be NULL. */
int dto_kkt_analyze(const dto_shape* s, int64_t* perm, int64_t* bandwidth);
/* What the H block of K is. EXACT: the Hessian of the Lagrangian from the callbacks (needs evaluate_hessian). KNOT_BLOCKS: one
 * dense symmetric block per knot over that knot's variables z[x_t; u_t] (the last knot: x_T), owned by the KKT handle and set
 * by its caller -- e.g. a quasi-Newton approximation for problems built without Hessians (the reference's evaluate_hessian =
 * false, which hands Ipopt's limited-memory mode the problem). The blocks are contiguous: block t is a dense row-major
 * n_t x n_t matrix, n_t = nx_t + nu_t, at offset sum_{s<t} n_s^2 of a problem's nnz_blk = sum_t n_t^2 values. */
#define DTO_KKT_HESSIAN_EXACT 0
#define DTO_KKT_HESSIAN_KNOT_BLOCKS 1
/* nnz_blk, and the (row, col) of every block entry, 1-based, sorted (both triangles, like dto_hessian_lagrangian_structure) */
int64_t dto_hessian_block_count(const dto_shape* s);
int dto_hessian_block_structure(const dto_shape* s, int64_t* rows, int64_t* cols);
/* dto_kkt_analyze for either Hessian structure; KNOT_BLOCKS fails with DTO_ERR_UNSUPPORTED when a knot has more than 32
 * variables or the ordered half bandwidth exceeds 31 */
int dto_kkt_analyze_ex(const dto_shape* s, int hessian, int64_t* perm, int64_t* bandwidth);
/* fails with DTO_ERR_UNSUPPORTED when the ordered half bandwidth exceeds 31. The handle borrows the
 * batch: destroy it BEFORE dto_batch_destroy(b); like the batch it is used from one host thread at a time. */
int dto_kkt_create(dto_batch* b, double primal_reg, double dual_reg, dto_kkt** out);
/* dto_kkt_create(...) = dto_kkt_create_ex(..., DTO_KKT_HESSIAN_EXACT, ...). With KNOT_BLOCKS the handle owns the blocks
 * [B][nnz_blk] (the identity at creation), the shape needs no Hessian, and every callback pass below evaluates the gradient,
 * the constraints and the Jacobian only (no Hessian pass). */
int dto_kkt_create_ex(dto_batch* b, double primal_reg, double dual_reg, int hessian, dto_kkt** out);
/* host <-> device copies of the knot blocks, [B][nnz_blk] (KNOT_BLOCKS handles only) */
int dto_kkt_set_hessian_blocks(dto_kkt* k, const double* blocks);
int dto_kkt_get_hessian_blocks(dto_kkt* k, double* blocks);
void dto_kkt_destroy(dto_kkt* k);
int64_t dto_kkt_dim(const dto_kkt* k);                       /* N_z + N_c                              */
int64_t dto_kkt_bandwidth(const dto_kkt* k);                 /* half bandwidth after ordering          */
int64_t dto_kkt_row_width(const dto_kkt* k);                 /* band entries kept per row: 16 or 32    */
int64_t dto_kkt_factor_bytes_per_problem(const dto_kkt* k);  /* factor storage written + read per solve */
int dto_kkt_permutation(const dto_kkt* k, int64_t* perm /* [dim], 1-based */);
/* gradient + constraint + fused Jacobian/Hessian callbacks at the resident (z, lambda, sigma), then
 * right-hand side, factorisation and solve; sol[B][dim] in the natural order [z; constraint rows]
 * (NULL: leave it on the device). pendulum.jl:141-211 in one call. */
int dto_kkt_solve(dto_kkt* k, double* sol);
/* the same as ONE pipelined host call: host z, lambda (and sigma; NULL = 1.0 for every problem, as in
 * pendulum.jl:136) in -- host sol out. Each shard is cut into `nchunks` (<= 0: library default)
 * sub-batches whose copy-in, kernels and copy-out overlap over several streams; page-locked host
 * buffers are needed for the overlap to happen. */
int dto_kkt_solve_host(dto_kkt* k, const double* z, const double* sigma, const double* lambda, double* sol, int nchunks);
/* the same, enqueued on the shard streams without synchronising; with_callbacks = 0 reuses the
 * g, c, J, H already on the device; with_callbacks = 2 runs the callbacks only (the caller may then change
 * lambda or c on the device before a dto_kkt_launch(k, 0): e.g. a Hessian evaluated with other multipliers
 * than the right-hand side, or a second-order-correction right-hand side) */
int dto_kkt_launch(dto_kkt* k, int with_callbacks);
/* Inertia control for a solver that drives the batch (reference: Ipopt perturbs the Hessian handed over by
 * MOI.eval_hessian_lagrangian, src/moi.jl:72, until the KKT matrix has N_c negative eigenvalues): reg[B] replaces
 * the scalar primal_reg problem by problem (NULL: back to the scalar); dto_kkt_inertia returns the number of
 * negative pivots of D per problem for the last factorisation (N_c when K is quasi-definite). */
int dto_kkt_set_primal_reg(dto_kkt* k, const double* reg /* [B] or NULL */);
/* Variables pinned by equal lower and upper bounds (Bound(state_lower = x1, state_upper = x1), /root/reference/test/solve.jl:
 * Ipopt's fixed-variable treatment): fixed[N_z], 1 = pinned, NULL = none. Their rows and columns of K become the identity
 * and their right-hand-side entries 0, so the solution holds a zero step for them and the reduced Newton step for the rest. */
int dto_kkt_set_fixed(dto_kkt* k, const uint8_t* fixed /* [num_variables] or NULL */);
/* dto_kkt_launch(k, 0) for a subset of the problems of a one-shard batch (the ones whose inertia was wrong, or that
 * need a second-order correction): idx is a DEVICE pointer to `count` int32 problem numbers; all other problems keep
 * their right-hand side, factor, solution and pivot count. */
int dto_kkt_launch_subset(dto_kkt* k, const int32_t* idx_device, int64_t count);
/* the same without factorising again: new right-hand side (the caller changed c, g or lambda on the device), forward and
 * backward solve with the factor of the last factorisation -- bit-identical to dto_kkt_launch(k, 0) as long as z, the
 * Hessian's multipliers and the regularisation are unchanged, at a fraction of its latency (second-order corrections).
 * idx_device NULL: every problem of the batch (any number of shards). */
int dto_kkt_resolve(dto_kkt* k, const int32_t* idx_device, int64_t count);
int dto_kkt_inertia(dto_kkt* k, int32_t* nneg /* [B] */);
/* which = 0: h [B][dim]; 1: sol [B][dim] (device -> host, after a solve) */
int dto_kkt_get(dto_kkt* k, int which, double* out);
/* inspection: dense row-major [dim][dim] assembled K of one problem (from the current device J, H,
 * through the factor kernel's gather tables), and its factor in the permuted order:
 * Lband[dim][row_width] with Lband[R][q] = L(R, R-q), D[dim]; P K P' = L D L' */
int dto_kkt_matrix(dto_kkt* k, int64_t problem, double* dense);
int dto_kkt_factor(dto_kkt* k, int64_t problem, double* Lband, double* D);
/* which = 0 h, 1 sol, 2 factor storage, 3 per-problem primal regularisation [shard size] (asking for it switches the
 * kernels to per-problem mode: the caller writes it on the device), 4 negative-pivot counts [shard size] int32,
 * 5 a per-problem diagonal [shard size][dim] (natural order: variables, then constraint rows) ADDED to K from then on (zero
 * at first: the barrier terms of an interior-point solver -- z_L / (x - l) + z_U / (u - x) on variables with Bound(...),
 * src/bounds.jl; -t_i / lambda_i on inequality rows, Constraint(...; indices_inequality), src/constraints.jl), 6 the knot blocks
 * [shard size][nnz_blk] (KNOT_BLOCKS handles only) */
void* dto_kkt_device_pointer(dto_kkt* k, int which, int shard);

/* ---- batched solver: the caller of the callback path (SURVEY 8f N1) ----
 * Replaces solve!(solver) (/root/reference/src/solver.jl:45-47: MOI.optimize! hands the five callbacks to Ipopt) for a
 * whole batch at once: a lock-step line-search Newton-KKT (SQP) method whose every step is a kernel of this library --
 * the callbacks above, the KKT consumer, and O(B N) bookkeeping kernels (csrc/dto_sqp.cu); only eight counters per
 * synchronisation cross PCIe during the iterations. It is NOT Ipopt (l1 merit line search instead of a filter, no feasibility
 * restoration). Scope: equality rows and inequality rows c_i(z) <= 0; variables free, pinned by equal bounds, or bounded --
 * inequalities by a primal-dual interior point on the same Newton-KKT step (the barrier terms are a diagonal the factor kernel
 * adds to K). The algorithm is stated
 * in directtrajectoryoptimization.jl_b200/sqp.py (`solve`); the fields below are that file's SQPOptions. */
typedef struct dto_sqp_options {
    int32_t max_iter;        /* Options.max_iter (src/options.jl:9) */
    int32_t max_refactor;    /* inertia-correction attempts per iteration */
    int32_t max_backtrack;   /* line-search rounds per iteration */
    int32_t soc;             /* 1: second-order correction after a rejected full step */
    double tol_constraint;   /* converged: ||c||_inf <= tol_constraint and ||g + J'lambda||_inf <= tol_dual */
    double tol_dual;
    double dual_reg;         /* delta_c of K = [[H + delta I, J'], [J, -delta_c I]] */
    double reg_first, reg_min, reg_max, reg_inc_first, reg_inc, reg_dec;   /* Ipopt's inertia-correction constants */
    double armijo, merit_margin, merit_rho, merit_min;                     /* l1 merit line search */
    double lm_first, lm_min, lm_grow, lm_shrink, lm_grow_below, lm_zero;   /* Levenberg-Marquardt damping of H */
    double lam_max;          /* multiplier estimates beyond this are reset to 0 (0 = off) */
    double exact_below;      /* ||c||_inf under which the Hessian of the Lagrangian is used (else the objective's: Gauss-Newton) */
    /* interior-point mode: inequality bounds on variables and inequality rows c_i(z) <= 0 */
    double mu_init;          /* first barrier parameter */
    double barrier_kappa_eps, barrier_kappa_mu, barrier_theta_mu;   /* monotone barrier update (Waechter & Biegler 2006, eq. 7) */
    double tau_min;          /* fraction to the boundary */
    double bound_push, bound_frac;   /* the starting point is moved this far inside its bounds */
    double kappa_sigma;      /* bound multipliers stay within [mu / (kappa s), kappa mu / s] */
    double tiny_step;        /* relative step size under which a step is taken without the merit test */
    double bound_relax;      /* > 1: problems left unconverged are solved again with two-sided bounds widened by this factor, then
                                the true bounds warm-started from there (<= 1: no such fallback) */
    int32_t hessian_approximation;   /* 0: the exact Hessian of the Lagrangian (needs evaluate_hessian); 1: knot-block damped BFGS
                                        (no Hessian needed: one dense block per knot, updated once per iteration from the change of
                                        the Lagrangian's gradient; Nocedal & Wright, Procedure 18.2) */
} dto_sqp_options;
void dto_sqp_default_options(dto_sqp_options* o);
/* Solves every problem of a one-shard batch (several devices: one batch and one host thread per device) from z0 [B][N_z] (lambda0 [B][N_c] or NULL = 0). lower / upper [N_z] or
 * NULL: primal_bounds (src/data.jl:123-133); a variable with lower == upper is pinned to that value, any other finite
 * bound is an inequality (interior point). Constraint rows other than equalities and (-Inf, 0] -> DTO_ERR_UNSUPPORTED. Outputs (each may be NULL): z [B][N_z],
 * lambda [B][N_c], iterations [B] (max_iter where not converged), converged [B] (1; 2 = by the bound continuation), constraint_violation [B] = ||c||_inf,
 * dual_residual [B], objective [B]; stats[16] = {iterations run, kernel launches, factorisation launches, host
 * synchronisations, inertia-correction factorisations, second-order-correction solves, sequential line-search rounds,
 * one-pass evaluations of all remaining step lengths, and host
 * microseconds spent in: callbacks + first factorisation, inertia correction, line search (with corrections),
 * second-order corrections; set-up (allocations, tables, host -> device), iteration loop, results (device -> host);
 * iterations whose predicted inertia corrections ran beside the first factorisation} -- summed over the direct solve and the
 * two passes of the bound continuation when that ran. The final iterate stays resident as the batch's z (dto_get_last_x). */
int dto_sqp_solve(dto_batch* b, const dto_sqp_options* options, const double* z0, const double* lambda0, const double* lower,
                  const double* upper, double* z, double* lambda, int32_t* iterations, uint8_t* converged,
                  double* constraint_violation, double* dual_residual, double* objective, int64_t* stats);

#ifdef __cplusplus
}
#endif
#endif /* DTO_H */

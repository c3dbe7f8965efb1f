/*
 * dto_b200.h -- C ABI of libdto_b200.so, the B200 (sm_100a) NLP-callback evaluator that replaces
 * DirectTrajOpt.jl's `Solvers.Evaluator <: MOI.AbstractNLPEvaluator` hot path.
 *
 * Every entry point is what the reference's FFI for this path binds (Julia `ccall`; Python `ctypes`
 * in this repo's host mirror).  Citations are into /root/reference (DirectTrajOpt.jl v0.9.7).
 *
 *   reference interface                                   (file:line)                 -> C entry point
 *   Evaluator(prob; eval_hessian)                          src/solvers/evaluator.jl:99-288  -> dto_create
 *   (GC finaliser of the evaluator)                        --                               -> dto_destroy
 *   n_constraints / n_dynamics_constraints / fields        src/solvers/evaluator.jl:71-77   -> dto_sizes
 *   MOI.jacobian_structure                                 src/solvers/evaluator.jl:364     -> dto_jac_structure
 *   MOI.hessian_lagrangian_structure                       src/solvers/evaluator.jl:385     -> dto_hess_structure
 *   MOI.eval_objective                                     src/solvers/evaluator.jl:304     -> dto_eval_objective
 *   MOI.eval_objective_gradient                            src/solvers/evaluator.jl:310     -> dto_eval_gradient
 *   MOI.eval_constraint                                    src/solvers/evaluator.jl:323     -> dto_eval_constraint
 *   MOI.eval_constraint_jacobian                           src/solvers/evaluator.jl:368     -> dto_eval_jacobian
 *   MOI.eval_hessian_lagrangian                            src/solvers/evaluator.jl:389     -> dto_eval_hessian
 *   MOI.eval_constraint_jacobian_product                   src/solvers/evaluator.jl:406     -> dto_eval_jacobian_product
 *   MOI.eval_constraint_jacobian_transpose_product         src/solvers/evaluator.jl:432     -> dto_eval_jacobian_transpose_product
 *   (benchmark/benchmarks.jl:23-38 times the five above on one iterate)                     -> dto_eval_all[_dev]
 *   get_nonlinear_constraints row bounds                   src/solvers/solve.jl:30-65       -> dto_constraint_bounds
 *   GlobalObjective / GlobalKnotPointObjective             src/objectives/global_objectives.jl:35-341          -> DTO_OBJ_GLOBAL_KNOT terms
 *   NonlinearGlobalConstraint                              src/constraints/nonlinear/global_constraint.jl:24-159 -> constraint with n_vars == 0
 *   NonlinearGlobalKnotPointConstraint                     src/constraints/nonlinear/global_knot_point_constraint.jl:30-256 -> constraint with n_gvars > 0
 *
 * Conventions
 *   - all values are IEEE double, all structure indices are 1-based int64 in the reference's order
 *     (column-major findnz of the Jacobian; upper triangle, column-major, of the Hessian).
 *   - Z is the solver's primal vector [vec(data[z x N]); global_data[global_dim]], knot-major
 *     (src/solvers/evaluator.jl:474-482); n_vars = z*N + global_dim.
 *   - every output buffer is owned and pre-allocated by the caller and is fully overwritten.
 *   - host-pointer entry points copy between the caller's buffers and device buffers owned by the handle and
 *     return after the stream has drained; with page-locked caller buffers the device->host copies of
 *     finished knot ranges overlap the remaining computation.  For bilinear/derivative problems the structural
 *     zeros of the Hessian (the cross-knot block and every column below the first one a term can touch) do not
 *     cross PCIe: a few host threads of the handle write them into the caller's buffer meanwhile
 *     (DTO_B200_HOST_THREADS, default 4; the constant identity/zero head of the Jacobian columns is skipped only for
 *     arrays given to dto_register_outputs).  `_dev` entry points take device pointers
 *     valid on the handle's device and enqueue on the handle's stream (dto_stream) without synchronising.
 *   - return value: 0 on success, negative dto_status otherwise; no exception crosses the boundary.
 *     dto_last_error() gives the message.  A handle is not thread-safe (matches the reference, whose
 *     callbacks mutate a shared cached trajectory: src/solvers/evaluator.jl:474-482).
 *   - there is no CPU fallback: without a CUDA device dto_create fails with DTO_ERR_CUDA.
 *   - `batch` > 1 evaluates `batch` independent problems of identical structure in one launch;
 *     all vectors are then laid out problem-major ([batch][n]) and structures describe ONE problem.
 *   - a knot-range shard (shard_k0/shard_k1) evaluates only its own knots of one long trajectory
 *     (SURVEY.md section 8e, partitioning B); see dto_shard_layout.
 */
#ifndef DTO_B200_H
#define DTO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DTO_B200_ABI_VERSION 4

typedef struct dto_handle dto_handle;

typedef enum {
    DTO_OK = 0,
    DTO_ERR_INVALID = -1,     /* malformed descriptor / argument */
    DTO_ERR_UNSUPPORTED = -2, /* component outside the device catalogue: raised at construction, never mid-solve */
    DTO_ERR_CUDA = -3,        /* CUDA runtime failure (incl. "no device": there is no CPU fallback) */
    DTO_ERR_ALLOC = -4
} dto_status;

/* integrator kinds (src/integrators/) */
enum { DTO_INT_BILINEAR = 1, DTO_INT_DERIVATIVE = 2, DTO_INT_TDBILINEAR = 3 };
/* objective kinds (src/objectives/) */
enum {
    DTO_OBJ_QUADREG = 1, DTO_OBJ_MINTIME = 2, DTO_OBJ_KNOT = 3, DTO_OBJ_NULL = 4, DTO_OBJ_LINREG = 5,
    /* J = sum_i Q_i l([knot vars at times[i]; global vars], p_i) (global_objectives.jl:139-341).  A GlobalObjective
     * (global_objectives.jl:35-130) is the same term with n_vars == 0, times = [1], Qs = [Q]. */
    DTO_OBJ_GLOBAL_KNOT = 6
};
/* device catalogue of knot constraint functions g(v; p) (replaces the Julia closure of
 * src/constraints/nonlinear/knot_point_constraint.jl:76-83) */
enum {
    DTO_G_NORM_MINUS_C = 1, DTO_G_NORMSQ_MINUS_C = 2, DTO_G_SQDIST_MINUS_C = 3, DTO_G_LINEAR = 4,
    /* [norm(v1) - c1; norm(v1) norm(v2) - c2], v = [v1 (n1 entries); v2], p = [c1, c2, n1]: the reference's test
     * function for knot + global variables (global_knot_point_constraint.jl:267-270) */
    DTO_G_NORM_PRODUCT = 5,
    /* a user function given as a knot program (dto_knot_program, below): `program` of the descriptor indexes
     * dto_problem_desc::programs (ABI version 4) */
    DTO_G_PROGRAM = 100
};
/* device catalogue of knot objective functions l(v; p) (src/objectives/knot_point_objectives.jl:65-72) */
enum {
    DTO_L_NORMSQ_PLUS_P = 1, DTO_L_SQDIST = 2, DTO_L_LINEAR = 3, DTO_L_ISO_INFIDELITY = 4,
    /* norm(v[0:h] - v[h:2h])^2, h = n/2: state against a goal held in a global (global_objectives.jl:364-369) */
    DTO_L_SPLIT_SQDIST = 5,
    DTO_L_PROGRAM = 100 /* a knot program with one output (ABI version 4) */
};

/* Knot programs: a user-written g(v; p) / l(v; p) as an SSA tape (the reference's closures of
 * knot_point_constraint.jl:76-83 and knot_point_objectives.jl:65-72, traced once by the front end).
 * Value i of the tape is defined by ops[3 i .. 3 i + 2] = {opcode, a, b}:
 *   DTO_OP_VAR    a = variable index < n_vars + n_gvars of the term (knot variables first, then global variables)
 *   DTO_OP_PARAM  a = index into this time's parameter row, < n_params
 *   DTO_OP_CONST  a = index into consts
 *   ADD SUB MUL DIV                  values a and b
 *   NEG SQRT EXP LOG SIN COS TANH    value a
 *   POWC          value a raised to consts[b] (an integer-valued exponent is valid for negative bases)
 * Operands of non-leaf operations reference earlier values (< i): the tape is acyclic by construction.  out[k] is the
 * value of output k (g_dim outputs for a constraint, one for an objective).  dto_create drops dead values, orders the
 * rest depth-first from the outputs and allocates registers of the device interpreter by linear scan; a program longer
 * than DTO_MAX_PROGRAM_OPS or needing more than DTO_MAX_PROGRAM_SLOTS live values is DTO_ERR_UNSUPPORTED, a malformed
 * one DTO_ERR_INVALID -- at construction, never mid-solve. */
enum {
    DTO_OP_VAR = 1, DTO_OP_PARAM = 2, DTO_OP_CONST = 3,
    DTO_OP_ADD = 4, DTO_OP_SUB = 5, DTO_OP_MUL = 6, DTO_OP_DIV = 7,
    DTO_OP_NEG = 8, DTO_OP_SQRT = 9, DTO_OP_EXP = 10, DTO_OP_LOG = 11, DTO_OP_SIN = 12, DTO_OP_COS = 13, DTO_OP_TANH = 14,
    DTO_OP_POWC = 15
};
#define DTO_MAX_PROGRAM_OPS 4096
#define DTO_MAX_PROGRAM_SLOTS 32

typedef struct {
    int32_t n_ops, n_out;
    const int32_t* ops;    /* n_ops x {opcode, a, b} */
    const int32_t* out;    /* n_out value indices */
    int32_t n_consts, _pad;
    const double* consts;
} dto_knot_program;

/* One dynamics integrator (src/integrators/{bilinear,derivative,time_dependent_bilinear}_integrator.jl).
 * Component offsets are 0-based positions inside one knot. */
typedef struct {
    int32_t kind;
    int32_t x_off, x_dim;  /* state component */
    int32_t u_off, u_dim;  /* bilinear / tdbilinear: drive component; derivative: the derivative component (u_dim == x_dim) */
    int32_t t_off;         /* tdbilinear: time component, else -1 */
    int32_t spline_order;  /* tdbilinear: 0 (hold) or 1 (linear, reference default) */
    int32_t n_carrier;     /* tdbilinear: number of undriven carrier terms D_j */
    /* bilinear: (u_dim+1) matrices x_dim x x_dim, column-major: G_drift, G_drive_1.. (G(u) lowered to data,
     * src/integrators/bilinear_integrator.jl:69).  tdbilinear: G0.  Per-problem generators in a batch
     * are laid out [batch][u_dim+1][n*n] when G_batch_stride != 0. */
    const double* G;
    int64_t G_batch_stride; /* doubles between consecutive problems' generator sets; 0 = shared */
    /* tdbilinear drive envelopes: G(u,t) = G0 + sum_i u_i (cos(w_i t + phi_i) A_i + sin(w_i t + phi_i) B_i)
     *                                        + sum_j cos(wd_j t + phd_j) D_j */
    const double* A;       /* u_dim matrices */
    const double* B;       /* u_dim matrices */
    const double* omega;   /* u_dim */
    const double* phi;     /* u_dim */
    const double* D;       /* n_carrier matrices */
    const double* omega_d; /* n_carrier */
    const double* phi_d;   /* n_carrier */
    int32_t tdb_steps;     /* tdbilinear: fixed number of RK steps per interval (0 = default) */
    int32_t _pad;
} dto_integrator_desc;

/* One term of the (composite) objective, J = sum_i weight_i * J_i (src/objectives/_objectives.jl:106-156). */
typedef struct {
    int32_t kind;
    int32_t fn;              /* DTO_OBJ_KNOT: catalogue id */
    double weight;
    int32_t n_vars;          /* length of var_offs */
    int32_t n_times;
    const int32_t* var_offs; /* 0-based positions inside a knot of the variables the term reads */
    const int32_t* times;    /* 1-based knots (quadreg: `times`; knot: `times`) */
    const double* R;         /* quadreg: n_vars diagonal weights (src/objectives/regularizers.jl:38-43);
                              * linreg: n_vars linear weights, J = sum_t dt_t R'v_t (regularizers.jl:207-313) */
    const double* baseline;  /* quadreg: n_vars x N column-major, may be NULL (= zeros) */
    double D;                /* mintime scale (src/objectives/minimum_time_objective.jl:24-26) */
    int32_t n_params;        /* knot: doubles of parameters per listed time */
    int32_t program;         /* fn == DTO_L_PROGRAM: index into dto_problem_desc::programs (ABI 3: padding) */
    const double* params;    /* knot: n_times x n_params, row-major */
    const double* Qs;        /* knot: n_times weights */
    int32_t n_gvars;         /* global_knot: global variables appended to the knot variables */
    int32_t _pad2;
    const int32_t* gvar_offs;/* 0-based positions inside global_data */
} dto_objective_desc;

/* One NonlinearKnotPointConstraint (src/constraints/nonlinear/knot_point_constraint.jl:27-107). */
typedef struct {
    int32_t fn;       /* catalogue id */
    int32_t equality; /* only affects dto_constraint_bounds (src/solvers/solve.jl:56-62) */
    int32_t n_vars;
    int32_t n_times;
    const int32_t* var_offs;
    const int32_t* times; /* rows are ordered by position in `times` */
    int32_t g_dim;
    int32_t n_params;
    const double* params; /* n_times x n_params, row-major */
    /* global variables appended to the knot variables: g([knot vars; global vars], p).  n_vars == 0 with
     * times = [1] is a NonlinearGlobalConstraint (rows = g_dim). */
    int32_t n_gvars;
    int32_t program;          /* fn == DTO_G_PROGRAM: index into dto_problem_desc::programs (ABI 3: padding) */
    const int32_t* gvar_offs; /* 0-based positions inside global_data */
} dto_constraint_desc;

typedef struct {
    int32_t abi_version; /* DTO_B200_ABI_VERSION */
    int32_t N;           /* knots of the whole trajectory */
    int32_t z;           /* variables per knot (traj.dim) */
    int32_t dt_off;      /* 0-based position of the timestep component inside a knot */
    int32_t batch;       /* independent problems of identical structure (>= 1) */
    int32_t eval_hessian;/* 0: Hessian entry points return DTO_ERR_INVALID (features [:Grad,:Jac]) */
    int32_t shard_k0;    /* 1-based first owned knot; 0 = whole trajectory */
    int32_t shard_k1;    /* 1-based last owned knot (inclusive) */
    int32_t device;      /* CUDA device ordinal, -1 = current */
    int32_t n_integrators;
    int32_t n_objectives;
    int32_t n_constraints;
    const dto_integrator_desc* integrators;
    const dto_objective_desc* objectives;
    const dto_constraint_desc* constraints;
    /* Initial trajectory ([batch][z*N + global_dim]); knot-constraint Jacobian entries are stored only where the
     * derivative at this point is nonzero (src/solvers/evaluator.jl:134-144 + SparseArrays setindex!).
     * With batch > 1 problem 0 defines the pattern.  May be NULL when there are no knot constraints. */
    const double* Z0;
    int32_t global_dim;  /* traj.global_dim: variables after the knots in Z (0 = none) */
    /* ABI version 4: the knot programs that DTO_G_PROGRAM / DTO_L_PROGRAM terms index.  dto_create accepts version 3
     * descriptors, which end before these fields and cannot name programs. */
    int32_t n_programs;
    const dto_knot_program* programs;
} dto_problem_desc;

typedef struct {
    int64_t n_vars;           /* z*N + global_dim */
    int64_t n_dynamics_cons;  /* sum_i d_i (N-1) */
    int64_t n_nonlinear_cons; /* sum_c g_dim_c * n_times_c */
    int64_t n_cons;
    int64_t nnz_jac;
    int64_t nnz_hess;
} dto_size_info;

/* What a knot-range shard owns, in terms of the whole problem's vectors (all 0-based, half-open). */
typedef struct {
    int64_t z_begin, z_end;       /* owned slice of Z */
    int64_t z_halo_end;           /* Z needed for evaluation = [z_begin, z_halo_end) (one-knot right halo) */
    int64_t n_local_cons;         /* rows this shard evaluates */
    int64_t n_local_jac;          /* Jacobian values this shard evaluates */
    int64_t n_local_hess;         /* Hessian values this shard evaluates */
} dto_shard_layout;

int dto_abi_version(void);
int dto_create(const dto_problem_desc* desc, dto_handle** out);
void dto_destroy(dto_handle* h);
const char* dto_last_error(const dto_handle* h); /* h may be NULL: error of the last failed dto_create */
int dto_sizes(const dto_handle* h, dto_size_info* out);
void* dto_stream(const dto_handle* h); /* cudaStream_t */

/* Structures of ONE problem, 1-based, reference order.  For a shard: the locally evaluated entries,
 * with GLOBAL row/column numbers, in the order of the local value arrays. */
int dto_jac_structure(const dto_handle* h, int64_t* rows, int64_t* cols);
int dto_hess_structure(const dto_handle* h, int64_t* rows, int64_t* cols);
/* for a shard: global 0-based positions of the local rows / Jacobian / Hessian values */
int dto_shard_info(const dto_handle* h, dto_shard_layout* out);
int dto_shard_maps(const dto_handle* h, int64_t* con_rows, int64_t* jac_pos, int64_t* hess_pos);
/* lower / upper bound of every constraint row: (0,0) or (-inf,0) */
int dto_constraint_bounds(const dto_handle* h, double* lower, double* upper);

/* ---- host-pointer callbacks (pageable or pinned host memory) ---- */
int dto_eval_objective(dto_handle* h, const double* Z, double* J);                 /* J[batch] */
int dto_eval_gradient(dto_handle* h, const double* Z, double* grad);               /* [batch][n_vars] */
int dto_eval_constraint(dto_handle* h, const double* Z, double* g);                /* [batch][n_cons] */
int dto_eval_jacobian(dto_handle* h, const double* Z, double* vals);               /* [batch][nnz_jac] */
int dto_eval_hessian(dto_handle* h, const double* Z, double sigma, const double* mu, double* vals); /* [batch][nnz_hess] */
int dto_eval_jacobian_product(dto_handle* h, const double* Z, const double* w, double* y);           /* y = J w   */
int dto_eval_jacobian_transpose_product(dto_handle* h, const double* Z, const double* w, double* y); /* y = J' w  */
/* One fused pass over one iterate: any output pointer may be NULL to skip that quantity. */
int dto_eval_all(dto_handle* h, const double* Z, double sigma, const double* mu, double* J, double* grad,
                 double* g, double* jac_vals, double* hess_vals);

/* Iterate cache.  The reference copies Z into its cached trajectory in EVERY callback (src/solvers/evaluator.jl:474-482) and
 * the solvers call the five callbacks separately on one iterate (src/solvers/ipopt_solver/solver.jl:85).  The handle
 * keeps a page-locked copy of the iterate that is resident on the device: a callback whose Z equals it (memcmp) skips the
 * upload and re-uses what earlier callbacks computed.  The first callback that needs the interval kernels on a NEW
 * iterate runs one mu-independent pass (residual + Jacobian + the second-order vectors of the forward jet); the
 * Hessian callback then runs only the adjoint recurrences, contracts the stored vectors with mu and assembles.
 * Early start: when the FIRST callback on a new iterate asks for the objective or its gradient only (the order Ipopt and
 * MadNLP use), it also enqueues that mu-independent pass and returns as soon as its own result is on the host; the
 * interval kernels run while the solver goes through its next callbacks, which then wait only for what they deliver
 * (the residual is staged in page-locked memory, the Jacobian goes to a registered array on the side).  Every output is
 * valid when its own callback returns; iterates that are dropped after the objective alone (line searches) pause the
 * early start.  Results are bit-identical to dto_eval_all.  dto_upload makes Z the resident iterate without evaluating
 * anything (and returns after the copy has completed: on knot-range shards, the point after which a neighbour may read
 * this rank's knots). */
int dto_upload(dto_handle* h, const double* Z);
int dto_cache_stats(const dto_handle* h, int64_t* hits, int64_t* misses);
/* Optional: tell the handle where the solver keeps its Jacobian / Hessian value arrays (either may be NULL; batch == 1).
 * The arrays are page-locked (cudaHostRegister) and their structural constants -- Hessian entries no term of the
 * problem can touch, the identity/zero head of the Jacobian columns (d r_{k-1}/d z_k of a bilinear or derivative
 * integrator) -- are written ONCE, here.  Later callbacks that are handed these pointers move only the value-dependent
 * entries (c2: 27 of 72 MB), with no host threads involved, and the Jacobian a constraint callback computes on a new
 * iterate starts leaving for the registered array at once (dto_eval_jacobian on the same iterate then only joins the
 * copy).  Contract: between dto_register_outputs and dto_unregister_outputs / dto_destroy the caller only READS the arrays
 * (what Ipopt and MadNLP do with the value arrays of MOI.eval_constraint_jacobian / eval_hessian_lagrangian), and the
 * Jacobian array may be written by any callback. */
int dto_register_outputs(dto_handle* h, double* jac_vals, double* hess_vals);
int dto_unregister_outputs(dto_handle* h);

/* ---- device-pointer callbacks: enqueue on dto_stream(h), no host synchronisation ---- */
int dto_eval_all_dev(dto_handle* h, const double* dZ, double sigma, const double* dmu, double* dJ, double* dgrad,
                     double* dg, double* djac_vals, double* dhess_vals);
/* max-norm constraint violation of residuals already on the device: max(|g_eq|, max(0, g_ineq)) -> dviol[batch] */
int dto_violation_dev(dto_handle* h, const double* dg, double* dviol);
int dto_synchronize(dto_handle* h);

/* ---- knot-range sharding: one-knot halo and the two scalars over NVLink peer memory ----
 * An unlinked shard reads its right halo knot from the caller's own slice of Z ([z_begin, z_halo_end)): no cross-rank
 * traffic, no ordering requirement.  LINKED shards (one per rank of a single box; CUDA IPC across processes) exchange
 * through windows in each other's HBM instead, inside the evaluation stream:
 *   - after uploading iterate e a shard pushes its first knot into the left neighbour's window and publishes e there;
 *     the left neighbour's kernels of iterate e wait for that flag on the device and read the knot from the window (shards
 *     linked across processes: the upload's own kernel copies, pushes and waits -- one launch).  The reader acknowledges
 *     when it moves on, so a rank runs at most one iterate ahead of the neighbour reading its knot.
 *   - dto_allreduce_scalars_dev: objective (sum) and violation (max) of all shards with one kernel per rank that
 *     stores into every peer's window and spins on its own (rank-ordered sum: identical bits on every rank; no NCCL).
 *   - time-dependent bilinear integrators with spline_order = 1: interval k0 - 1, which the left neighbour owns, adds
 *     to the Hessian region of this shard's first knot k0 (its (u, u) entries and the whole (k0 - 1, k0) cross block).
 *     Every Hessian evaluation the left neighbour pushes the compact second derivatives of its last interval into this
 *     shard's window; this shard assembles its first knot last, after waiting for them.  The reassembled Hessian is
 *     bit-identical to the unsharded one.
 * Protocol: EVERY rank uploads EVERY iterate exactly once, with dto_upload (host Z slice) or dto_upload_dev (device);
 * callbacks are then called with that same Z (iterate-cache hits) or through the _dev entry points on dto_local_Z.
 * With a linear-spline time-dependent integrator, a linked shard's Hessian evaluation s (counted from the link, any
 * entry point) reads what its left neighbour's Hessian evaluation s produced: EVERY rank evaluates EVERY Hessian, and a
 * thread that drives several linked shards calls them in rank order.  Such a shard that starts after knot 1 and is not
 * linked has no Hessian (DTO_ERR_INVALID; everything else evaluates).
 * A wait that sees no progress for 20 s fails the evaluation with DTO_ERR_CUDA instead of hanging. */
/* 64-byte cudaIpcMemHandle_t of this shard's exchange window */
int dto_shard_export(dto_handle* h, void* ipc_handle_64B);
/* map the windows of all `world` shards (handles64 = world x 64 bytes in rank order; the own entry is ignored).  Linking
 * (again) clears this shard's window: every rank links before any rank uploads an iterate. */
int dto_shard_link(dto_handle* h, int rank, int world, const void* handles64);
/* several shards in ONE process (tests, one-process multi-device drivers): handles in rank order */
int dto_shard_link_local(dto_handle* const* handles, int world);
/* a new iterate that already lives on the device: copies it into the resident buffer (unless dZ == dto_local_Z) and
 * publishes it to the neighbours; enqueues on dto_stream(h) without synchronising */
int dto_upload_dev(dto_handle* h, const double* dZ);
/* in place: dJ[0] <- sum over shards, dviol[0] <- max over shards; enqueues on dto_stream(h) */
int dto_allreduce_scalars_dev(dto_handle* h, double* dJ, double* dviol);
/* the same with the shard's violation computed from its residuals dg in the SAME kernel (instead of dto_violation_dev +
 * dto_allreduce_scalars_dev): dJ[0] <- sum over shards of dJ[0], dviol[0] <- max over shards */
int dto_shard_scalars_dev(dto_handle* h, const double* dg, double* dJ, double* dviol);
/* device pointer of this shard's resident Z buffer ([z_begin, z_halo_end) of the global Z) */
double* dto_local_Z(dto_handle* h);

/* ---- instrumentation ---- */
/* kernels launched by this handle since creation (bench.py's gpu_launches) */
int64_t dto_launch_count(const dto_handle* h);
/* bytes the last host-pointer evaluation moved device -> host.  Less than the size of the outputs when structural zeros
 * of the Hessian (columns no term of the problem can touch) are written by host threads instead of crossing PCIe. */
int64_t dto_last_download_bytes(const dto_handle* h);
/* name of the bilinear kernel variant chosen for integrator i ("dmma", "generic", ...) */
const char* dto_kernel_variant(const dto_handle* h, int integrator);
/* CUDA-event timing of the interval kernels (K1/K7) on the handle's stream: enable, run evaluations,
 * then read the summed device time and the number of timed launches (resets on enable). */
int dto_kernel_timing(dto_handle* h, int enable);
int dto_kernel_time_ms(dto_handle* h, double* ms_sum, int64_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* DTO_B200_H */

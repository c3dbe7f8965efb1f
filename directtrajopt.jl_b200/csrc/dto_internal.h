// Internal device/host structures of libdto_b200.so.  Not part of the ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/dto_b200.h"

#define DTO_MAX_INT 8
#define DTO_MAX_OBJ 16
#define DTO_MAX_CON 8
#define DTO_MAX_KNOTFN_VARS 128

// ---- device views (passed by value to kernels) ------------------------------------------------
// A compiled knot program (knot_program.cuh): n_code words {opcode, dst slot, a, b}, then the constants as doubles, in
// one device allocation.  Outputs are DTO_OP_OUT words (dst = output index, a = slot).
enum { DTO_OP_OUT = 16 };
struct DProgram {
    const int4* code;  // null: the term is a catalogue function
    int n_code;
    int _pad;
    __host__ __device__ const double* consts() const { return reinterpret_cast<const double*>(code + n_code); }
};
struct DInt {
    int kind, x_off, n, u_off, m, t_off, order, n_carrier;
    int doff;           // sum of x_dim of the integrators before this one
    int hs_stride;      // doubles of compact Hessian scratch per interval
    int steps;          // tdbilinear: minimum number of macro steps per interval (the kernels raise it per interval, tdb_item_steps)
    double tdb_gnorm;   // tdbilinear: ||G0||_1 + sum_j ||D_j||_1
    double tdb_wmax;    // tdbilinear: largest carrier frequency |w_i|, |wd_j|
    double tdb_tol;     // tdbilinear: extrapolation-error target that sizes the columns per interval (0: always the maximum)
    const double* tdb_bnorm;  // tdbilinear: [m] ||A_i||_1 + ||B_i||_1
    int variant;        // kernel variant chosen on the host
    long long row_off;  // local row of this integrator's first residual
    long long G_stride;
    const double* G;    // column-major matrices
    const double* Grm;  // bilinear: row-major copies of the same matrices
    const double* bfrag;  // bilinear, octet variant with per-problem generators: fragment-ordered copies [batch][...]
    const double *A, *B, *omega, *phi, *D, *omega_d, *phi_d;
    const double *Asw, *Bsw, *Dsw;  // tdbilinear, DMMA variant: swizzled row-major copies (Grm holds G0)
    double* tdb_scratch;            // tdbilinear, DMMA variant: per-CTA extrapolation scratch
    int tdb_scratch_ctas;           // CTAs the scratch was sized for (one per SM)
    double* hs;         // [batch][n_intervals][hs_stride]
    // bilinear (persistent / octet variants): the second-order vectors of the forward jet, kept between the mu-independent
    // pass over a new iterate and the Hessian callback on the same iterate (EvalFlags::jets):
    // [batch][n_intervals][jet_stride], jet_stride = (m(m+1)/2 + 1 + 2m) n :
    //   d2(Ex)/(du_a du_b) (a <= b, row-major over the upper triangle) | G G E x | G_i E x (i < m) | G d(Ex)/du_i (i < m)
    double* jets;
    int jet_stride;
    // bilinear (persistent / octet variants): per-interval series plan {alpha, theta1} written by series_plan_kernel
    // before the interval kernels of an iterate (series_plan.cu); nullptr: the kernels size the series from ||dt G(u)||_1
    const double2* plan;
    const double* Gsw;     // persistent variant: the swizzled shared-memory image of Grm (bulk-copied by the prologue)
    const float* planmat;  // series_plan.cu: FP32 [G_0..G_m | pair products | norms] (shared generator sets only)
    unsigned long long* wq;  // bilinear, persistent variant: three work-queue counters (FWD, EXP, ADJ)
};

struct DObj {
    int kind, fn;
    double weight;
    int nv, nt, np;
    int nvk;                  // variables 0..nvk-1 are knot components, nvk..nv-1 global variables (nvk == nv without globals)
    double D;
    const int* var_offs;      // knot component offsets, then offsets into global_data
    const int* g2l;           // terms with globals: [global_dim] -> variable index (>= nvk) or -1
    const int* own_ti;        // owned entries -> index into params/Qs (original position in `times`)
    const int* own_knot;      // owned entries -> local knot (0-based)
    int nt_own;
    int own_kmin, own_kmax;   // smallest / largest owned local knot (host-side launch pruning)
    const int* knot_to_own;   // [local knots] -> owned entry index or -1
    long long side_off;       // knot objectives: offset of this term's [owned knot][variable pair] block in DProb::knot_side
    const double* R;
    const double* baseline;   // nv x N (global knots), may be null
    const double* params;
    const double* Qs;
    DProgram prog;            // fn == DTO_L_PROGRAM
};

struct DCon {
    int fn, nv, nt_own, gd, np;
    int nvk;                      // as in DObj
    long long row_off;            // local row of the first owned row
    const int* var_offs;
    const int* g2l;
    const int* own_ti;
    const int* own_knot;          // local knot (0-based) of each owned entry
    const int* knot_to_own;
    const double* params;
    const long long* jac_pos;     // [nt_own][gd][nv] local Jacobian position or -1
    DProgram prog;                // fn == DTO_G_PROGRAM
};

// Terms that read global variables (global_objectives.jl, global_constraint.jl, global_knot_point_constraint.jl):
// one "slot" per (term, listed time); objective slots first.
struct DGlob {
    int G;                    // traj.global_dim
    int S, S_obj;             // slots; the first S_obj belong to objective terms
    int KV;                   // largest number of knot variables among the terms with globals
    const int* slot_term;     // objective index (s < S_obj) or constraint index
    const int* slot_j;        // owned entry of the term
    const long long* kg_pos;  // [S][KV][G]: position inside the Hessian tail of (knot variable a, global g) or -1
    const long long* gg_pos;  // [G(G+1)/2]: position inside the Hessian tail of (g, g'), g <= g', or -1
    double* scratchG;         // [batch][S_obj][G] per-slot gradient of the globals
    double* scratchH;         // [batch][S][G(G+1)/2] per-slot global x global Hessian
    long long hess_tail_off;  // local Hessian values: [knot regions | global columns]
    long long n_hess_tail;
};

// The (knot variable, global) Hessian entries of the terms with global variables, summed in a fixed order: every slot
// writes its contribution to the scratch, kg_sum_kernel adds each entry's contributors in ascending slot order.  Kept
// beside DProb, not in it: the kernels that never read it keep their parameter block.
struct DGlobKG {
    double* scratch;       // [batch][S][KV][G] per-slot (knot variable a, global g) entries
    int n;                 // Hessian tail entries of (knot variable, global) pairs
    const long long* dst;  // [n] their positions inside the Hessian tail
    const int* ptr;        // [n + 1]: the contributors of entry i are src[ptr[i] .. ptr[i+1])
    const long long* src;  // index (s KV + a) G + g into a problem's scratch rows, ascending slot s
};

struct DProb {
    int N;          // global knots
    int z, dt_off, batch;
    int kb;         // global 1-based knot of local knot 0
    int nK;         // local knots including the right halo knot (if any)
    int nOwn;       // owned knots
    int nI;         // local intervals (owned knots that have a successor)
    int kc0, kc1;   // active local-knot range of this launch [kc0, kc1): intervals kc0 <= k < min(kc1, nI), owned knots kc0 <= k < min(kc1, nOwn)
    int first_has_cross;  // shard does not start at knot 1: its first knot still owns a cross block
    int any_cross;        // some integrator produces cross-knot Hessian entries (tdbilinear order 1)
    int analytic_fused;   // index+1 of the bilinear integrator whose kernel also writes the derivative integrators' rows (0: analytic_kernel does)
    int reserve_sms;      // host side: SMs the persistent interval kernels leave free for small kernels running beside them on another stream
    int n_int, n_obj, n_con;
    int Dsum;       // sum of x_dim over integrators
    long long n_vars_local;   // nK * z + global_dim  (stride of one problem in the local Z buffer)
    long long n_grad_local;   // nOwn * z + global_dim (stride of one problem's gradient)
    DGlob gl;
    long long n_cons_local, nnz_jac_local, nnz_hess_local;
    const long long* jac_colptr;  // [nK*z + 1] local
    int jac_closed;               // no knot-constraint entries: column starts follow in closed form (no loads in the kernels)
    const unsigned int* hess_tab;  // stream-out gather table of a knot WITH cross rows: region entry -> index into [diag | cross] tiles, 0xFFFFFFFF = structural zero
    double* knot_side;            // knot-objective Hessian pairs w Q d2l (without sigma), written beside the interval kernels
    long long side_stride;        //   doubles per problem of the batch
    const double* halo;           // if non-null: knot nK-1 is read from here (peer memory) instead of local Z
    DInt in[DTO_MAX_INT];
    DObj ob[DTO_MAX_OBJ];
    DCon co[DTO_MAX_CON];
};
// every kernel takes the problem by value: it must fit the kernel-parameter space of sm_70+ (32764 bytes since CUDA 12.1)
static_assert(sizeof(DProb) <= 32764, "DProb exceeds the kernel-parameter limit");

// Macro steps of one tdbilinear interval.  The extrapolation scheme (8 columns of the modified midpoint rule, order 16) is
// accurate to ~1e-13 per macro step while theta = |dt| (||G(u, .)||_1 bound + carrier frequency) stays below 1: the error of
// a macro step of size theta behaves like theta^17 / prod_j (2j)^2 ~ theta^17 1e-14.  The reference controls its error by
// adaptive Tsit5 steps (time_dependent_bilinear_integrator.jl:117-127); here the step count follows the iterate.
// Same arithmetic in every kernel (role CTAs of one interval must agree).
// Macro steps AND extrapolation columns of one interval, from the iterate.  With the modified-midpoint sequence
// n_k = 2, 4, .., 2K the extrapolated value of a linear system with ||dt G|| = theta per macro step has the error
// theta^(2K+1) / (2^K K!)^2 (the product of the n_k^2: 1e-14 at K = 8, theta = 1): `cols` is the smallest K (>= 3, <= kmax)
// that keeps it below I.tdb_tol -- an interval with theta = 0.2 needs 5 columns = 35 right-hand sides, not 8 = 80.
// `poison`: 1, or NaN where the step count would exceed its cap (|dt| (||G|| + omega) > 256 per interval) or the iterate is
// not finite -- the kernels multiply their initial values by it, so such an interval's outputs are NaN (an evaluation
// error the solver sees) instead of silently inaccurate numbers.
__device__ inline int tdb_item_steps(const DInt& I, const double* zk, const double* zk1, int dt_off, double& poison, int kmax, int& cols) {
    double g = I.tdb_gnorm;
    for (int i = 0; i < I.m; ++i) {
        const double u0 = fabs(zk[I.u_off + i]), u1 = I.order == 1 ? fabs(zk1[I.u_off + i]) : u0;
        g += fmax(u0, u1) * I.tdb_bnorm[i];
    }
    const double theta = fabs(zk[dt_off]) * (g + I.tdb_wmax);
    int s = I.steps;
    poison = theta <= 256.0 ? 1.0 : __longlong_as_double(0x7ff8000000000000LL);
    if (theta > (double)s && theta <= 256.0) s = (int)ceil(theta);
    s = s < 256 ? s : 256;
    cols = kmax;
    if (I.tdb_tol > 0.0 && theta <= 256.0) {
        const double ths = theta / (double)s, t2 = ths * ths;
        double pw = ths * t2 * t2 * t2, den = 2304.0;  // theta^7, (2^3 3!)^2
        for (int K = 3; K < kmax; ++K) {
            if (pw <= I.tdb_tol * den) {
                cols = K;
                break;
            }
            pw *= t2;
            den *= 4.0 * (K + 1) * (K + 1);
        }
    }
    return s;
}

// max that keeps a NaN operand (fmax drops it): a residual poisoned with NaN must not reduce to a feasible violation
__host__ __device__ inline double nan_max(double a, double b) { return (b > a || b != b) ? b : a; }

// Jacobian position helpers (local numbering) --------------------------------------------------
// column of local knot kl (0-based), component l: [I1 prev | I1 own | I2 prev | I2 own | ... | constraints]
__host__ __device__ inline long long jac_own_off(const DProb& P, int kl, int doff, int d) {
    return (kl >= 1) ? 2LL * doff + d : doff;
}
__host__ __device__ inline long long jac_prev_off(const DProb& P, int kl, int doff) {
    return (kl < P.nI) ? 2LL * doff : doff;
}
// start of local column (knot kl, component l)
__host__ __device__ inline long long jac_col(const DProb& P, long long kl, int l) {
    if (P.jac_closed) {  // every column of a knot holds Dsum rows per adjacent interval
        const long long D = P.Dsum;
        const long long start = kl == 0 ? 0 : (long long)P.z * D * (2 * kl - 1);
        return start + (long long)l * D * ((kl >= 1 ? 1 : 0) + (kl < P.nI ? 1 : 0));
    }
    return P.jac_colptr[kl * P.z + l];
}
// Hessian: start of local knot kl's region and of column l inside it
__host__ __device__ inline long long hess_knot_base(const DProb& P, int kl) {
    long long z = P.z, tri = z * (z + 1) / 2;
    if (P.first_has_cross) return (long long)kl * (z * z + tri);
    return kl == 0 ? 0 : tri + (long long)(kl - 1) * (z * z + tri);
}
__host__ __device__ inline bool hess_knot_has_cross(const DProb& P, int kl) { return kl > 0 || P.first_has_cross; }

// Exchange window of a knot-range shard: device memory its neighbours map (CUDA IPC, or directly in one process).  See
// shard_link.cu for the protocol.
#define DTO_MAX_RANKS 16
struct XWin {
    unsigned long long halo_epoch;  // written by the RIGHT neighbour: halo[epoch & 1] holds its first knot of iterate `epoch`
    unsigned long long ack;         // written by the LEFT neighbour: it no longer reads this shard's knot of iterates <= ack
    unsigned long long err;         // a wait timed out (1: acknowledgement, 2: halo, 3: scalar exchange, 4: Hessian block
                                    // acknowledgement, 5: Hessian block)
    unsigned long long hs_seq;      // written by the LEFT neighbour: hblk slot hs_seq & 1 holds its boundary block of Hessian evaluation hs_seq
    unsigned long long hs_ack;      // written by the RIGHT neighbour: it has copied this shard's boundary blocks <= hs_ack out of its window
    unsigned long long pad;
    double scal[2][DTO_MAX_RANKS][4];  // [seq & 1][rank] = {objective, violation, seq (as u64), -}
    double halo[2];                    // really [2][z], then hblk [2][hblk_len]: allocated with the window
};
// The boundary Hessian block of a linked shard (linear-spline time-dependent bilinear integrators): one compact-scratch
// row per such integrator.  Pushing side: the rows of the last local interval; receiving side: the leading row of DInt::hs.
struct HsRows {
    double* row[DTO_MAX_INT];
    int len[DTO_MAX_INT];
    int n;
};
// hblk slots of a window: they follow the [2][z] halo slots
__host__ __device__ inline double* xwin_hblk(XWin* w, int z) { return w->halo + 2 * (size_t)z; }
void launch_shard_publish(XWin* own, XWin* left, XWin* right, double* dst, const double* src, long long n, int z,
                          unsigned long long epoch, bool wait_right, cudaStream_t st, long long* launches);
void launch_shard_wait(XWin* own, unsigned long long epoch, cudaStream_t st, long long* launches);
// push this shard's boundary rows into the right neighbour's window (Hessian evaluation `seq`) / wait for the left
// neighbour's block of `seq`, copy it into the local rows and acknowledge it
void launch_hs_push(XWin* own, XWin* right, const HsRows& rows, int z, long long hblk_len, unsigned long long seq, cudaStream_t st,
                    long long* launches);
void launch_hs_receive(XWin* own, XWin* left, const HsRows& rows, int z, long long hblk_len, unsigned long long seq, cudaStream_t st,
                       long long* launches);
void launch_scalar_exchange(XWin* own, XWin* const* peers, int rank, int world, unsigned long long seq, double* J, double* viol,
                            cudaStream_t st, long long* launches);

void launch_shard_scalars(XWin* own, XWin* const* peers, int rank, int world, unsigned long long seq, long long n_cons, const double* g,
                          const int* row_is_eq, unsigned long long* scratch, double* J, double* viol, cudaStream_t st, long long* launches);

// variants of the bilinear kernel
enum { DTO_VAR_GENERIC = 0, DTO_VAR_DMMA = 1, DTO_VAR_PERSISTENT = 2, DTO_VAR_OCTET = 3 };

// Opts `kern` into `bytes` of dynamic shared memory on the current device; a failure names the kernel in `err`
template <class F>
bool opt_in_smem(F* kern, size_t bytes, const std::string& name, std::string& err) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) err = "cannot opt " + name + " into " + std::to_string(bytes) + " bytes of shared memory: " + cudaGetErrorString(e);
    return e == cudaSuccess;
}

// f(std::integral_constant<int, n / 8>()) for the states of the tensor-core kernels, n = 8, 16, 24, 32, 48 and 64
template <class F>
auto with_nt(int n, F&& f) {
    switch (n / 8) {
        case 1: return f(std::integral_constant<int, 1>());
        case 2: return f(std::integral_constant<int, 2>());
        case 3: return f(std::integral_constant<int, 3>());
        case 4: return f(std::integral_constant<int, 4>());
        case 6: return f(std::integral_constant<int, 6>());
        default: return f(std::integral_constant<int, 8>());
    }
}

// ---- kernel launchers (defined in the .cu files) ------------------------------------------------
// jets: 0 = single pass (the Hessian pass contracts the second-order jet with mu in the interval kernel);
//       1 = mu-independent pass over a new iterate: the forward role also carries the second-order rows and STORES the
//           vectors the (parameter, parameter) Hessian entries are contractions of (DInt::jets); no mu is read;
//       2 = Hessian pass on an iterate whose jets are stored: only the adjoint role runs (want_hess must be set), the
//           (parameter, parameter) entries come from launch_hpp_contract.
enum { DTO_JETS_NONE = 0, DTO_JETS_STORE = 1, DTO_JETS_USE = 2 };
struct EvalFlags {
    bool want_g, want_jac, want_hess;
    int jets = DTO_JETS_NONE;
};
// (parameter, parameter) block of the compact Hessian from stored jets: hpp = -mu' W, same summation order as the kernels
void launch_hpp_contract(const DProb& P, int ii, const double* mu, cudaStream_t st, long long* launches);
// The interval-kernel launchers launch the variant dto_create chose (DInt::variant) and never decline: construction
// accepts only shapes they launch and opts their kernels into shared memory (*_configure).  ne_cap and split carry the
// switches the handle read when it was built (dto_host.cu).
void launch_bilinear_generic(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f,
                             cudaStream_t st, long long* launches);
bool bilinear_generic_configure(int n, int m, std::string& err);
size_t generic_smem_bytes(int n, int m, bool want_jac, bool want_hess);  // dynamic shared memory of one generic K1 block
void launch_bilinear_dmma(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f,
                          cudaStream_t st, long long* launches);
bool bilinear_dmma_supported(int n, int m);
bool bilinear_dmma_configure(int n, std::string& err);
void launch_bilinear_persistent(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f,
                                int ne_cap, cudaStream_t st, long long* launches);
bool bilinear_persistent_supported(int n, int m);
bool bilinear_persistent_configure(int n, bool interval, bool product, std::string& err);
void launch_bilinear_octet(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, int split,
                           cudaStream_t st, long long* launches);
bool bilinear_octet_supported(int n, int m);
void bilinear_octet_fragments(int n, int m, const double* Gcm, double* out);
size_t bilinear_octet_fragment_doubles(int n, int m);
void launch_bilinear_product(const DProb& P, int ii, const double* Z, const double* w, double* y, bool transpose, cudaStream_t st,
                             long long* launches);
bool bilinear_product_supported(int n, int m);  // the product kernel's shared memory fits (persistent-supported shapes)
void launch_analytic_product(const DProb& P, const double* Z, const double* w, double* y, bool transpose, cudaStream_t st,
                             long long* launches);
size_t series_plan_smem(int n, int m);
void series_plan_matrices(int n, int m, const double* Gcm, std::vector<float>& out);
void launch_series_plan(const DProb& P, int ii, const double* Z, cudaStream_t st, long long* launches);
bool series_plan_configure(int m, std::string& err);
bool tdb_dmma_supported(const DInt& I);
bool tdb_dmma_configure(int n, std::string& err);
void launch_tdb_dmma(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, bool split,
                     cudaStream_t st, long long* launches);
bool tdb_fits(const DInt& I, size_t smem_limit);
void launch_tdb(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, cudaStream_t st,
                long long* launches);
bool tdb_configure(std::string& err);
void launch_analytic(const DProb& P, const double* Z, double* g, double* jac, EvalFlags f, cudaStream_t st, long long* launches);
void launch_constraints(const DProb& P, const double* Z, double* g, double* jac, EvalFlags f, cudaStream_t st, long long* launches);
bool launch_knot_objective_pairs(const DProb& P, const double* Z, cudaStream_t st, long long* launches);
// left_block: a linked shard's first knot (the only knot of the active range, kc0 = 0) also gets the previous interval's
// share, from the leading row of DInt::hs that launch_hs_receive filled (hessian_assemble_left_kernel)
void launch_hessian_assemble(const DProb& P, const double* Z, double sigma, const double* mu, double* hess, cudaStream_t st,
                             long long* launches, bool left_block = false);
size_t hessian_assemble_smem_bytes(const DProb& P);  // dynamic shared memory of one assembler block (depends on z, any_cross)
bool hessian_assemble_configure(const DProb& P, bool left_block, std::string& err);
void launch_objective(const DProb& P, const double* Z, double* J, double* grad, double* partials, cudaStream_t st,
                      long long* launches);
void launch_violation(const DProb& P, const double* g, const int* row_is_eq, double* viol, cudaStream_t st, long long* launches);
// terms with global variables: global part of the gradient, (knot, global) and (global, global) Hessian entries
void launch_global_gradient(const DProb& P, const double* Z, double* grad, cudaStream_t st, long long* launches);
void launch_global_hessian(const DProb& P, const DGlobKG& kg, const double* Z, double sigma, const double* mu, double* hess, double* kg_probe,
                           cudaStream_t st, long long* launches);
void launch_jac_product(const DProb& P, const double* jac, const long long* rows0, const long long* cols0, const double* w,
                        double* y, bool transpose, cudaStream_t st, long long* launches);
// knot-constraint Jacobian at a host point (used at construction for the stored pattern): runs the
// same device templates so that pattern and values come from one implementation.
// knot programs: one thread per (problem, owned time, seed) for the values and Jacobian of a DTO_G_PROGRAM constraint
void launch_knot_program(const DProb& P, int ci, const double* Z, double* g, double* jac, double* dense_probe, cudaStream_t st,
                         long long* launches);
void launch_constraint_pattern_probe(const DProb& P, const double* Z, double* dense_jac /*[sum nt_own*gd*nv]*/, cudaStream_t st,
                                     long long* launches);

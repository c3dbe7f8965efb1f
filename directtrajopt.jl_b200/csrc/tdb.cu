// K7: TimeDependentBilinearIntegrator interval kernel.
//
// Replaces `solve(ODEProblem, Tsit5())` + ForwardDiff through it
// (/root/reference/src/integrators/time_dependent_bilinear_integrator.jl:102-128,145-244) for the generator family
//     G(u, t) = G0 + sum_i u_i (cos(w_i t + phi_i) A_i + sin(w_i t + phi_i) B_i) + sum_j cos(wd_j t + phd_j) D_j
// with u(tau) = u_k (order 0) or u_k + tau (u_{k+1} - u_k) (order 1), d/dtau Phi = dt G(u(tau), t_k + tau dt) Phi.
//
// One CTA per (problem, interval, role).  Every role integrates a *linear* ODE for a set of vectors with the
// Gragg-Bulirsch-Stoer scheme: modified-midpoint sweeps with n_k = 2,4,..,2K substeps, Gragg smoothing and
// polynomial extrapolation in h^2 (the extrapolation is linear, so the K sweeps are accumulated with fixed
// Lagrange weights and only three copies of the vector set live in shared memory):
//   FWD  x and its first/second-order parameter sensitivities (the dual-number propagation of the reference's
//        ForwardDiff pass, written out as the exact variational equations); parameters
//        theta = [u_k (m), u_{k+1} (m, order 1), dt, t_k]
//   EXP  the columns of the identity -> fundamental matrix Phi(1) for the -Phi Jacobian block
//   ADJ  lambda' = M(1 - s)' lambda in reflected time with first-order sensitivities -> (d Phi/d theta)' mu
// The reference's adaptive Tsit5 runs at reltol 1e-3 by default; this kernel converges to the exact solution
// (error ~1e-12 at the default K = 8 for ||dt G|| ~ 1) -- see DESIGN.md "TDBI parity".
//
// This is the correctness-first CUDA-core variant (LDS-bound dot products); DESIGN.md lists the DMMA port as
// the next step for BASELINE config c3.
#include "dto_internal.h"
#include <algorithm>

namespace {

constexpr int kMaxM = 4;       // drives
constexpr int kMaxC = 4;       // carriers
constexpr int kMaxCols = 10;   // extrapolation columns
constexpr int kThreads = 256;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct Scal {  // per-evaluation scalars at time tau
    double dt, tau, w0, w1;
    double u[kMaxM], c[kMaxM], s[kMaxM], om[kMaxM];
    double e[kMaxC], es[kMaxC], omd[kMaxC];  // carriers: cos, sin, omega
};

enum { ROLE_FWD = 0, ROLE_EXP = 1, ROLE_ADJ = 2 };

struct Ctx {
    int n, m, nc, order, np, ld;
    const double *G0, *A, *B, *D;  // column-major basis matrices in global memory
    double* Gs;                    // n x n, column-major with odd ld: G(u(tau), t(tau))
};

__device__ void make_scal(const DInt& I, const double* zk, const double* zk1, int dt_off, double tau, Scal& S) {
    S.dt = zk[dt_off];
    S.tau = tau;
    const double t = zk[I.t_off] + tau * S.dt;
    S.w0 = I.order == 1 ? 1.0 - tau : 1.0;
    S.w1 = I.order == 1 ? tau : 0.0;
    for (int i = 0; i < I.m; ++i) {
        const double u0 = zk[I.u_off + i], u1 = I.order == 1 ? zk1[I.u_off + i] : u0;
        S.u[i] = S.w0 * u0 + S.w1 * u1;
        S.om[i] = I.omega[i];
        sincos(I.omega[i] * t + I.phi[i], &S.s[i], &S.c[i]);
    }
    for (int j = 0; j < I.n_carrier; ++j) {
        S.omd[j] = I.omega_d[j];
        sincos(I.omega_d[j] * t + I.phi_d[j], &S.es[j], &S.e[j]);
    }
}

// G(tau) into shared memory (all threads)
__device__ void assemble_G(const Ctx& C, const Scal& S) {
    const int n = C.n;
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int r = e % n, c = e / n;
        double v = C.G0[e];
        for (int i = 0; i < C.m; ++i) v = fma(S.u[i], fma(S.c[i], C.A[(size_t)i * n * n + e], S.s[i] * C.B[(size_t)i * n * n + e]), v);
        for (int j = 0; j < C.nc; ++j) v = fma(S.e[j], C.D[(size_t)j * n * n + e], v);
        C.Gs[r + c * C.ld] = v;
    }
}

__device__ __forceinline__ double dot_smem(const double* Gs, int ld, int r, const double* v, int n, bool transpose) {
    double a = 0.0;
    if (!transpose)
        for (int k = 0; k < n; ++k) a = fma(Gs[r + k * ld], v[k], a);
    else
        for (int k = 0; k < n; ++k) a = fma(Gs[k + r * ld], v[k], a);
    return a;
}
__device__ __forceinline__ double dot_glob(const double* M, int n, int r, const double* v, bool transpose) {
    double a = 0.0;
    if (!transpose)
        for (int k = 0; k < n; ++k) a = fma(M[r + (size_t)k * n], v[k], a);
    else
        for (int k = 0; k < n; ++k) a = fma(M[k + (size_t)r * n], v[k], a);
    return a;
}

// ---- right-hand sides -----------------------------------------------------------------------------
// tables: for the first 1+np vectors v (x and first-order): PG[v] = G v, PA[i][v] = A_i v, PB[i][v] = B_i v, PD[j][v] = D_j v
struct Tables {
    double *PG, *PA, *PB, *PD;
    int nv1;  // 1 + np
};

__device__ __forceinline__ double Ci(const Tables& T, const Scal& S, int n, int i, int v, int r) {  // (C_i Z_v)[r]
    return S.c[i] * T.PA[((size_t)i * T.nv1 + v) * n + r] + S.s[i] * T.PB[((size_t)i * T.nv1 + v) * n + r];
}
__device__ __forceinline__ double Cpi(const Tables& T, const Scal& S, int n, int i, int v, int r) {  // (dC_i/dt Z_v)[r]
    return S.om[i] * (-S.s[i] * T.PA[((size_t)i * T.nv1 + v) * n + r] + S.c[i] * T.PB[((size_t)i * T.nv1 + v) * n + r]);
}
__device__ double Gt_v(const Tables& T, const Scal& S, const Ctx& C, int v, int r) {  // (dG/dt Z_v)[r]
    double a = 0.0;
    for (int i = 0; i < C.m; ++i) a = fma(S.u[i], Cpi(T, S, C.n, i, v, r), a);
    for (int j = 0; j < C.nc; ++j) a = fma(-S.omd[j] * S.es[j], T.PD[((size_t)j * T.nv1 + v) * C.n + r], a);
    return a;
}
__device__ double Gtt_v(const Tables& T, const Scal& S, const Ctx& C, int v, int r) {  // (d2G/dt2 Z_v)[r]
    double a = 0.0;
    for (int i = 0; i < C.m; ++i) a = fma(-S.u[i] * S.om[i] * S.om[i], Ci(T, S, C.n, i, v, r), a);
    for (int j = 0; j < C.nc; ++j) a = fma(-S.omd[j] * S.omd[j] * S.e[j], T.PD[((size_t)j * T.nv1 + v) * C.n + r], a);
    return a;
}
// parameter index helpers: [u0 (m), u1 (m, order 1), dt, t]
__device__ __forceinline__ int p_dt(const Ctx& C) { return C.np - 2; }
__device__ __forceinline__ int p_t(const Ctx& C) { return C.np - 1; }

// (dM/dtheta_a Z_v)[r]
__device__ double Ma_v(const Tables& T, const Scal& S, const Ctx& C, int a, int v, int r) {
    const int nu = C.np - 2;
    if (a < nu) {
        const int i = a % C.m;
        const double w = a < C.m ? S.w0 : S.w1;
        return S.dt * w * Ci(T, S, C.n, i, v, r);
    }
    if (a == p_dt(C)) return T.PG[(size_t)v * C.n + r] + S.dt * S.tau * Gt_v(T, S, C, v, r);
    return S.dt * Gt_v(T, S, C, v, r);
}
// (d2M/(dtheta_a dtheta_b) x)[r], a <= b
__device__ double Mab_x(const Tables& T, const Scal& S, const Ctx& C, int a, int b, int r) {
    const int nu = C.np - 2;
    if (b < nu) return 0.0;  // u-u
    if (a < nu) {
        const int i = a % C.m;
        const double w = a < C.m ? S.w0 : S.w1;
        if (b == p_dt(C)) return w * (Ci(T, S, C.n, i, 0, r) + S.dt * S.tau * Cpi(T, S, C.n, i, 0, r));
        return S.dt * w * Cpi(T, S, C.n, i, 0, r);
    }
    if (a == p_dt(C) && b == p_dt(C)) return 2.0 * S.tau * Gt_v(T, S, C, 0, r) + S.dt * S.tau * S.tau * Gtt_v(T, S, C, 0, r);
    if (a == p_dt(C)) return Gt_v(T, S, C, 0, r) + S.dt * S.tau * Gtt_v(T, S, C, 0, r);
    return S.dt * Gtt_v(T, S, C, 0, r);
}

// D = L(tau) Zc for the role's vector set.  nvec vectors of length n, vector-major.
__device__ void rhs(int role, const Ctx& C, const Scal& S, const Tables& T, const double* Zc, double* Dv, int nvec) {
    const int n = C.n, tid = threadIdx.x, nt = blockDim.x;
    const bool tr = role == ROLE_ADJ;
    if (role == ROLE_EXP) {
        for (int e = tid; e < nvec * n; e += nt) {
            const int v = e / n, r = e % n;
            Dv[e] = S.dt * dot_smem(C.Gs, C.ld, r, Zc + (size_t)v * n, n, false);
        }
        __syncthreads();
        return;
    }
    const int nv1 = T.nv1;  // FWD: 1 + np ; ADJ: 1 (only lambda feeds the coupling terms)
    // products with G for every vector; basis products for the leading nv1 vectors
    const int nbasis = 2 * C.m + C.nc;
    for (int e = tid; e < (nvec + nbasis * nv1) * n; e += nt) {
        const int item = e / n, r = e % n;
        if (item < nvec) {
            const double a = dot_smem(C.Gs, C.ld, r, Zc + (size_t)item * n, n, tr);
            if (item < nv1) T.PG[(size_t)item * n + r] = a;
            Dv[(size_t)item * n + r] = S.dt * a;
        } else {
            const int bi = (item - nvec) / nv1, v = (item - nvec) % nv1;
            const double* vec = Zc + (size_t)v * n;
            if (bi < C.m) T.PA[((size_t)bi * nv1 + v) * n + r] = dot_glob(C.A + (size_t)bi * n * n, n, r, vec, tr);
            else if (bi < 2 * C.m) T.PB[((size_t)(bi - C.m) * nv1 + v) * n + r] = dot_glob(C.B + (size_t)(bi - C.m) * n * n, n, r, vec, tr);
            else T.PD[((size_t)(bi - 2 * C.m) * nv1 + v) * n + r] = dot_glob(C.D + (size_t)(bi - 2 * C.m) * n * n, n, r, vec, tr);
        }
    }
    __syncthreads();
    const int np = C.np;
    if (role == ROLE_FWD) {
        for (int e = tid; e < (nvec - 1) * n; e += nt) {
            const int v = 1 + e / n, r = e % n;
            double add;
            if (v <= np) {
                add = Ma_v(T, S, C, v - 1, 0, r);
            } else {
                int p = v - 1 - np, a = 0;
                while (p >= np - a) {
                    p -= np - a;
                    ++a;
                }
                const int b = a + p;
                add = Ma_v(T, S, C, a, 1 + b, r) + Ma_v(T, S, C, b, 1 + a, r) + Mab_x(T, S, C, a, b, r);
            }
            Dv[(size_t)v * n + r] += add;
        }
    } else {  // ADJ: d lambda^a = M' lambda^a + (M^a)' lambda
        for (int e = tid; e < (nvec - 1) * n; e += nt) {
            const int v = 1 + e / n, r = e % n;
            Dv[(size_t)v * n + r] += Ma_v(T, S, C, v - 1, 0, r);
        }
    }
    __syncthreads();
}

__global__ void __launch_bounds__(kThreads) tdb_kernel(DProb P, int ii, const double* __restrict__ Z, const double* __restrict__ mu,
                                                       double* __restrict__ g, double* __restrict__ jac, int want_jac, int want_hess,
                                                       int Kmax) {
    extern __shared__ double sm[];
    const DInt& I = P.in[ii];
    const int n = I.n, m = I.m, z = P.z, tid = threadIdx.x, nt = blockDim.x;
    const int nIc = min(P.kc1, P.nI) - P.kc0;  // intervals of the active range
    const int b = blockIdx.x / nIc, kl = P.kc0 + blockIdx.x % nIc;
    int role = blockIdx.y;
    if (role == 1 && !want_jac) role = ROLE_ADJ;
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * z;
    const double* zk1 = zk + z;
    if (P.halo != nullptr && kl + 1 == P.nK - 1) zk1 = P.halo;
    double poison;
    int Ki;
    const int steps = tdb_item_steps(I, zk, zk1, P.dt_off, poison, Kmax, Ki);
    const int K = Ki;  // extrapolation columns of THIS interval

    Ctx C;
    C.n = n;
    C.m = m;
    C.nc = I.n_carrier;
    C.order = I.order;
    C.np = (I.order == 1 ? 2 * m : m) + 2;
    C.ld = n | 1;
    C.G0 = I.G;
    C.A = I.A;
    C.B = I.B;
    C.D = I.D;
    const int np = C.np, npairs = np * (np + 1) / 2;
    int nvec;
    if (role == ROLE_FWD) nvec = want_hess ? 1 + np + npairs : (want_jac ? 1 + np : 1);
    else if (role == ROLE_EXP) nvec = n;
    else nvec = 1 + np;
    const int nv1 = role == ROLE_FWD ? (nvec > 1 ? (want_hess ? 1 + np : 1) : 0) : (role == ROLE_ADJ ? 1 : 0);
    const int nbasis = 2 * m + C.nc;

    C.Gs = sm;
    double* Zp = C.Gs + (size_t)C.ld * n;
    double* Zc = Zp + (size_t)nvec * n;
    double* Acc = Zc + (size_t)nvec * n;
    double* Y0 = Acc + (size_t)nvec * n;
    double* Dv = Y0 + (size_t)nvec * n;
    Tables T;
    T.nv1 = nv1 > 0 ? nv1 : 1;
    T.PG = Dv + (size_t)nvec * n;
    T.PA = T.PG + (size_t)T.nv1 * n;
    T.PB = T.PA + (size_t)m * T.nv1 * n;
    T.PD = T.PB + (size_t)m * T.nv1 * n;
    (void)nbasis;

    // extrapolation weights w_k = prod_{l != k} n_k^2 / (n_k^2 - n_l^2), n_k = 2(k+1)
    double wk[kMaxCols];
    for (int k = 0; k < K; ++k) {
        double w = 1.0;
        const double nk2 = 4.0 * (k + 1) * (k + 1);
        for (int l = 0; l < K; ++l)
            if (l != k) w *= nk2 / (nk2 - 4.0 * (l + 1) * (l + 1));
        wk[k] = w;
    }
    const long long mu_off = (long long)b * P.n_cons_local + I.row_off + (long long)kl * n;

    // initial values
    for (int e = tid; e < nvec * n; e += nt) {
        const int v = e / n, r = e % n;
        double val = 0.0;
        if (role == ROLE_FWD) val = v == 0 ? zk[I.x_off + r] : 0.0;
        else if (role == ROLE_EXP) val = v == r ? 1.0 : 0.0;
        else val = v == 0 ? mu[mu_off + r] : 0.0;
        Y0[e] = val * poison;
    }
    __syncthreads();

    // the ODE variable is tau in [0,1] (ADJ: s = 1 - tau, generator transposed); `steps` macro steps
    // a FWD role that only needs the value still takes this path with nvec = 1 (rhs skips the couplings)
    const bool couple = (role == ROLE_FWD && nvec > 1) || role == ROLE_ADJ;
    for (int ms = 0; ms < steps; ++ms) {
        const double H = 1.0 / steps, s0 = ms * H;
        for (int e = tid; e < nvec * n; e += nt) Acc[e] = 0.0;
        for (int k = 0; k < K; ++k) {
            const int nk = 2 * (k + 1);
            const double h = H / nk;
            Scal S;
            auto eval = [&](double s, const double* Zin) {
                const double tau = role == ROLE_ADJ ? 1.0 - s : s;
                make_scal(I, zk, zk1, P.dt_off, tau, S);
                __syncthreads();
                assemble_G(C, S);
                __syncthreads();
                if (couple || role == ROLE_EXP) rhs(role, C, S, T, Zin, Dv, nvec);
                else {  // value-only forward
                    for (int e = tid; e < n; e += nt) Dv[e] = S.dt * dot_smem(C.Gs, C.ld, e, Zin, n, false);
                    __syncthreads();
                }
            };
            // z0 = Y0 ; z1 = z0 + h f(s0, z0)
            eval(s0, Y0);
            for (int e = tid; e < nvec * n; e += nt) {
                Zp[e] = Y0[e];
                Zc[e] = Y0[e] + h * Dv[e];
            }
            __syncthreads();
            for (int q = 1; q < nk; ++q) {
                eval(s0 + q * h, Zc);
                for (int e = tid; e < nvec * n; e += nt) {
                    const double znew = Zp[e] + 2.0 * h * Dv[e];
                    Zp[e] = Zc[e];
                    Zc[e] = znew;
                }
                __syncthreads();
            }
            eval(s0 + H, Zc);
            for (int e = tid; e < nvec * n; e += nt) Acc[e] += wk[k] * 0.5 * (Zc[e] + Zp[e] + h * Dv[e]);
            __syncthreads();
        }
        for (int e = tid; e < nvec * n; e += nt) Y0[e] = Acc[e];
        __syncthreads();
    }
    const double* F = Y0;

    // ---- outputs ----
    const int nu = np - 2;
    if (role == ROLE_FWD) {
        if (g != nullptr)
            for (int r = tid; r < n; r += nt) g[mu_off + r] = zk1[I.x_off + r] - F[r];
        if (want_jac) {
            double* jp = jac + (long long)b * P.nnz_jac_local;
            const long long own_off = jac_own_off(P, kl, I.doff, n);
            const long long prev_off = jac_prev_off(P, kl + 1, I.doff);
            for (int e = tid; e < 2 * z * n; e += nt) {
                const int l = e / n, a = e % n;
                double v = 0.0;
                long long pos;
                if (l < z) {
                    if (l >= I.x_off && l < I.x_off + n) continue;  // EXP role
                    if (l >= I.u_off && l < I.u_off + m) v = -F[(size_t)(1 + (l - I.u_off)) * n + a];
                    else if (l == P.dt_off) v = -F[(size_t)(1 + nu) * n + a];
                    else if (l == I.t_off) v = -F[(size_t)(2 + nu) * n + a];
                    pos = jac_col(P, kl, l) + own_off + a;
                } else {
                    const int lp = l - z;
                    if (lp - I.x_off == a) v = 1.0;
                    if (I.order == 1 && lp >= I.u_off && lp < I.u_off + m) v = -F[(size_t)(1 + m + (lp - I.u_off)) * n + a];
                    pos = jac_col(P, (kl + 1), lp) + prev_off + a;
                }
                jp[pos] = v;
            }
        }
        if (want_hess) {
            double* hpp = I.hs + ((long long)b * P.nI + kl) * I.hs_stride + (long long)np * n;
            const int warp = tid >> 5, lane = tid & 31, nwarp = nt >> 5;
            for (int p = warp; p < npairs; p += nwarp) {
                int pp = p, a = 0;
                while (pp >= np - a) {
                    pp -= np - a;
                    ++a;
                }
                const int bb = a + pp;
                double s = 0.0;
                for (int r = lane; r < n; r += 32) s = fma(mu[mu_off + r], F[(size_t)(1 + np + p) * n + r], s);
                s = warp_sum(s);
                if (lane == 0) {
                    hpp[a * np + bb] = -s;
                    hpp[bb * np + a] = -s;
                }
            }
        }
    } else if (role == ROLE_EXP) {
        double* jp = jac + (long long)b * P.nnz_jac_local;
        const long long own_off = jac_own_off(P, kl, I.doff, n);
        for (int e = tid; e < n * n; e += nt) {
            const int c = e / n, a = e % n;  // column c of Phi = vector c
            jp[jac_col(P, kl, I.x_off + c) + own_off + a] = -F[(size_t)c * n + a];
        }
    } else {
        double* hx = I.hs + ((long long)b * P.nI + kl) * I.hs_stride;
        for (int e = tid; e < np * n; e += nt) hx[e] = -F[(size_t)n + e];
    }
}

size_t tdb_smem_bytes(const DInt& I, bool want_jac, bool want_hess) {
    const int n = I.n, m = I.m, np = (I.order == 1 ? 2 * m : m) + 2, npairs = np * (np + 1) / 2;
    size_t worst = 0;
    for (int role = 0; role < 3; ++role) {
        int nvec = role == 0 ? (want_hess ? 1 + np + npairs : (want_jac ? 1 + np : 1)) : (role == 1 ? n : 1 + np);
        int nv1 = role == 0 ? (want_hess ? 1 + np : 1) : 1;
        if (role == 1 && !want_jac) continue;
        if (role == 2 && !want_hess) continue;
        size_t d = (size_t)(n | 1) * n + 5 * (size_t)nvec * n + (size_t)nv1 * n * (1 + 2 * m + I.n_carrier);
        worst = d > worst ? d : worst;
    }
    return worst * sizeof(double);
}

}  // namespace

bool tdb_available() { return true; }

void launch_tdb(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, cudaStream_t st,
                long long* launches) {
    const DInt& I = P.in[ii];
    const int nIc = std::min(P.kc1, P.nI) - P.kc0;
    if (nIc <= 0) return;
    const size_t smem = tdb_smem_bytes(I, f.want_jac, f.want_hess);
    static PerDeviceOnce configured;
    if (configured.first()) {
        cudaFuncSetAttribute(tdb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    }
    const int K = 8;
    dim3 grid((unsigned)(nIc * P.batch), 1 + (f.want_jac ? 1 : 0) + (f.want_hess ? 1 : 0));
    tdb_kernel<<<grid, kThreads, smem, st>>>(P, ii, Z, mu, f.want_g ? g : nullptr, jac, f.want_jac ? 1 : 0, f.want_hess ? 1 : 0, K);
    ++*launches;
}

bool tdb_fits(const DInt& I, size_t smem_limit) {
    return I.m <= kMaxM && I.n_carrier <= kMaxC && tdb_smem_bytes(I, true, true) <= smem_limit;
}

// K7 (DMMA variant): TimeDependentBilinearIntegrator interval kernel on the FP64 tensor pipe.
//
// Same mathematics as tdb.cu (Gragg-Bulirsch-Stoer extrapolation of the exact first/second-order
// variational equations of  dPhi/dtau = dt G(u(tau), t_k + tau dt) Phi  for the carrier family
//     G(u, t) = G0 + sum_i u_i (cos(w_i t + phi_i) A_i + sin(w_i t + phi_i) B_i) + sum_j cos(wd_j t + phd_j) D_j,
// replacing solve(ODEProblem, Tsit5()) + ForwardDiff of
// /root/reference/src/integrators/time_dependent_bilinear_integrator.jl:102-128,145-244), different mapping:
//
// One CTA per (problem, interval).  Every warp owns ONE 8-row tile of vectors for the whole integration and
// keeps it in registers in tensor-core fragment layout (dmma_tiles.cuh): the modified-midpoint update
// z_{q+1} = z_{q-1} + 2h f(z_q) is element-wise, and the C fragment of G(tau) * tile is already the A
// fragment of the next right-hand side, so the vectors never touch shared memory:
//   FWD tiles  [x; dx/dtheta_a; d2x/dtheta_a dtheta_b], theta = [u_k (m), u_{k+1} (m, order 1), dt, t_k]
//   EXP tiles  columns of the identity -> Phi(1), the -Phi Jacobian block
//   ADJ tile   [lambda; dlambda/dtheta_a] in reflected time through G' -> (dPhi/dtheta)' mu
// Per right-hand side the CTA (1) assembles G(tau) and G(1 - tau)' in shared memory from the basis matrices
// (swizzled row-major copies in global memory, L2-resident), (2) every warp multiplies its tile by it, the
// basis products A_i, B_i, D_j times the leading forward tile (needed by the parameter couplings) are spread
// over the lightly loaded warps, the transposed basis products of lambda run on the FP64 FMA pipe, (3) the
// couplings are added from the shared tables.  Two block barriers per right-hand side.
#include <stdlib.h>

#include "dmma_tiles.cuh"
#include "dto_internal.h"

namespace {

using namespace dmma_tiles;

constexpr int kMaxM = 4;      // drives
constexpr int kMaxC = 4;      // carriers
constexpr int kMaxCols = 10;  // extrapolation columns
constexpr int kMaxWarpsT = 16;  // 16 warps x 128 registers (the allocation granularity makes 13..16 warps cost the same)

struct Scal {  // what the generator assembly needs at one node
    double dt;
    double u[kMaxM], c[kMaxM], s[kMaxM];
    double e[kMaxC];
    double pad_;
};

struct Ctx {
    int n, m, nc, order, np;
};

// Node values NV[]: every coupling coefficient of the jet recurrence is  NV[i1] NV[i2] + NV[i3] NV[i4]  (times the step
// factor) with indices that depend only on the (row, slot, table) position, not on the node.  One array per node, written
// by the lane that evaluates the node's sines and cosines.
enum { NV_ONE = 0, NV_ZERO, NV_DT, NV_DTTAU, NV_2TAU, NV_DTTAU2, NV_W0, NV_W1, NV_DTW0, NV_DTW1, NV_W0DTTAU, NV_W1DTTAU, NV_BASE };
// per drive i, 8 values at NV_BASE + 8 i:  C_i = (c, s);  C_i' = w (-s, c);  dG/dt part u w (-s, c);  d2G/dt2 part -u w^2 (c, s)
enum { ND_C = 0, ND_S, ND_CP_A, ND_CP_B, ND_GT_A, ND_GT_B, ND_GTT_A, ND_GTT_B };
// per carrier j, 2 values at NV_BASE + 8 m + 2 j:  dG/dt part -wd sin,  d2G/dt2 part -wd^2 cos
__host__ __device__ inline int nv_count(int m, int nc) { return NV_BASE + 8 * m + 2 * nc; }

__device__ void make_scal(const DInt& I, const double* zk, const double* zk1, int dt_off, double tau, Scal& S, double* nv) {
    const double dt = zk[dt_off];
    S.dt = dt;
    const double t = zk[I.t_off] + tau * dt;
    const double w0 = I.order == 1 ? 1.0 - tau : 1.0, w1 = I.order == 1 ? tau : 0.0;
    if (nv != nullptr) {
        nv[NV_ONE] = 1.0;
        nv[NV_ZERO] = 0.0;
        nv[NV_DT] = dt;
        nv[NV_DTTAU] = dt * tau;
        nv[NV_2TAU] = 2.0 * tau;
        nv[NV_DTTAU2] = dt * tau * tau;
        nv[NV_W0] = w0;
        nv[NV_W1] = w1;
        nv[NV_DTW0] = dt * w0;
        nv[NV_DTW1] = dt * w1;
        nv[NV_W0DTTAU] = w0 * dt * tau;
        nv[NV_W1DTTAU] = w1 * dt * tau;
    }
    for (int i = 0; i < I.m; ++i) {
        const double u0 = zk[I.u_off + i], u1 = I.order == 1 ? zk1[I.u_off + i] : u0;
        const double u = w0 * u0 + w1 * u1, om = I.omega[i];
        double sn, cs;
        sincos(om * t + I.phi[i], &sn, &cs);
        S.u[i] = u;
        S.c[i] = cs;
        S.s[i] = sn;
        if (nv != nullptr) {
            double* d = nv + NV_BASE + 8 * i;
            d[ND_C] = cs;
            d[ND_S] = sn;
            d[ND_CP_A] = -om * sn;
            d[ND_CP_B] = om * cs;
            d[ND_GT_A] = u * om * (-sn);
            d[ND_GT_B] = u * om * cs;
            d[ND_GTT_A] = -u * om * om * cs;
            d[ND_GTT_B] = -u * om * om * sn;
        }
    }
    for (int j = 0; j < I.n_carrier; ++j) {
        const double omd = I.omega_d[j];
        double es, ec;
        sincos(omd * t + I.phi_d[j], &es, &ec);
        S.e[j] = ec;
        if (nv != nullptr) {
            nv[NV_BASE + 8 * I.m + 2 * j] = -omd * es;
            nv[NV_BASE + 8 * I.m + 2 * j + 1] = -omd * omd * ec;
        }
    }
}

// ---- parameter couplings ------------------------------------------------------------------------------------------
// Tables (shared memory): T_0[v] = G Z_v (before the dt factor), T_{1+i}[v] = A_i Z_v, T_{1+m+i}[v] = B_i Z_v,
// T_{1+2m+j}[v] = D_j Z_v.  The coupling of a row is  sum_t coef[t] * T_t[source row]  with, per (row, slot):
//   first-order row a:  slot 0 = dM/dtheta_a            (source row 0 = x)
//   pair row (a, b):    slot 0 = M_a (2 M_a if a == b)  (source row 1 + b)
//                       slot 1 = M_b                    (source row 1 + a, a != b)
//                       slot 2 = M_ab                   (source row 0)
// M = dt G(u(tau), t_k + tau dt), theta = [u_k (m), u_{k+1} (m, order 1), dt, t_k];  dG/dt, d2G/dt2 act on the carriers.
// coef_indices() gives the NV indices of entry t of one of those matrices' coefficient vectors:
//   value = NV[i1] NV[i2] + NV[i3] NV[i4]      (packed i1 | i2 << 8 | i3 << 16 | i4 << 24)
enum { AT_ZERO = 0, AT_EG, AT_GT, AT_GTT, AT_C, AT_CP };
__device__ __forceinline__ int atom_index(int atom, int i, int t, int m) {  // NV index of component t of an atom
    if (atom == AT_ZERO) return NV_ZERO;
    if (atom == AT_EG) return t == 0 ? NV_ONE : NV_ZERO;
    if (t == 0) return NV_ZERO;
    if (t <= 2 * m) {
        const bool isb = t > m;
        const int it = isb ? t - 1 - m : t - 1;
        const int base = NV_BASE + 8 * it;
        if (atom == AT_GT) return base + (isb ? ND_GT_B : ND_GT_A);
        if (atom == AT_GTT) return base + (isb ? ND_GTT_B : ND_GTT_A);
        if (it != i) return NV_ZERO;
        if (atom == AT_C) return base + (isb ? ND_S : ND_C);
        return base + (isb ? ND_CP_B : ND_CP_A);
    }
    const int j = t - 1 - 2 * m;
    if (atom == AT_GT) return NV_BASE + 8 * m + 2 * j;
    if (atom == AT_GTT) return NV_BASE + 8 * m + 2 * j + 1;
    return NV_ZERO;
}
// dM/dtheta_a -> (atom A, scalar A, atom B, scalar B, drive index)
__device__ __forceinline__ void terms_Ma(const Ctx& C, int a, int& aA, int& sA, int& aB, int& sB, int& drive) {
    const int nu = C.np - 2;
    aA = aB = AT_ZERO;
    sA = sB = NV_ZERO;
    drive = 0;
    if (a < nu) {  // dt w C_i
        drive = a % C.m;
        aA = AT_C;
        sA = a < C.m ? NV_DTW0 : NV_DTW1;
    } else if (a == nu) {  // G + dt tau dG/dt
        aA = AT_EG;
        sA = NV_ONE;
        aB = AT_GT;
        sB = NV_DTTAU;
    } else {  // dt dG/dt
        aA = AT_GT;
        sA = NV_DT;
    }
}
// d2M/(dtheta_a dtheta_b), a <= b
__device__ __forceinline__ void terms_Mab(const Ctx& C, int a, int b, int& aA, int& sA, int& aB, int& sB, int& drive) {
    const int nu = C.np - 2;
    aA = aB = AT_ZERO;
    sA = sB = NV_ZERO;
    drive = 0;
    if (b < nu) return;  // u-u
    if (a < nu) {
        drive = a % C.m;
        const bool k0 = a < C.m;
        if (b == nu) {  // w (C_i + dt tau C_i')
            aA = AT_C;
            sA = k0 ? NV_W0 : NV_W1;
            aB = AT_CP;
            sB = k0 ? NV_W0DTTAU : NV_W1DTTAU;
        } else {  // dt w C_i'
            aA = AT_CP;
            sA = k0 ? NV_DTW0 : NV_DTW1;
        }
        return;
    }
    if (a == nu && b == nu) {  // 2 tau dG/dt + dt tau^2 d2G/dt2
        aA = AT_GT;
        sA = NV_2TAU;
        aB = AT_GTT;
        sB = NV_DTTAU2;
    } else if (a == nu) {  // dG/dt + dt tau d2G/dt2
        aA = AT_GT;
        sA = NV_ONE;
        aB = AT_GTT;
        sB = NV_DTTAU;
    } else {  // dt d2G/dt2
        aA = AT_GTT;
        sA = NV_DT;
    }
}

// NV indices of coefficient-table entry `en` = ((row * 3 + slot) * KCr + t): packed i1 | i2 << 8 | i3 << 16 | i4 << 24, and
// whether the entry carries the factor 2 of a diagonal pair.  Rows [0, nrowsF) are the forward rows 1.., then np adjoint rows.
__device__ int coef_entry(const Ctx& C, int KCr, int nrowsF, int en, bool& twice) {
    const int t = en % KCr, it = en / KCr, slot = it % 3, r = it / 3, np = C.np;
    int aA = AT_ZERO, sA = NV_ZERO, aB = AT_ZERO, sB = NV_ZERO, drive = 0;
    twice = false;
    if (r < nrowsF) {
        const int v = r + 1;
        if (v <= np) {
            if (slot == 0) terms_Ma(C, v - 1, aA, sA, aB, sB, drive);
        } else {
            int pp = v - 1 - np, a = 0;
            while (a < np && pp >= np - a) {
                pp -= np - a;
                ++a;
            }
            const int bb = a + pp;
            if (slot == 0) {
                terms_Ma(C, a, aA, sA, aB, sB, drive);
                twice = a == bb;
            } else if (slot == 1) {
                if (a != bb) terms_Ma(C, bb, aA, sA, aB, sB, drive);
            } else {
                terms_Mab(C, a, bb, aA, sA, aB, sB, drive);
            }
        }
    } else if (slot == 0) {
        terms_Ma(C, r - nrowsF, aA, sA, aB, sB, drive);
    }
    return atom_index(aA, drive, t, C.m) | (sA << 8) | (atom_index(aB, drive, t, C.m) << 16) | (sB << 24);
}

// D += cf * row   (this lane's states 8 nt + 2q + {0,1})
template <int NT>
__device__ __forceinline__ void axpy_row(double (&D)[1][NT][2], double cf, const double* src) {
    if (cf == 0.0) return;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        const double2 x = *reinterpret_cast<const double2*>(src + 8 * nt);
        D[0][nt][0] = fma(cf, x.x, D[0][nt][0]);
        D[0][nt][1] = fma(cf, x.y, D[0][nt][1]);
    }
}
enum { W_FWD = 0, W_EXP = 1, W_ADJ = 2, W_IDLE = 3 };

#ifdef DTO_TDB_PROFILE
// debug build only (DTO_EXTRA_NVCC_FLAGS=-DDTO_TDB_PROFILE): cycles of CTA x = 0 per warp and segment of a right-hand side
__device__ unsigned long long g_tdb_prof[2][16][8];
#endif

// out += V * M' for one tile, the output n-tiles in two halves (half the B fragments live at a time)
template <int NT>
__device__ __forceinline__ void mma_tile(double (&out)[1][NT][2], const double (&v)[1][NT][2], const double* __restrict__ M, int lane) {
    constexpr int n = 8 * NT, NH = (NT + 1) / 2;
    const int row8 = lane >> 2;
    const int d = (NT % 2 == 0) ? ((row8 & 1) << 3) : 0;
    const double* base = M + row8 * n + 2 * (lane & 3);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int off = 8 * t + ((t & 1) ? -d : d);
            double2 bf[NH];
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) bf[x] = *reinterpret_cast<const double2*>(base + 8 * (half * NH + x) * n + off);
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) dmma(out[0][half * NH + x][0], out[0][half * NH + x][1], v[0][t][0], bf[x].x);
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) dmma(out[0][half * NH + x][0], out[0][half * NH + x][1], v[0][t][1], bf[x].y);
        }
    }
}

// R += s * (V * M') for one tile, by output halves: only half a tile of accumulators is live beside the two state tiles
// (previous and current vector of the midpoint rule), so that 16 warps fit the register file without spills.  The raw
// products go to `tab` (this lane's row of a coupling table, 8 doubles apart per n-tile) when `to_tab` is set.
template <int NT>
__device__ __forceinline__ void mma_tile_axpy(double (&R)[1][NT][2], const double (&v)[1][NT][2], const double* __restrict__ M, double s, int lane,
                                              double* __restrict__ tab, bool to_tab) {
    constexpr int n = 8 * NT, NH = (NT + 1) / 2;
    const int row8 = lane >> 2;
    const int d = (NT % 2 == 0) ? ((row8 & 1) << 3) : 0;
    const double* base = M + row8 * n + 2 * (lane & 3);
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        double acc[NH][2];
#pragma unroll
        for (int x = 0; x < NH; ++x) acc[x][0] = acc[x][1] = 0.0;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int off = 8 * t + ((t & 1) ? -d : d);
            double2 bf[NH];
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) bf[x] = *reinterpret_cast<const double2*>(base + 8 * (half * NH + x) * n + off);
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) dmma(acc[x][0], acc[x][1], v[0][t][0], bf[x].x);
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) dmma(acc[x][0], acc[x][1], v[0][t][1], bf[x].y);
        }
#pragma unroll
        for (int x = 0; x < NH; ++x) {
            const int nt = half * NH + x;
            if (nt < NT) {
                if (to_tab) {
                    tab[8 * nt] = acc[x][0];
                    tab[8 * nt + 1] = acc[x][1];
                }
                R[0][nt][0] = fma(s, acc[x][0], R[0][nt][0]);
                R[0][nt][1] = fma(s, acc[x][1], R[0][nt][1]);
            }
        }
    }
}

// R += s * (V * M) for one tile with M in the forward (row-major, swizzled) layout, i.e. the product with the TRANSPOSE of the
// matrix mma_tile_axpy would use: B fragments are read by columns (two 8-byte loads per pair of k-steps, 4-way bank conflicts).
// Only the adjoint tile uses it -- one warp -- in exchange for a generator assembly without the transposed, scattered stores.
template <int NT>
__device__ __forceinline__ void mma_tile_axpy_T(double (&R)[1][NT][2], const double (&v)[1][NT][2], const double* __restrict__ M, double s, int lane,
                                                double* __restrict__ tab, bool to_tab) {
    constexpr int n = 8 * NT, NH = (NT + 1) / 2;
    const int row8 = lane >> 2, q = lane & 3;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        double acc[NH][2];
#pragma unroll
        for (int x = 0; x < NH; ++x) acc[x][0] = acc[x][1] = 0.0;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int k0 = 8 * t + 2 * q;  // k-steps (t, 0) and (t, 1) contract over states k0 and k0 + 1: rows of M
            const double* r0 = M + k0 * n;
            const double* r1 = r0 + n;
            double b0[NH], b1[NH];
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) {
                    const int col = 8 * (half * NH + x) + row8;
                    b0[x] = r0[(NT % 2 == 0) ? col : col];                   // even row: not swizzled
                    b1[x] = r1[(NT % 2 == 0) ? (col ^ 8) : col];             // odd row: 8-double blocks swapped pairwise
                }
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) dmma(acc[x][0], acc[x][1], v[0][t][0], b0[x]);
#pragma unroll
            for (int x = 0; x < NH; ++x)
                if (half * NH + x < NT) dmma(acc[x][0], acc[x][1], v[0][t][1], b1[x]);
        }
#pragma unroll
        for (int x = 0; x < NH; ++x) {
            const int nt = half * NH + x;
            if (nt < NT) {
                if (to_tab) {
                    tab[8 * nt] = acc[x][0];
                    tab[8 * nt + 1] = acc[x][1];
                }
                R[0][nt][0] = fma(s, acc[x][0], R[0][nt][0]);
                R[0][nt][1] = fma(s, acc[x][1], R[0][nt][1]);
            }
        }
    }
}

// basis matrix b (0..2m+nc-1) of the swizzled row-major copies
__device__ __forceinline__ const double* basis_global(const DInt& I, int b, int nn) {
    if (b < I.m) return I.Asw + (size_t)b * nn;
    if (b < 2 * I.m) return I.Bsw + (size_t)(b - I.m) * nn;
    return I.Dsw + (size_t)(b - 2 * I.m) * nn;
}

// G(tau) -> Gf and G(1 - tau) -> Ga (both in the forward layout) from the drift entries already sitting in Gf (cp.async) and the basis matrices.
// A 4 x 8 block of the matrix per warp pass: few bank conflicts on both the straight and the transposed store.
// CACHED: every basis matrix is in the shared cache Bs (plain offset arithmetic in the inner loop).  The node's
// coefficients u_i cos, u_i sin, carrier cos are lifted into registers first (MM drives, CC carriers at most):
// the stores to Gf/Ga would otherwise force the compiler to re-read them from shared memory per element.
template <int NT, bool CACHED, int MM, int CC>
__device__ __forceinline__ void assemble_generators(double* Gf, double* Ga, const double* Bs, const DInt& I, const Scal& Sf, const Scal& Sa,
                                                    int m, int nc, bool want_adj, int b0, int b1, int lane) {
    constexpr int n = 8 * NT, nn = n * n;
    const double* gA = I.Asw;
    const double* gB = I.Bsw;
    const double* gD = I.Dsw;
    double fc[MM], fs[MM], ac[MM], as[MM], fe[CC > 0 ? CC : 1], ae[CC > 0 ? CC : 1];
#pragma unroll
    for (int i = 0; i < MM; ++i) {
        fc[i] = i < m ? Sf.u[i] * Sf.c[i] : 0.0;
        fs[i] = i < m ? Sf.u[i] * Sf.s[i] : 0.0;
        ac[i] = i < m ? Sa.u[i] * Sa.c[i] : 0.0;
        as[i] = i < m ? Sa.u[i] * Sa.s[i] : 0.0;
    }
#pragma unroll
    for (int j = 0; j < CC; ++j) {
        fe[j] = j < nc ? Sf.e[j] : 0.0;
        ae[j] = j < nc ? Sa.e[j] : 0.0;
    }
    // two adjacent columns per thread (16-byte loads and stores; a swizzled pair stays adjacent): an 8 x 8 block of
    // the matrix per warp pass
    for (int blk = b0; blk < b1; ++blk) {
        const int r = (blk / NT) * 8 + (lane >> 2), c = (blk % NT) * 8 + 2 * (lane & 3);
        const int p = sw<NT>(r, c);
        const double2 g0 = *reinterpret_cast<const double2*>(Gf + p);  // the drift entries, prefetched by this very thread
        double vf0 = g0.x, vf1 = g0.y, va0 = g0.x, va1 = g0.y;
#pragma unroll
        for (int i = 0; i < MM; ++i)
            if (i < m) {
                const double2 a = *reinterpret_cast<const double2*>((CACHED ? Bs + i * nn : gA + (size_t)i * nn) + p);
                const double2 bb = *reinterpret_cast<const double2*>((CACHED ? Bs + (m + i) * nn : gB + (size_t)i * nn) + p);
                vf0 = fma(fc[i], a.x, fma(fs[i], bb.x, vf0));
                vf1 = fma(fc[i], a.y, fma(fs[i], bb.y, vf1));
                va0 = fma(ac[i], a.x, fma(as[i], bb.x, va0));
                va1 = fma(ac[i], a.y, fma(as[i], bb.y, va1));
            }
#pragma unroll
        for (int j = 0; j < CC; ++j)
            if (j < nc) {
                const double2 d = *reinterpret_cast<const double2*>((CACHED ? Bs + (2 * m + j) * nn : gD + (size_t)j * nn) + p);
                vf0 = fma(fe[j], d.x, vf0);
                vf1 = fma(fe[j], d.y, vf1);
                va0 = fma(ae[j], d.x, va0);
                va1 = fma(ae[j], d.y, va1);
            }
        *reinterpret_cast<double2*>(Gf + p) = make_double2(vf0, vf1);
        if (want_adj) *reinterpret_cast<double2*>(Ga + p) = make_double2(va0, va1);  // same layout: the adjoint tile reads it by columns
    }
}

// MAXW = 8: up to 255 registers per thread (no spills at n = 64); MAXW = 16: 128 registers
template <int NT, int MAXW>
__global__ void __launch_bounds__(MAXW * 32, 1)
    tdb_dmma_kernel(DProb P, int ii, const double* __restrict__ Z, const double* __restrict__ mu, double* __restrict__ g,
                    double* __restrict__ jac, int want_jac, int want_hess, int Kmax, int TF, int TE, int TA, int split, int nbs,
                    double* __restrict__ scratch) {
    extern __shared__ __align__(16) double sm[];
    constexpr int n = 8 * NT, nn = n * n, FR = NT * 2 * 32;  // FR: doubles of one tile in per-lane fragment order
    const DInt& I = P.in[ii];
    const int m = I.m, nc = I.n_carrier, z = P.z;
    Ctx C{n, m, nc, I.order, (I.order == 1 ? 2 * m : m) + 2};
    const int np = C.np, npairs = np * (np + 1) / 2, nbasis = 2 * m + nc, nu = np - 2;
    const int nwarps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = lane & 3, row8 = lane >> 2;
    if (split) {  // two CTAs per interval: forward + adjoint tiles / propagator tiles
        if (blockIdx.y == 0) TE = 0;
        else TF = TA = 0;
    }
    const int nvecF = TF == 0 ? 0 : (want_hess ? 1 + np + npairs : (want_jac ? 1 + np : 1));
    const bool couple = nvecF > 1;
    const int nv1 = couple ? (want_hess ? 1 + np : 1) : 0;  // leading forward rows whose basis products are needed

    int role = W_IDLE, tile = 0;
    if (warp < TF) { role = W_FWD; tile = warp; }
    else if (warp < TF + TE) { role = W_EXP; tile = warp - TF; }
    else if (warp < TF + TE + TA) { role = W_ADJ; tile = 0; }
    const int scal_warp = nwarps - 1;
    int pair_a = 0, pair_b = 0;  // forward rows beyond 1 + np: the parameter pair (a <= b) of this lane's row
    if (role == W_FWD) {
        int p = 8 * tile + row8 - 1 - np;
        if (p >= 0) {
            int a = 0;
            while (a < np && p >= np - a) {
                p -= np - a;
                ++a;
            }
            pair_a = a;
            pair_b = a + p;
        }
    }

    // ---- shared memory -----------------------------------------------------------------------------------
    double* Gf = sm;                                          // G(tau), swizzled row-major
    double* Ga = Gf + nn;                                     // G(1 - tau)', swizzled row-major
    Scal* scal = reinterpret_cast<Scal*>(Ga + nn);            // [2 buffers][forward, adjoint]
    double* pub0 = reinterpret_cast<double*>(scal + 4);       // leading forward tile in fragment order
    double* lam = pub0 + FR;                                  // lambda (n)
    // table rows are TS doubles apart    // (n + 4: the 8-byte B-fragment reads of the coupling product -- 4 table rows x 8 states per k-step -- and the 16-byte
    // C-fragment stores that fill the tables both spread evenly over the banks)
    constexpr int TS = n + 4;
    double* PG = lam + n;                                     // [8][TS]   G Z_v (before the dt factor)
    double* Pb = PG + 8 * TS;                                 // [nbasis][8][TS]
    double* PGa = Pb + (size_t)nbasis * 8 * TS;               // [n]       G' lambda
    double* PT = PGa + n;                                     // [nbasis][n] basis' lambda
    double* wk = PT + (size_t)nbasis * n;                     // [kMaxCols] extrapolation weights
    // coupling coefficients of the current node, built ONCE per right-hand side (one (row, slot) per thread, during the
    // product phase) instead of by every lane of every forward row: [forward rows 1.. | adjoint rows][3 slots][KCr]
    const int KCr = 1 + 2 * m + nc;
    double* CT = wk + kMaxCols + (kMaxCols & 1);
    const int ctRows = (nvecF > 1 ? nvecF - 1 : 0) + (TA > 0 ? np : 0);
    double* NV = CT + ((size_t)ctRows * 3 * KCr + 1) / 2 * 2;   // [2 buffers][forward, adjoint][NVn] node values
    const int NVn = (nv_count(m, nc) + 1) / 2 * 2;
    double* Bs = NV + 4 * (size_t)NVn;                           // cached basis matrices
    // Coupling GEMM of the forward tiles (phase 3): per k-step this lane's A element comes from CT[ctoff] (or is zero) and
    // its B elements from table row boff; both are fixed for the kernel's lifetime -> packed once: ctoff | boff << 13.
    constexpr int kPackedKS = 10, kNoCoef = 0x1FFF;
    const int nsrc = 1 + np, Kdim = KCr * nsrc;
    const bool packed = Kdim <= 4 * kPackedKS;
    int pk[kPackedKS];
#pragma unroll
    for (int ks = 0; ks < kPackedKS; ++ks) {
        const int k = 4 * ks + q, kc = k < Kdim ? k : Kdim - 1;
        const int t = kc / nsrc, vs = kc - t * nsrc;
        const int v = 8 * tile + row8;
        int slot = -1;
        if (role == W_FWD && v >= 1 && v < nvecF && k < Kdim) {
            if (v <= np) slot = vs == 0 ? 0 : -1;
            else if (vs == 1 + pair_b) slot = 0;
            else if (vs == 1 + pair_a) slot = 1;  // only reached when a != b
            else if (vs == 0) slot = 2;
        }
        pk[ks] = (slot >= 0 ? ((v - 1) * 3 + slot) * KCr + t : kNoCoef) | (((t * 8 + vs) * TS) << 13);
    }
    // Coefficient-table entries this lane rebuilds at every node: the rows of its own tile (forward warps) or the adjoint
    // rows (adjoint warp), entries ct_lo + lane + 32 j.  Their NV indices never change: decoded once, kept packed.
    constexpr int kEntPerLane = 4;
    const int nrowsF = couple ? nvecF - 1 : 0;
    int ct_lo = 0, ct_hi = 0;  // [ct_lo, ct_hi) entries of CT
    if (role == W_FWD && couple) {
        ct_lo = (8 * tile == 0 ? 0 : 8 * tile - 1) * 3 * KCr;
        ct_hi = min(8 * tile + 7, nrowsF) * 3 * KCr;
    } else if (role == W_ADJ) {
        ct_lo = nrowsF * 3 * KCr;
        ct_hi = (nrowsF + np) * 3 * KCr;
    }
    const bool ct_packed = ct_hi - ct_lo <= 32 * kEntPerLane;
    int ctd[kEntPerLane];
    int ct_twice = 0;
#pragma unroll
    for (int j = 0; j < kEntPerLane; ++j) {
        const int en = ct_lo + lane + 32 * j;
        bool tw = false;
        ctd[j] = en < ct_hi ? coef_entry(C, KCr, nrowsF, en, tw) : 0;
        ct_twice |= tw ? 1 << j : 0;
    }
    // extrapolation accumulator and macro-step start of this warp: touched only at sweep boundaries, kept in a
    // per-CTA global scratch (L2-resident) so that shared memory can hold the basis matrices instead
    double* AccS = scratch + (((size_t)blockIdx.y * gridDim.x + blockIdx.x) * kMaxWarpsT + warp) * 2 * FR;
    double* Y0S = AccS + FR;
    for (int i = threadIdx.x; i < nbs * nn; i += blockDim.x) {
        const int bi = i / nn, p = i % nn;
        Bs[i] = basis_global(I, bi, nn)[p];
    }
    auto basis_ptr = [&](int bi) -> const double* { return bi < nbs ? Bs + (size_t)bi * nn : basis_global(I, bi, nn); };
    // The drift matrix does not fit beside the basis cache: every thread copies the entries it will assemble
    // from L2 straight into their place in Gf, asynchronously, while the previous right-hand side finishes.
    // Who assembles G: all warps, except that forward-tile warps with parameter couplings are exempt when at least
    // three other warps exist -- their coupling phase is the long one, and the assembly of node q+1 by the others
    // then overlaps it.  (aw, na) = this warp's index among the assemblers and their number; aw < 0: not one.
    // Who assembles G: every warp takes a contiguous run of 8 x 8 blocks; forward-tile warps with parameter couplings take
    // half a share when at least three other warps exist -- they arrive late from the coupling phase of the previous node,
    // while the others start right after the second barrier.  [ab0, ab1) = this warp's blocks.
    int ab0, ab1;
    {
        const bool light = TF > 0 && (want_hess || want_jac) && nwarps - TF >= 3;
        const int wF = light ? 1 : 2, total = TF * wF + (nwarps - TF) * 2, nblk = nn / 64;
        const int before = warp < TF ? warp * wF : TF * wF + (warp - TF) * 2;
        ab0 = nblk * before / total;
        ab1 = nblk * (before + (warp < TF ? wF : 2)) / total;
    }
    auto prefetch_drift = [&]() {
        for (int blk = ab0; blk < ab1; ++blk) {
            const int p = sw<NT>((blk / NT) * 8 + (lane >> 2), (blk % NT) * 8 + 2 * (lane & 3));
            const unsigned dst = (unsigned)__cvta_generic_to_shared(Gf + p);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(I.Grm + p) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    // PG/Pb and PGa/PT are laid out back to back: table t of the forward set is PG + t*8n, of the adjoint set PGa + t*n

    const int nIc = min(P.kc1, P.nI) - P.kc0;  // intervals of the active range
    const int n_items = nIc * P.batch;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
    const int b = item / nIc, kl = P.kc0 + item % nIc;
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * z;
    const double* zk1 = zk + z;
    if (P.halo != nullptr && kl + 1 == P.nK - 1) zk1 = P.halo;
    double poison;
    int K;  // extrapolation columns of THIS interval
    const int steps = tdb_item_steps(I, zk, zk1, P.dt_off, poison, Kmax, K);  // macro steps of THIS interval
    __syncthreads();  // the previous item's tables and scalars are dead
    if (threadIdx.x < kMaxCols) {
        // w_k = prod_{l != k} n_k^2 / (n_k^2 - n_l^2), n_k = 2(k+1)
        const int k = threadIdx.x;
        double w = 1.0;
        const double nk2 = 4.0 * (k + 1) * (k + 1);
        for (int l = 0; l < K; ++l)
            if (l != k) w *= nk2 / (nk2 - 4.0 * (l + 1) * (l + 1));
        wk[k] = k < K ? w : 0.0;
    }
    const long long mu_off = (long long)b * P.n_cons_local + I.row_off + (long long)kl * n;

    // ---- initial values (fragment element (nt, j): vector 8*tile + row8, state 8*nt + 2q + j) ------------
    {
        const int v = 8 * tile + row8;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int r = 8 * nt + 2 * q + j;
                double val = 0.0;
                if (role == W_FWD) val = v == 0 ? zk[I.x_off + r] : 0.0;
                else if (role == W_EXP) val = v == r ? 1.0 : 0.0;
                else if (role == W_ADJ) val = v == 0 ? mu[mu_off + r] : 0.0;
                if (role != W_IDLE) Y0S[(nt * 2 + j) * 32 + lane] = val * poison;
            }
    }
    if (warp == scal_warp && lane < 2) make_scal(I, zk, zk1, P.dt_off, lane == 0 ? 0.0 : 1.0, scal[lane], NV + (size_t)lane * NVn);
    prefetch_drift();
    __syncthreads();

    // Midpoint rule with TWO state tiles: Zp (z_{q-1}) is updated in place to z_{q+1} = z_{q-1} + 2h f(z_q) -- product and
    // couplings accumulate straight into it -- and then the two tiles trade names.
    double Zp[1][NT][2], Zc[1][NT][2];
    int e = 0;  // right-hand sides evaluated so far (parity selects the scalar buffer)
    for (int ms = 0; ms < steps; ++ms) {
        const double H = 1.0 / steps, s0 = ms * H;
        if (role != W_IDLE)
            for (int i = lane; i < FR; i += 32) AccS[i] = 0.0;
        for (int k = 0; k < K; ++k) {
            const int nk = 2 * (k + 1);
            const double h = H / nk;
            if (role != W_IDLE) {
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    Zc[0][nt][0] = Y0S[(nt * 2) * 32 + lane];
                    Zc[0][nt][1] = Y0S[(nt * 2 + 1) * 32 + lane];
                }
            }
            for (int qq = 0; qq <= nk; ++qq, ++e) {
                const Scal& Sf = scal[(e & 1) * 2];
                const Scal& Sa = scal[(e & 1) * 2 + 1];
                // ---- phase 1: generators of this node, published operands --------------------------------
#ifdef DTO_TDB_PROFILE
                long long tp0 = clock64();
#endif
                asm volatile("cp.async.wait_all;" ::: "memory");
#ifdef DTO_TDB_PROFILE
                long long tp1 = clock64();
#endif
                if (nbs == nbasis && m <= 2 && nc == 0) assemble_generators<NT, true, 2, 0>(Gf, Ga, Bs, I, Sf, Sa, m, nc, TA > 0, ab0, ab1, lane);
                else if (nbs == nbasis) assemble_generators<NT, true, kMaxM, kMaxC>(Gf, Ga, Bs, I, Sf, Sa, m, nc, TA > 0, ab0, ab1, lane);
                else assemble_generators<NT, false, kMaxM, kMaxC>(Gf, Ga, Bs, I, Sf, Sa, m, nc, TA > 0, ab0, ab1, lane);
                if (role == W_FWD && tile == 0 && couple) {
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        pub0[(nt * 2) * 32 + lane] = Zc[0][nt][0];
                        pub0[(nt * 2 + 1) * 32 + lane] = Zc[0][nt][1];
                    }
                }
                // step factor of this node: z_1 = z_0 + h f(z_0); z_{q+1} = z_{q-1} + 2h f(z_q); smoothing uses z_{n-1} + h f(z_n)
                const double hs = (qq == 0 || qq == nk) ? h : 2.0 * h;
                if (ct_hi > ct_lo) {
                    // Coupling coefficients of this node (times the step factor): CT[en] = hs (NV[i1] NV[i2] + NV[i3] NV[i4]).  Every
                    // warp rebuilds the rows of ITS OWN tile (it is their only reader: no hazard with a neighbour still in the
                    // previous node's couplings), here in the assembly phase -- the forward warps do not assemble and the FP64
                    // pipe is not yet busy with this node's products.
                    const double* nv = NV + (size_t)((e & 1) * 2 + (role == W_ADJ ? 1 : 0)) * NVn;  // adjoint rows: the reflected node
                    if (ct_packed) {
#pragma unroll
                        for (int j = 0; j < kEntPerLane; ++j) {
                            const int en = ct_lo + lane + 32 * j;
                            if (en < ct_hi) {
                                const int d = ctd[j];
                                const double va = nv[d & 255] * nv[(d >> 8) & 255];
                                CT[en] = ((ct_twice >> j) & 1 ? 2.0 * hs : hs) * fma(nv[(d >> 16) & 255], nv[(d >> 24) & 255], va);
                            }
                        }
                    } else {
                        for (int en = ct_lo + lane; en < ct_hi; en += 32) {
                            bool tw = false;
                            const int d = coef_entry(C, KCr, nrowsF, en, tw);
                            const double va = nv[d & 255] * nv[(d >> 8) & 255];
                            CT[en] = (tw ? 2.0 * hs : hs) * fma(nv[(d >> 16) & 255], nv[(d >> 24) & 255], va);
                        }
                    }
                }
                if (role == W_ADJ && row8 == 0) {
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        lam[8 * nt + 2 * q] = Zc[0][nt][0];
                        lam[8 * nt + 2 * q + 1] = Zc[0][nt][1];
                    }
                }
#ifdef DTO_TDB_PROFILE
                long long tp2 = clock64();
#endif
                __syncthreads();
#ifdef DTO_TDB_PROFILE
                long long tp3 = clock64();
#endif
                // ---- phase 2: products ------------------------------------------------------------------
                if (warp == scal_warp && lane < 2) {  // scalars of the next node, into the other buffer
                    bool has_next = true;
                    double sn;
                    if (qq < nk) sn = (qq + 1 == nk) ? s0 + H : s0 + (qq + 1) * h;
                    else if (k + 1 < K) sn = s0;
                    else if (ms + 1 < steps) sn = s0 + H;
                    else { has_next = false; sn = 0.0; }
                    if (has_next) make_scal(I, zk, zk1, P.dt_off, lane == 0 ? sn : 1.0 - sn, scal[((e + 1) & 1) * 2 + lane],
                                            NV + (size_t)(((e + 1) & 1) * 2 + lane) * NVn);
                }
                // basis' lambda on the FMA pipe, one output per thread, taken from the top of the CTA.  It is a chain of
                // dependent FMAs fed from shared memory (latency-bound): the two warps of a scheduler run it at
                // opposite ends of the phase so that it hides behind the other warp's DMMAs.
                auto adjoint_basis_products = [&]() {
                    const int nh = nwarps > TF ? ((int)blockDim.x - TF * 32) : (int)blockDim.x;  // the warps without a forward tile, if any
                    if (nwarps > TF && warp < TF) return;
                    // two outputs per pass, four partial sums each: eight independent FMA chains of n / 4 links instead of one
                    // output at a time with two chains of n / 2 (the chains queue behind the other warps' DMMAs on the shared pipe)
                    for (int idx = (int)blockDim.x - 1 - (int)threadIdx.x; idx < nbasis * n; idx += 2 * nh) {
                        const int idx2 = idx + nh < nbasis * n ? idx + nh : idx;
                        const int s1 = idx % n, s2 = idx2 % n;
                        const double* M1 = basis_ptr(idx / n);
                        const double* M2 = basis_ptr(idx2 / n);
                        double a1[4] = {0.0, 0.0, 0.0, 0.0}, a2[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 4
                        for (int kk = 0; kk < n; kk += 4) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const double l = lam[kk + j];
                                a1[j] = fma(M1[sw<NT>(kk + j, s1)], l, a1[j]);
                                a2[j] = fma(M2[sw<NT>(kk + j, s2)], l, a2[j]);
                            }
                        }
                        PT[idx] = (a1[0] + a1[1]) + (a1[2] + a1[3]);
                        if (idx2 != idx) PT[idx2] = (a2[0] + a2[1]) + (a2[2] + a2[3]);
                    }
                };
                const bool matvec_first = (warp & 4) == 0;
                if (TA > 0 && matvec_first) adjoint_basis_products();
                if (couple) {
                    // basis products of the leading forward tile, one per warp, starting at the last (idle helper) warps
                    // one per forward warp (their own product is the only other work they have in this phase), the rest from the
                    // top.  The scheduler of forward warp 0 also carries the adjoint tile (warp TF): its basis product goes, in two
                    // output halves, to the next two warps instead (2.5 tile products per scheduler at most instead of 3).
                    const bool halves0 = TA > 0 && TF >= 2 && nwarps >= TF + 3 && NT >= 2;
                    for (int bi = 0; bi < nbasis; ++bi) {
                        int own_half = -1;  // -1: both output halves
                        if (bi == 0 && halves0) {
                            if (warp == TF + 1) own_half = 0;
                            else if (warp == TF + 2) own_half = 1;
                            else continue;
                        } else if ((bi < TF ? bi : nwarps - 1 - (bi - TF) % nwarps) != warp) {
                            continue;
                        }
                        const double* Mb = basis_ptr(bi);
                        double* out = Pb + (size_t)bi * 8 * TS + (size_t)row8 * TS + 2 * q;
#pragma unroll
                        for (int half = 0; half < 2; ++half) {
                            if (own_half >= 0 && half != own_half) continue;
                            constexpr int NH = (NT + 1) / 2;
                            double acc[NH][2];
#pragma unroll
                            for (int x = 0; x < NH; ++x) acc[x][0] = acc[x][1] = 0.0;
                            const int dsw = (NT % 2 == 0) ? ((row8 & 1) << 3) : 0;
                            const double* base = Mb + row8 * n + 2 * q;
#pragma unroll
                            for (int t = 0; t < NT; ++t) {
                                const double a0 = pub0[(t * 2) * 32 + lane], a1 = pub0[(t * 2 + 1) * 32 + lane];
                                const int off = 8 * t + ((t & 1) ? -dsw : dsw);
                                double2 bf[NH];
#pragma unroll
                                for (int x = 0; x < NH; ++x)
                                    if (half * NH + x < NT) bf[x] = *reinterpret_cast<const double2*>(base + 8 * (half * NH + x) * n + off);
#pragma unroll
                                for (int x = 0; x < NH; ++x)
                                    if (half * NH + x < NT) dmma(acc[x][0], acc[x][1], a0, bf[x].x);
#pragma unroll
                                for (int x = 0; x < NH; ++x)
                                    if (half * NH + x < NT) dmma(acc[x][0], acc[x][1], a1, bf[x].y);
                            }
#pragma unroll
                            for (int x = 0; x < NH; ++x) {
                                const int nt = half * NH + x;
                                if (nt < NT) {
                                    out[8 * nt] = acc[x][0];
                                    out[8 * nt + 1] = acc[x][1];
                                }
                            }
                        }
                    }
                }
                if (role != W_IDLE) {
                    if (qq == 0) {
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            Zp[0][nt][0] = Zc[0][nt][0];
                            Zp[0][nt][1] = Zc[0][nt][1];
                        }
                    }
                    const bool pubG = role == W_FWD && tile == 0 && couple;
                    const bool pubA = role == W_ADJ && row8 == 0;
                    double* tab = pubG ? PG + row8 * TS + 2 * q : PGa + 2 * q;
                    if (role == W_ADJ) mma_tile_axpy_T<NT>(Zp, Zc, Ga, hs * Sf.dt, lane, tab, pubA);
                    else mma_tile_axpy<NT>(Zp, Zc, Gf, hs * Sf.dt, lane, tab, pubG);
                }
                if (TA > 0 && !matvec_first) adjoint_basis_products();
#ifdef DTO_TDB_PROFILE
                long long tp4 = clock64();
#endif
                __syncthreads();
#ifdef DTO_TDB_PROFILE
                long long tp5 = clock64();
#endif
                prefetch_drift();  // Gf is free again: fetch the drift entries of the next node
                // ---- phase 3: parameter couplings, midpoint update ---------------------------------------
#ifdef DTO_TDB_PROFILE
                long long tc0 = clock64();
#endif
                {
                    if (role == W_FWD && couple) {
                        // The couplings of a forward tile are one small GEMM on the tensor pipe: Zp[8 rows][n] += W[8][K] T[K][n],
                        // T = the table rows (k = table t * nsrc + source row vs: G Z_vs, A_i Z_vs, B_i Z_vs, D_j Z_vs for the
                        // nsrc = 1 + np leading rows), W = this node's coefficients (CT) placed at the (row, source) pairs
                        // of the jet recurrence: first-order row a <- (x; dM/dtheta_a); pair row (a, b) <- (Z_b; M_a), (Z_a; M_b),
                        // (x; M_ab).  The accumulators are the state tile itself.
                        const int v = 8 * tile + row8;
                        const bool rowact = v >= 1 && v < nvecF;
                        if (packed) {
#pragma unroll
                            for (int ks = 0; ks < kPackedKS; ++ks) {
                                if (4 * ks < Kdim) {
                                    const int co = pk[ks] & kNoCoef;
                                    const double a = co != kNoCoef ? CT[co] : 0.0;
                                    const double* brow = PG + (pk[ks] >> 13) + row8;
#pragma unroll
                                    for (int nt = 0; nt < NT; ++nt) dmma(Zp[0][nt][0], Zp[0][nt][1], a, brow[8 * nt]);
                                }
                            }
                        } else
                        for (int k0 = 0; k0 < Kdim; k0 += 4) {
                            const int k = k0 + q;                       // A fragment: column k; B fragment: row k (same lane%4)
                            const int kc = k < Kdim ? k : Kdim - 1;
                            const int t = kc / nsrc, vs = kc - t * nsrc;
                            double a = 0.0;
                            if (rowact && k < Kdim) {
                                int slot = -1;
                                if (v <= np) slot = vs == 0 ? 0 : -1;
                                else if (vs == 1 + pair_b) slot = 0;
                                else if (vs == 1 + pair_a) slot = 1;    // only reached when a != b
                                else if (vs == 0) slot = 2;
                                if (slot >= 0) a = CT[((size_t)(v - 1) * 3 + slot) * KCr + t];
                            }
                            const double* brow = PG + (size_t)(t * 8 + vs) * TS + row8;  // PG and Pb are back to back: table t, row vs
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt) dmma(Zp[0][nt][0], Zp[0][nt][1], a, brow[8 * nt]);
                        }
                    } else if (role == W_ADJ) {
                        // d lambda^a = M' lambda^a + (M^a)' lambda: the same small GEMM with K = the tables (G' lambda, basis' lambda)
                        const bool rowact = row8 >= 1 && row8 <= np;
                        for (int k0 = 0; k0 < KCr; k0 += 4) {
                            const int k = k0 + q, kc = k < KCr ? k : KCr - 1;
                            const double a = rowact && k < KCr ? CT[((size_t)(nrowsF + row8 - 1) * 3) * KCr + k] : 0.0;
                            const double* brow = PGa + (size_t)kc * n + row8;  // PGa and PT are back to back
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt) dmma(Zp[0][nt][0], Zp[0][nt][1], a, brow[8 * nt]);
                        }
                    }
                }
#ifdef DTO_TDB_PROFILE
                if (lane == 0 && blockIdx.x == 0) g_tdb_prof[blockIdx.y][warp][7] += (unsigned long long)(Zp[0][0][0] != 12345.678 ? clock64() - tc0 : 0);
#endif
                if (role != W_IDLE) {
                    if (qq < nk) {  // Zp holds z_{q+1}: the tiles trade names
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                            for (int j = 0; j < 2; ++j) {
                                const double znew = Zp[0][nt][j];
                                Zp[0][nt][j] = Zc[0][nt][j];
                                Zc[0][nt][j] = znew;
                            }
                    } else {  // Gragg smoothing: 1/2 (z_n + z_{n-1} + h f(z_n)), weighted into the extrapolation
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                            for (int j = 0; j < 2; ++j) AccS[(nt * 2 + j) * 32 + lane] += wk[k] * 0.5 * (Zc[0][nt][j] + Zp[0][nt][j]);
                    }
                }
#ifdef DTO_TDB_PROFILE
                if (lane == 0 && blockIdx.x == 0) {
                    long long tp6 = clock64();
                    unsigned long long* pr = &g_tdb_prof[blockIdx.y][warp][0];
                    pr[0] += tp1 - tp0; pr[1] += tp2 - tp1; pr[2] += tp3 - tp2; pr[3] += tp4 - tp3; pr[4] += tp5 - tp4; pr[5] += tp6 - tp5; pr[6] += 1;
                }
#endif
            }
        }
        if (role != W_IDLE)
            for (int i = lane; i < FR; i += 32) Y0S[i] = AccS[i];
        __syncwarp();
    }

    // ---- outputs -----------------------------------------------------------------------------------------
    if (role != W_IDLE) {
    double F[NT][2];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
        F[nt][0] = Y0S[(nt * 2) * 32 + lane];
        F[nt][1] = Y0S[(nt * 2 + 1) * 32 + lane];
    }
    if (role == W_FWD) {
        const int v = 8 * tile + row8;
        if (g != nullptr && v == 0) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                g[mu_off + 8 * nt + 2 * q] = zk1[I.x_off + 8 * nt + 2 * q] - F[nt][0];
                g[mu_off + 8 * nt + 2 * q + 1] = zk1[I.x_off + 8 * nt + 2 * q + 1] - F[nt][1];
            }
        }
        if (want_jac) {
            double* jp = jac + (long long)b * P.nnz_jac_local;
            const long long own_off = jac_own_off(P, kl, I.doff, n);
            const long long prev_off = jac_prev_off(P, kl + 1, I.doff);
            if (v >= 1 && v <= np) {  // first-order rows are Jacobian columns
                const int a = v - 1;
                double* col;
                if (a < m) col = jp + jac_col(P, kl, I.u_off + a) + own_off;
                else if (a < nu) col = jp + jac_col(P, (kl + 1), I.u_off + (a - m)) + prev_off;
                else if (a == nu) col = jp + jac_col(P, kl, P.dt_off) + own_off;
                else col = jp + jac_col(P, kl, I.t_off) + own_off;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    col[8 * nt + 2 * q] = -F[nt][0];
                    col[8 * nt + 2 * q + 1] = -F[nt][1];
                }
            }
            if (tile == 0) {  // zero and identity columns
                for (int e2 = lane; e2 < 2 * z * n; e2 += 32) {
                    const int l = e2 / n, a = e2 % n;
                    if (l < z) {
                        if ((l >= I.x_off && l < I.x_off + n) || (l >= I.u_off && l < I.u_off + m) || l == P.dt_off || l == I.t_off) continue;
                        jp[jac_col(P, kl, l) + own_off + a] = 0.0;
                    } else {
                        const int lp = l - z;
                        if (I.order == 1 && lp >= I.u_off && lp < I.u_off + m) continue;
                        jp[jac_col(P, (kl + 1), lp) + prev_off + a] = (lp - I.x_off == a) ? 1.0 : 0.0;
                    }
                }
            }
        }
        if (want_hess) {
            // -mu' d2Phi x / (dtheta_a dtheta_b): every row reduces over its quad (uniform shuffles), pair rows store
            double s1 = 0.0;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt)
                s1 = fma(mu[mu_off + 8 * nt + 2 * q], F[nt][0], fma(mu[mu_off + 8 * nt + 2 * q + 1], F[nt][1], s1));
            s1 = quad_sum(s1);
            if (q == 0 && v > np && v < nvecF) {
                int p = v - 1 - np, a = 0;
                while (p >= np - a) {
                    p -= np - a;
                    ++a;
                }
                const int bb = a + p;
                double* hpp = I.hs + ((long long)b * P.nI + kl) * I.hs_stride + (long long)np * n;
                hpp[a * np + bb] = -s1;
                hpp[bb * np + a] = -s1;
            }
        }
    } else if (role == W_EXP) {
        double* jp = jac + (long long)b * P.nnz_jac_local;
        const long long own_off = jac_own_off(P, kl, I.doff, n);
        const int col = 8 * tile + row8;
        double* cp = jp + jac_col(P, kl, I.x_off + col) + own_off;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            cp[8 * nt + 2 * q] = -F[nt][0];
            cp[8 * nt + 2 * q + 1] = -F[nt][1];
        }
    } else {
        double* hx = I.hs + ((long long)b * P.nI + kl) * I.hs_stride;
        const int v = row8;
        if (v >= 1 && v <= np) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                hx[(size_t)(v - 1) * n + 8 * nt + 2 * q] = -F[nt][0];
                hx[(size_t)(v - 1) * n + 8 * nt + 2 * q + 1] = -F[nt][1];
            }
        }
    }
    }  // role != W_IDLE
    }  // items
}

// ------------------------------------------------------------------------------------------------------------------
// Propagator-only CTA (the second half of a split interval): the columns of the identity need no couplings, tables or
// adjoint generator, so G(tau) is double-buffered -- while the warps multiply their tiles by G(node q) they also
// assemble G(node q+1) into the other buffer (drift entries prefetched with cp.async one node earlier, node scalars
// computed two nodes ahead by one warp): ONE block barrier per right-hand side and assembly overlapped with DMMAs.
// ------------------------------------------------------------------------------------------------------------------
struct NodeIter {
    int ms, k, qq, steps, K;
    __device__ bool valid() const { return ms < steps; }
    __device__ double time() const {
        const double H = 1.0 / steps, s0 = ms * H;
        const int nk = 2 * (k + 1);
        return qq == nk ? s0 + H : s0 + qq * (H / nk);
    }
    __device__ void next() {
        if (qq < 2 * (k + 1)) ++qq;
        else {
            qq = 0;
            if (++k == K) {
                k = 0;
                ++ms;
            }
        }
    }
};

template <int NT>
__global__ void __launch_bounds__(8 * 32, 1)
    tdb_exp_kernel(DProb P, int ii, const double* __restrict__ Z, double* __restrict__ jac, int Kmax, int TE, int nbs,
                   double* __restrict__ scratch) {
    extern __shared__ __align__(16) double sm[];
    constexpr int n = 8 * NT, nn = n * n, FR = NT * 2 * 32;
    const DInt& I = P.in[ii];
    const int m = I.m, nc = I.n_carrier, z = P.z, nbasis = 2 * m + nc;
    const int nwarps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = lane & 3, row8 = lane >> 2;
    const bool active = warp < TE;
    const int tile = warp;
    double* G0b = sm;                                          // G of even nodes
    double* G1b = G0b + nn;                                    // G of odd nodes
    Scal* scal = reinterpret_cast<Scal*>(G1b + nn);            // [node parity]
    double* wk = reinterpret_cast<double*>(scal + 2);          // [kMaxCols] extrapolation weights
    double* Bs = wk + kMaxCols + (kMaxCols & 1);               // cached basis matrices
    double* AccS = scratch + ((size_t)(gridDim.x + blockIdx.x) * kMaxWarpsT + warp) * 2 * FR;  // second half of the scratch
    double* Y0S = AccS + FR;
    for (int i = threadIdx.x; i < nbs * nn; i += blockDim.x) Bs[i] = basis_global(I, i / nn, nn)[i % nn];
    auto prefetch_drift = [&](double* Gd) {
        for (int blk = (nn / 64) * warp / nwarps; blk < (nn / 64) * (warp + 1) / nwarps; ++blk) {
            const int p = sw<NT>((blk / NT) * 8 + (lane >> 2), (blk % NT) * 8 + 2 * (lane & 3));
            const unsigned dst = (unsigned)__cvta_generic_to_shared(Gd + p);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(I.Grm + p) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    const int eb0 = (nn / 64) * warp / nwarps, eb1 = (nn / 64) * (warp + 1) / nwarps;  // this warp's 8 x 8 blocks of G
    auto assemble = [&](double* Gd, const Scal& S) {
        asm volatile("cp.async.wait_all;" ::: "memory");
        if (nbs == nbasis && m <= 2 && nc == 0) assemble_generators<NT, true, 2, 0>(Gd, nullptr, Bs, I, S, S, m, nc, false, eb0, eb1, lane);
        else if (nbs == nbasis) assemble_generators<NT, true, kMaxM, kMaxC>(Gd, nullptr, Bs, I, S, S, m, nc, false, eb0, eb1, lane);
        else assemble_generators<NT, false, kMaxM, kMaxC>(Gd, nullptr, Bs, I, S, S, m, nc, false, eb0, eb1, lane);
    };

    const int nIc = min(P.kc1, P.nI) - P.kc0;
    const int n_items = nIc * P.batch;
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
        const int b = item / nIc, kl = P.kc0 + item % nIc;
        const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * z;
        const double* zk1 = zk + z;
        if (P.halo != nullptr && kl + 1 == P.nK - 1) zk1 = P.halo;
        const double dts = zk[P.dt_off];
        double poison;
        int K;
        const int steps = tdb_item_steps(I, zk, zk1, P.dt_off, poison, Kmax, K);  // the same counts as the forward/adjoint CTA of this interval
        __syncthreads();  // previous item done with both generators and the scalars
        if (threadIdx.x < kMaxCols) {
            const int k = threadIdx.x;
            double w = 1.0;
            const double nk2 = 4.0 * (k + 1) * (k + 1);
            for (int l = 0; l < K; ++l)
                if (l != k) w *= nk2 / (nk2 - 4.0 * (l + 1) * (l + 1));
            wk[k] = k < K ? w : 0.0;
        }
        if (active) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                for (int j = 0; j < 2; ++j) Y0S[(nt * 2 + j) * 32 + lane] = ((8 * tile + row8 == 8 * nt + 2 * q + j) ? 1.0 : 0.0) * poison;
        }
        // scalars of nodes 0 and 1, G(node 0), drift of node 1
        NodeIter ahead{0, 0, 0, steps, K};
        if (warp == nwarps - 1 && lane == 0) {
            NodeIter it = ahead;
            make_scal(I, zk, zk1, P.dt_off, it.time(), scal[0], nullptr);
            it.next();
            if (it.valid()) make_scal(I, zk, zk1, P.dt_off, it.time(), scal[1], nullptr);
        }
        ahead.next();
        ahead.next();  // the node whose scalars are computed during right-hand side 0
        prefetch_drift(G0b);
        __syncthreads();
        assemble(G0b, scal[0]);
        prefetch_drift(G1b);
        __syncthreads();

        double Zp[1][NT][2], Zc[1][NT][2], D[1][NT][2];
        int e = 0;
        for (int ms = 0; ms < steps; ++ms) {
            const double H = 1.0 / steps;
            if (active)
                for (int i = lane; i < FR; i += 32) AccS[i] = 0.0;
            for (int k = 0; k < K; ++k) {
                const int nk = 2 * (k + 1);
                const double h = H / nk;
                if (active) {
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        Zc[0][nt][0] = Y0S[(nt * 2) * 32 + lane];
                        Zc[0][nt][1] = Y0S[(nt * 2 + 1) * 32 + lane];
                    }
                }
                for (int qq = 0; qq <= nk; ++qq, ++e) {
                    double* Gcur = (e & 1) ? G1b : G0b;
                    double* Gnext = (e & 1) ? G0b : G1b;
                    const bool last = (ms == steps - 1 && k == K - 1 && qq == nk);
                    // the two warps of a scheduler take the two jobs in opposite order, so that one assembles
                    // (shared-memory loads, few FMAs) while the other keeps the FP64 pipe busy with its products
                    const bool asm_first = (warp & 4) != 0;
                    if (asm_first && !last) assemble(Gnext, scal[(e + 1) & 1]);
                    if (active) {
                        frag_zero(D);
                        mma_tile<NT>(D, Zc, Gcur, lane);
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            D[0][nt][0] *= dts;
                            D[0][nt][1] *= dts;
                        }
                        if (qq == 0) {
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                                for (int j = 0; j < 2; ++j) {
                                    Zp[0][nt][j] = Zc[0][nt][j];
                                    Zc[0][nt][j] = fma(h, D[0][nt][j], Zc[0][nt][j]);
                                }
                        } else if (qq < nk) {
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                                for (int j = 0; j < 2; ++j) {
                                    const double znew = fma(2.0 * h, D[0][nt][j], Zp[0][nt][j]);
                                    Zp[0][nt][j] = Zc[0][nt][j];
                                    Zc[0][nt][j] = znew;
                                }
                        } else {
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                                for (int j = 0; j < 2; ++j)
                                    AccS[(nt * 2 + j) * 32 + lane] += wk[k] * 0.5 * (Zc[0][nt][j] + Zp[0][nt][j] + h * D[0][nt][j]);
                        }
                    }
                    if (!asm_first && !last) assemble(Gnext, scal[(e + 1) & 1]);  // G of the next node, behind this node's products
                    if (warp == nwarps - 1 && lane == 0 && ahead.valid()) make_scal(I, zk, zk1, P.dt_off, ahead.time(), scal[e & 1], nullptr);
                    ahead.next();
                    __syncthreads();
                    if (!last) prefetch_drift(Gcur);  // free now: drift entries of the node after next
                }
            }
            if (active)
                for (int i = lane; i < FR; i += 32) Y0S[i] = AccS[i];
            __syncwarp();
        }
        if (active) {
            double* jp = jac + (long long)b * P.nnz_jac_local;
            const long long own_off = jac_own_off(P, kl, I.doff, n);
            double* cp = jp + jac_col(P, kl, I.x_off + 8 * tile + row8) + own_off;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                cp[8 * nt + 2 * q] = -Y0S[(nt * 2) * 32 + lane];
                cp[8 * nt + 2 * q + 1] = -Y0S[(nt * 2 + 1) * 32 + lane];
            }
        }
    }
}

struct Plan {
    int TF, TE, TA, split, warps, nbs;
    size_t smem;
};

bool make_plan(const DInt& I, bool want_jac, bool want_hess, bool allow_split, Plan& pl) {
    const int n = I.n, m = I.m, nc = I.n_carrier;
    if (n % 8 != 0 || n > 64 || (n / 8 == 5) || (n / 8 == 7) || m > kMaxM || nc > kMaxC || I.Asw == nullptr) return false;
    const int np = (I.order == 1 ? 2 * m : m) + 2, npairs = np * (np + 1) / 2;
    if (1 + np > 8) return false;  // the first-order rows (and the adjoint set) must fit one tile
    const int nvecF = want_hess ? 1 + np + npairs : (want_jac ? 1 + np : 1);
    pl.TF = (nvecF + 7) / 8;
    pl.TE = want_jac ? n / 8 : 0;
    pl.TA = want_hess ? 1 : 0;
    // one CTA per interval if its tiles fit 8 warps (255 registers each); else two CTAs per interval (forward +
    // adjoint tiles / propagator tiles) if each half fits 8 warps: both assemble the generators, neither spills;
    // else 16 warps at 128 registers
    pl.split = 0;
    pl.warps = pl.TF + pl.TE + pl.TA;
    if (pl.warps > 8) {
        const int half = std::max(pl.TF + pl.TA, pl.TE);
        // two kernels of 8-warp CTAs (forward + adjoint tiles / propagator tiles, 255 registers each); !allow_split = one
        // 16-warp CTA at 128 registers (measured slower: 11.1 against 9.2 ms at c3)
        if (half <= 8 && pl.TE > 0 && (allow_split || pl.warps > kMaxWarpsT)) {
            pl.split = 1;
            pl.warps = half;
        } else if (pl.warps > kMaxWarpsT) {
            pl.split = 1;
            pl.warps = half;
            if (pl.warps > kMaxWarpsT) return false;
        }
    }
    pl.warps = std::max(pl.warps, n >= 32 ? 8 : 4);  // idle warps still help assembling the generators (and take the basis mat-vecs)
    if (!pl.split && pl.warps > 8) pl.warps = kMaxWarpsT;  // the spare warps take the basis products and the assembly
    const size_t FR = (size_t)(n / 8) * 2 * 32, nbasis = 2 * m + nc;
    // coupling coefficient table + node values (2 buffers x forward/adjoint)
    const size_t ct = (((size_t)(nvecF > 1 ? nvecF - 1 : 0) + (want_hess ? np : 0)) * 3 * (1 + 2 * m + nc) + 1) / 2 * 2 +
                      4 * (((size_t)nv_count(m, nc) + 1) / 2 * 2);
    const size_t doubles = 2 * (size_t)n * n + 4 * sizeof(Scal) / sizeof(double) + FR + n + 8 * (n + 4) + nbasis * 8 * (n + 4) + n + nbasis * n + 12 + ct;
    const size_t budget = 227 * 1024 - 64;
    if (doubles * sizeof(double) > budget) return false;
    pl.nbs = (int)std::min<size_t>(nbasis, (budget - doubles * sizeof(double)) / ((size_t)n * n * sizeof(double)));
    pl.smem = (doubles + (size_t)pl.nbs * n * n) * sizeof(double);
    return I.tdb_scratch != nullptr;
}

template <int NT, int MAXW>
void launch_nt_w(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, cudaStream_t st,
                 const Plan& pl) {
    auto kern = tdb_dmma_kernel<NT, MAXW>;
    const DInt& I = P.in[ii];
    const int ctas = std::min((std::min(P.kc1, P.nI) - P.kc0) * P.batch, I.tdb_scratch_ctas / 2);  // persistent: one CTA per SM
    if (!pl.split) {
        kern<<<ctas, pl.warps * 32, pl.smem, st>>>(P, ii, Z, mu, f.want_g ? g : nullptr, jac, f.want_jac ? 1 : 0, f.want_hess ? 1 : 0, 8,
                                                   pl.TF, pl.TE, pl.TA, 0, pl.nbs, I.tdb_scratch);
        return;
    }
    // split interval: forward + adjoint tiles in one kernel, the propagator tiles in the double-buffered one
    kern<<<ctas, std::min(MAXW, std::max(pl.TF + pl.TA + 3, I.n >= 32 ? 8 : 4)) * 32, pl.smem, st>>>(P, ii, Z, mu, f.want_g ? g : nullptr, jac, f.want_jac ? 1 : 0,
                                                                    f.want_hess ? 1 : 0, 8, pl.TF, 0, pl.TA, 0, pl.nbs, I.tdb_scratch);
    const int n = I.n, nbasis = 2 * I.m + I.n_carrier;
    const size_t fixed = (2 * (size_t)n * n + 2 * sizeof(Scal) / sizeof(double) + 12) * sizeof(double);
    const int nbs = (int)std::min<size_t>(nbasis, (226 * 1024 - fixed) / ((size_t)n * n * sizeof(double)));
    tdb_exp_kernel<NT><<<ctas, std::max(pl.TE, 4) * 32, fixed + (size_t)nbs * n * n * sizeof(double), st>>>(P, ii, Z, jac, 8, pl.TE, nbs,
                                                                                                       I.tdb_scratch);
}

}  // namespace

// the plan of a Jacobian and Hessian pass: every other pass needs fewer tiles and no more shared memory
bool tdb_dmma_supported(const DInt& I) {
    Plan pl;
    return make_plan(I, true, true, true, pl);
}

bool tdb_dmma_configure(int n, std::string& err) {
    return with_nt(n, [&](auto nt) {
        constexpr int NT = decltype(nt)::value;
        const std::string s = std::to_string(NT);
        return opt_in_smem(tdb_dmma_kernel<NT, 8>, 227 * 1024, "tdb_dmma_kernel<" + s + ", 8>", err) &&
               opt_in_smem(tdb_dmma_kernel<NT, 16>, 227 * 1024, "tdb_dmma_kernel<" + s + ", 16>", err) &&
               opt_in_smem(tdb_exp_kernel<NT>, 227 * 1024, "tdb_exp_kernel<" + s + ">", err);
    });
}

void launch_tdb_dmma(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, bool split,
                     cudaStream_t st, long long* launches) {
    const DInt& I = P.in[ii];
    if (std::min(P.kc1, P.nI) - P.kc0 <= 0) return;
    Plan pl;
    make_plan(I, f.want_jac, f.want_hess, split, pl);  // succeeds where tdb_dmma_supported did
    with_nt(I.n, [&](auto nt) {
        if (pl.warps <= 8) launch_nt_w<decltype(nt)::value, 8>(P, ii, Z, mu, g, jac, f, st, pl);
        else launch_nt_w<decltype(nt)::value, 16>(P, ii, Z, mu, g, jac, f, st, pl);
    });
    ++*launches;
}

#ifdef DTO_TDB_PROFILE
extern "C" void dto_debug_tdb_profile(unsigned long long* out /* [2][16][8] */, int reset) {
    cudaDeviceSynchronize();
    cudaMemcpyFromSymbol(out, g_tdb_prof, sizeof(unsigned long long) * 2 * 16 * 8);
    if (reset) {
        unsigned long long z[2 * 16 * 8] = {0};
        cudaMemcpyToSymbol(g_tdb_prof, z, sizeof(z));
    }
}
#endif

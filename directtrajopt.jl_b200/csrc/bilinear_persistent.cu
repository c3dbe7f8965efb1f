// K1 (persistent DMMA variant): BilinearIntegrator interval kernel on the FP64 tensor pipe
// (mma.sync m8n8k4 -> SASS DMMA.8x8x4) for state dimensions 8..64 (multiples of 8), up to 4 drives and
// generators shared by the whole batch.
//
// One CTA per SM, up to 12 warps (3 per scheduler: the register file allows 168 registers/thread), alive
// for the whole launch.  The drift and drive matrices are staged in shared memory ONCE per CTA; every
// warp then pulls (role, interval) work items from three global counters until they run dry:
//   FWD  [x; dx/du_i; d2x/du_i du_j] rows through the scaled Taylor series of exp(dt G(u)): residual,
//        d/du, d/ddt Jacobian columns, identity/zero columns, (u,dt)x(u,dt) block of the compact Hessian
//   EXP  the propagator itself (-E Jacobian block).  Warps that own two spare matrices evaluate the Taylor
//        polynomial by Paterson-Stockmeyer in A^3 (2 + ceil(T/3) - 1 products instead of T), with
//        scaling and squaring above ||A||_1 = 1.5; otherwise columns of the identity go through the series
//   ADJ  [mu; dmu/du_i] through the transposed generator: (x,u), (x,dt) rows of the compact Hessian
// Big items first (FWD), small ones fill the tail, so the 148 SMs drain together.
//
// DFMA and DMMA share one datapath on B200 (tools/fp64_peak.cu: issuing both is no faster than either),
// so the design minimises FP64 issue slots of either kind, not just DMMAs.
//
// Operand layout: vectors are the ROWS of the A operand (Out[vec][s] = sum_k V[vec][k] * M[s][k]); the C
// fragment of one product (lane holds row lane/4, columns 2*(lane%4)+{0,1} of each 8-wide tile) is already
// the A fragment of the next product when k-step 2t contracts over the even and k-step 2t+1 over the odd
// states of tile t: the matching B fragments are one 16-byte LDS from the row-major matrix.  Matrices are
// stored unpadded; when n is a multiple of 16 the 8-double blocks of odd rows are swapped pairwise
// (XOR swizzle) so that the 8 rows x 64 bytes of one LDS.128 phase fall into distinct banks.
#include <stdlib.h>

#include "dto_internal.h"
#include "series_tables.cuh"
#include "bulk_copy.cuh"

namespace {

constexpr int kMaxDrives = 4;
constexpr int kMaxWarps = 12;

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

__device__ __forceinline__ double quad_sum(double v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// offset of element (row s, column k) of an n x n row-major matrix, n = 8*NT
template <int NT>
__device__ __forceinline__ int sw(int s, int k) {
    if constexpr (NT % 2 == 0) return s * (8 * NT) + (k ^ ((s & 1) << 3));
    else return s * (8 * NT) + k;
}

// out[mt][nt] += V[mt] * M'   (M row-major, swizzled): out[vec][s] += sum_k V[vec][k] M[s][k]
// MT = tiles used, MD = tiles the source array is declared with (MT <= MD)
template <int MT, int NT, int MD>
__device__ __forceinline__ void mma_apply(double (&out)[MT][NT][2], const double (&v)[MD][NT][2], const double* __restrict__ M,
                                          int lane) {
    constexpr int n = 8 * NT;
    const int row8 = lane >> 2;
    const int d = (NT % 2 == 0) ? ((row8 & 1) << 3) : 0;
    const double* base = M + row8 * n + 2 * (lane & 3);
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        const int off = 8 * t + ((t & 1) ? -d : d);  // 8 * (t ^ (row & 1)): rows 8*nt + row8 have the parity of row8
        double2 b[NT];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) b[nt] = *reinterpret_cast<const double2*>(base + 8 * nt * n + off);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) dmma(out[mt][nt][0], out[mt][nt][1], v[mt][t][0], b[nt].x);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) dmma(out[mt][nt][0], out[mt][nt][1], v[mt][t][1], b[nt].y);
    }
}

template <int MT, int NT>
__device__ __forceinline__ void frag_zero(double (&f)[MT][NT][2]) {
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) f[mt][nt][0] = f[mt][nt][1] = 0.0;
}

enum { ROLE_FWD = 0, ROLE_EXP = 1, ROLE_ADJ = 2 };

// Everything a work item needs, resolved once per warp.
template <int NT>
struct Ctx {
    const DProb* P;
    const DInt* I;
    const double* Z;
    const double* mu;
    double* g;
    double* jac;
    const double* Gs;  // (m+1) matrices in shared memory, drift first
    double* Gu;        // this warp's generator
    double* vbuf;      // (1 + kMaxDrives) * n doubles
    double* M3;        // EXP (Paterson-Stockmeyer) only
    double* S2;
    int lane, want_jac, want_hess;
    int jets;          // EvalFlags::jets
    const double2* plan;  // per-interval series plan (series_plan.cu) or nullptr
};

// G(u) = G_0 + sum_i u_i G_i in the shared layout; returns ||G(u)||_1 (identical arithmetic in every role)
template <int NT>
__device__ __forceinline__ double build_generator(const Ctx<NT>& c, const double (&uu)[kMaxDrives], int m, bool need_norm = true) {
    constexpr int n = 8 * NT, nn = n * n;
    for (int p = c.lane; p < nn; p += 32) {
        double v = c.Gs[p];
#pragma unroll
        for (int i = 0; i < kMaxDrives; ++i)
            if (i < m) v = fma(uu[i], c.Gs[(1 + i) * nn + p], v);
        c.Gu[p] = v;
    }
    __syncwarp();
    if (!need_norm) return 0.0;  // the series plan of this interval is already known (series_plan.cu)
    double cmax = 0.0;
    for (int k = c.lane; k < n; k += 32) {
        double s1 = 0.0;
        for (int s = 0; s < n; ++s) s1 += fabs(c.Gu[sw<NT>(s, k)]);
        cmax = fmax(cmax, s1);
    }
    return warp_max(cmax);
}

// series plan of interval (b, kk): from the pre-computed plan, else from ||dt G(u)||_1
template <int NT>
__device__ __forceinline__ Series interval_series(const Ctx<NT>& c, int b, int kk, double dt, const double (&uu)[kMaxDrives], int m) {
    if (c.plan != nullptr) {
        build_generator<NT>(c, uu, m, false);
        return choose_series(c.plan[(long long)b * c.P->nI + kk]);
    }
    return choose_series(fabs(dt) * build_generator<NT>(c, uu, m));
}

// y_i = G_i' a for every drive on the FP64 FMA pipe (one vector times m matrices would waste 7/8 of a DMMA tile).
// Lane s reads column s of G_i, i.e. consecutive elements of row k of the row-major matrix: conflict-free.
// For n < 32 the contraction index is split over the 32/n lane groups and reduced with shuffles, so that all
// lanes (not n of 32) carry FMAs.
template <int NT>
__device__ __forceinline__ void adjoint_drive_products(const double* __restrict__ Gs, const double* __restrict__ avec,
                                                       double* __restrict__ ybuf, int m, int lane) {
    constexpr int n = 8 * NT, nn = n * n;
    if constexpr (n >= 32) {
        for (int s = lane; s < n; s += 32) {
            double y[kMaxDrives] = {0.0, 0.0, 0.0, 0.0};
            for (int k = 0; k < n; k += 2) {
                const double2 a2 = *reinterpret_cast<const double2*>(avec + k);
                const int p0 = sw<NT>(k, s), p1 = sw<NT>(k + 1, s);
#pragma unroll
                for (int i = 0; i < kMaxDrives; ++i)
                    if (i < m) {
                        y[i] = fma(Gs[(1 + i) * nn + p0], a2.x, y[i]);
                        y[i] = fma(Gs[(1 + i) * nn + p1], a2.y, y[i]);
                    }
            }
#pragma unroll
            for (int i = 0; i < kMaxDrives; ++i)
                if (i < m) ybuf[i * n + s] = y[i];
        }
    } else {
        constexpr int KS = 32 / n;       // lane groups (n = 8: 4, n = 16: 2, n = 24: 1)
        constexpr int KL = n / KS;       // contraction indices per group
        const int s = lane % n, part = lane / n;
        double y[kMaxDrives] = {0.0, 0.0, 0.0, 0.0};
        if (part < KS) {
#pragma unroll
            for (int kk = 0; kk < KL; kk += 2) {
                const int k = part * KL + kk;
                const double2 a2 = *reinterpret_cast<const double2*>(avec + k);
                const int p0 = sw<NT>(k, s), p1 = sw<NT>(k + 1, s);
#pragma unroll
                for (int i = 0; i < kMaxDrives; ++i)
                    if (i < m) {
                        y[i] = fma(Gs[(1 + i) * nn + p0], a2.x, y[i]);
                        y[i] = fma(Gs[(1 + i) * nn + p1], a2.y, y[i]);
                    }
            }
        }
#pragma unroll
        for (int i = 0; i < kMaxDrives; ++i)
            if (i < m) {
#pragma unroll
                for (int off = n; off < 32 && off < n * KS; off <<= 1) y[i] += __shfl_xor_sync(0xffffffffu, y[i], off);
                if (lane < n) ybuf[i * n + s] = y[i];
            }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// FWD
// ------------------------------------------------------------------------------------------------------------------
template <int NT, int MT>
__device__ __forceinline__ void role_forward(const Ctx<NT>& c, int b, int kk, const int (&src)[kMaxDrives][MT],
                                             const double (&coef)[kMaxDrives][MT]) {
    constexpr int n = 8 * NT, nn = n * n;
    const DProb& P = *c.P;
    const DInt& I = *c.I;
    const int m = I.m, z = P.z, lane = c.lane, q = lane & 3, row8 = lane >> 2;
    const double* zk = c.Z + (long long)b * P.n_vars_local + (long long)kk * z;
    const double* zk1 = zk + z;
    if (P.halo != nullptr && kk + 1 == P.nK - 1) zk1 = P.halo;
    const double dt = zk[P.dt_off];
    double uu[kMaxDrives];
#pragma unroll
    for (int i = 0; i < kMaxDrives; ++i) uu[i] = i < m ? zk[I.u_off + i] : 0.0;
    const Series ser = interval_series<NT>(c, b, kk, dt, uu, m);
    const long long mu_off = (long long)b * P.n_cons_local + I.row_off + (long long)kk * n;
    const bool deriv = c.want_jac || c.want_hess || c.jets == DTO_JETS_STORE;
    const double* Gu = c.Gu;

    double F[MT][NT][2], term[MT][NT][2];
    frag_zero(F);
    if (row8 == 0) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            F[0][nt][0] = zk[I.x_off + 8 * nt + 2 * q];
            F[0][nt][1] = zk[I.x_off + 8 * nt + 2 * q + 1];
        }
    }
    for (int st = 0; st < ser.stages; ++st) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                term[mt][nt][0] = F[mt][nt][0];
                term[mt][nt][1] = F[mt][nt][1];
            }
        for (int t = 1; t <= ser.terms; ++t) {
            const double cf = dt * ser.inv_stages * kInv[t];
            double nw[MT][NT][2];
            frag_zero(nw);
            mma_apply<MT, NT, MT>(nw, term, Gu, lane);
#pragma unroll
            for (int i = 0; i < kMaxDrives; ++i) {
                if (i < m && deriv) {
                    double tmp[1][NT][2];
                    frag_zero(tmp);
                    mma_apply<1, NT, MT>(tmp, term, c.Gs + (1 + i) * nn, lane);
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            const double v0 = __shfl_sync(0xffffffffu, tmp[0][nt][0], src[i][mt]);
                            const double v1 = __shfl_sync(0xffffffffu, tmp[0][nt][1], src[i][mt]);
                            nw[mt][nt][0] = fma(coef[i][mt], v0, nw[mt][nt][0]);
                            nw[mt][nt][1] = fma(coef[i][mt], v1, nw[mt][nt][1]);
                        }
                }
            }
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    term[mt][nt][0] = cf * nw[mt][nt][0];
                    term[mt][nt][1] = cf * nw[mt][nt][1];
                    F[mt][nt][0] += term[mt][nt][0];
                    F[mt][nt][1] += term[mt][nt][1];
                }
        }
    }
    // ---- epilogue: GF = G(u) * rows of tile 0 (row 0: G F, rows 1+i: G dF/du_i) ----
    double GF[1][NT][2];
    frag_zero(GF);
    mma_apply<1, NT, MT>(GF, F, Gu, lane);
    if (c.g != nullptr && row8 == 0) {
        double* gp = c.g + mu_off;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            gp[8 * nt + 2 * q] = zk1[I.x_off + 8 * nt + 2 * q] - F[0][nt][0];
            gp[8 * nt + 2 * q + 1] = zk1[I.x_off + 8 * nt + 2 * q + 1] - F[0][nt][1];
        }
    }
    if (c.want_jac) {
        double* jp = c.jac + (long long)b * P.nnz_jac_local;
        const long long own_off = jac_own_off(P, kk, I.doff, n);
        const long long prev_off = jac_prev_off(P, kk + 1, I.doff);
        // zero and identity columns (everything except the x, u, dt columns of the own knot)
        for (int e = lane; e < 2 * z * n; e += 32) {
            const int l = e / n, a = e % n;
            if (l < z) {
                if ((l >= I.x_off && l < I.x_off + n) || (l >= I.u_off && l < I.u_off + m) || l == P.dt_off) continue;
                jp[jac_col(P, kk, l) + own_off + a] = 0.0;
            } else {
                jp[jac_col(P, (kk + 1), (l - z)) + prev_off + a] = (l - z - I.x_off == a) ? 1.0 : 0.0;
            }
        }
        // d/du_i columns from rows 1+i of tile 0, d/ddt column from row 0 of GF
        if (row8 >= 1 && row8 <= m) {
            double* col = jp + jac_col(P, kk, I.u_off + (row8 - 1)) + own_off;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                col[8 * nt + 2 * q] = -F[0][nt][0];
                col[8 * nt + 2 * q + 1] = -F[0][nt][1];
            }
        }
        if (row8 == 0) {
            double* col = jp + jac_col(P, kk, P.dt_off) + own_off;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                col[8 * nt + 2 * q] = -GF[0][nt][0];
                col[8 * nt + 2 * q + 1] = -GF[0][nt][1];
            }
        }
    }
    if (c.want_hess && c.jets == DTO_JETS_NONE) {
        // hpp[p][q] over parameters [u_1..u_m, dt]; hs = hx[np][n] | hpp[np][np]
        const int np = m + 1;
        double* hpp = I.hs + ((long long)b * P.nI + kk) * I.hs_stride + (long long)np * n;
        double muf[NT][2];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            muf[nt][0] = c.mu[mu_off + 8 * nt + 2 * q];
            muf[nt][1] = c.mu[mu_off + 8 * nt + 2 * q + 1];
        }
        // (u_i, u_j) = -mu' d2F/(du_i du_j): each second-order row reduces over its quad
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            double s1 = 0.0;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) s1 = fma(muf[nt][0], F[mt][nt][0], fma(muf[nt][1], F[mt][nt][1], s1));
            s1 = quad_sum(s1);
            const int r = mt * 8 + row8;
            if (q == 0 && r >= 1 + m && r < 1 + m + m * (m + 1) / 2) {
                int p = r - 1 - m, a = 0;
                while (p >= m - a) {
                    p -= m - a;
                    ++a;
                }
                const int bb = a + p;
                hpp[a * np + bb] = -s1;
                hpp[bb * np + a] = -s1;
            }
        }
        // (u_i, dt) = -mu' (G_i F + G dF/du_i);  (dt, dt) = -mu' G G F
        double dB = 0.0;  // mu' (G dF/du_i) in quad 1+i
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) dB = fma(muf[nt][0], GF[0][nt][0], fma(muf[nt][1], GF[0][nt][1], dB));
        dB = quad_sum(dB);
        double GGF[1][NT][2];
        frag_zero(GGF);
        mma_apply<1, NT, 1>(GGF, GF, Gu, lane);
        double dtt = 0.0;
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) dtt = fma(muf[nt][0], GGF[0][nt][0], fma(muf[nt][1], GGF[0][nt][1], dtt));
        dtt = quad_sum(dtt);
        if (lane == 0) hpp[m * np + m] = -dtt;
#pragma unroll
        for (int i = 0; i < kMaxDrives; ++i) {
            if (i < m) {
                double GiF[1][NT][2];
                frag_zero(GiF);
                mma_apply<1, NT, MT>(GiF, F, c.Gs + (1 + i) * nn, lane);
                double dA = 0.0;  // valid in quad 0
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) dA = fma(muf[nt][0], GiF[0][nt][0], fma(muf[nt][1], GiF[0][nt][1], dA));
                dA = quad_sum(dA);
                const double dBi = __shfl_sync(0xffffffffu, dB, 4 * (1 + i));
                if (lane == 0) {
                    hpp[i * np + m] = -(dA + dBi);
                    hpp[m * np + i] = -(dA + dBi);
                }
            }
        }
    }
    if (c.jets == DTO_JETS_STORE) {
        // the vectors the (parameter, parameter) entries are contractions of, for launch_hpp_contract (same order of
        // summation there: the two passes give the bits of the single pass)
        const int J2 = m * (m + 1) / 2;
        double* W = I.jets + ((long long)b * P.nI + kk) * I.jet_stride;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            const int r = mt * 8 + row8;
            if (r >= 1 + m && r < 1 + m + J2) {
                double* w = W + (long long)(r - 1 - m) * n;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    w[8 * nt + 2 * q] = F[mt][nt][0];
                    w[8 * nt + 2 * q + 1] = F[mt][nt][1];
                }
            }
        }
        double GGF[1][NT][2];
        frag_zero(GGF);
        mma_apply<1, NT, 1>(GGF, GF, Gu, lane);
        if (row8 == 0) {
            double* w = W + (long long)J2 * n;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                w[8 * nt + 2 * q] = GGF[0][nt][0];
                w[8 * nt + 2 * q + 1] = GGF[0][nt][1];
            }
        }
        if (row8 >= 1 && row8 <= m) {  // G dF/du_i sits in row 1+i of GF
            double* w = W + (long long)(J2 + 1 + m + (row8 - 1)) * n;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                w[8 * nt + 2 * q] = GF[0][nt][0];
                w[8 * nt + 2 * q + 1] = GF[0][nt][1];
            }
        }
#pragma unroll
        for (int i = 0; i < kMaxDrives; ++i) {
            if (i < m) {
                double GiF[1][NT][2];
                frag_zero(GiF);
                mma_apply<1, NT, MT>(GiF, F, c.Gs + (1 + i) * nn, lane);
                if (row8 == 0) {
                    double* w = W + (long long)(J2 + 1 + i) * n;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        w[8 * nt + 2 * q] = GiF[0][nt][0];
                        w[8 * nt + 2 * q + 1] = GiF[0][nt][1];
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// EXP, series mode: columns of the identity, MT tiles at a time, through the Taylor series
// ------------------------------------------------------------------------------------------------------------------
template <int NT, int MT>
__device__ __forceinline__ void role_exp_series(const Ctx<NT>& c, int b, int kk) {
    constexpr int n = 8 * NT;
    const DProb& P = *c.P;
    const DInt& I = *c.I;
    const int m = I.m, z = P.z, lane = c.lane, q = lane & 3, row8 = lane >> 2;
    const double* zk = c.Z + (long long)b * P.n_vars_local + (long long)kk * z;
    const double dt = zk[P.dt_off];
    double uu[kMaxDrives];
#pragma unroll
    for (int i = 0; i < kMaxDrives; ++i) uu[i] = i < m ? zk[I.u_off + i] : 0.0;
    const Series ser = interval_series<NT>(c, b, kk, dt, uu, m);
    double* jp = c.jac + (long long)b * P.nnz_jac_local;
    const long long own_off = jac_own_off(P, kk, I.doff, n);
    for (int c0 = 0; c0 < n; c0 += 8 * MT) {
        double F[MT][NT][2], term[MT][NT][2];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const int col = c0 + mt * 8 + row8;
                F[mt][nt][0] = (8 * nt + 2 * q == col) ? 1.0 : 0.0;
                F[mt][nt][1] = (8 * nt + 2 * q + 1 == col) ? 1.0 : 0.0;
            }
        for (int st = 0; st < ser.stages; ++st) {
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    term[mt][nt][0] = F[mt][nt][0];
                    term[mt][nt][1] = F[mt][nt][1];
                }
            for (int t = 1; t <= ser.terms - 2; ++t) {  // value series only
                const double cf = dt * ser.inv_stages * kInv[t];
                double nw[MT][NT][2];
                frag_zero(nw);
                mma_apply<MT, NT, MT>(nw, term, c.Gu, lane);
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        term[mt][nt][0] = cf * nw[mt][nt][0];
                        term[mt][nt][1] = cf * nw[mt][nt][1];
                        F[mt][nt][0] += term[mt][nt][0];
                        F[mt][nt][1] += term[mt][nt][1];
                    }
            }
        }
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            const int col = c0 + mt * 8 + row8;
            if (col < n) {
                double* cp = jp + jac_col(P, kk, I.x_off + col) + own_off;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    cp[8 * nt + 2 * q] = -F[mt][nt][0];
                    cp[8 * nt + 2 * q + 1] = -F[mt][nt][1];
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// EXP, Paterson-Stockmeyer mode.  A = dt G(u) / 2^s;  exp(A) ~ sum_{j<nb} B_j (A^3)^j + (A^3)^nb / (3nb)!,
// B_j = c_{3j} I + c_{3j+1} A + c_{3j+2} A^2, Horner in A^3 (nb - 1 products), then s squarings.
// Columns are processed ME tiles at a time: the lane holds its fragment of A, A^2 and the running
// polynomial for those columns in registers; A^3 (later the matrix being squared) sits row-major in M3 as
// the tensor-core operand and S2 keeps per-lane fragments (A^2, later the current power) between phases.
// ------------------------------------------------------------------------------------------------------------------
template <int NT>
__device__ __forceinline__ void role_exp_ps(const Ctx<NT>& c, int b, int kk) {
    constexpr int n = 8 * NT, nn = n * n;
    constexpr int ME = (NT == 2 || NT == 4) ? 2 : 1;  // column tiles per pass (register budget)
    constexpr int NCB = NT / ME;
    constexpr int SWZ = (NT % 2 == 0) ? 1 : 0;
    const DProb& P = *c.P;
    const DInt& I = *c.I;
    const int m = I.m, z = P.z, lane = c.lane, q = lane & 3, row8 = lane >> 2;
    const double* zk = c.Z + (long long)b * P.n_vars_local + (long long)kk * z;
    const double dt = zk[P.dt_off];
    double uu[kMaxDrives];
#pragma unroll
    for (int i = 0; i < kMaxDrives; ++i) uu[i] = i < m ? zk[I.u_off + i] : 0.0;
    double theta, alpha;
    if (c.plan != nullptr) {
        build_generator<NT>(c, uu, m, false);
        const double2 pl = c.plan[(long long)b * P.nI + kk];
        alpha = pl.x;
        theta = pl.y;
    } else {
        theta = alpha = fabs(dt) * build_generator<NT>(c, uu, m);
    }
    int sq = 0, nb = 1;
    double scale = dt;
    if (theta < 1e8) {
        double th = theta;
        while (th > 1.5) {
            th *= 0.5;
            alpha *= 0.5;
            scale *= 0.5;
            ++sq;
        }
        nb = (taylor_terms(fmin(th, alpha)) + 2) / 3;  // polynomial degree from alpha_2(A / 2^sq), squarings from ||A||_1
    } else {
        scale = __longlong_as_double(0x7ff8000000000000LL);  // not finite / absurd: NaN out, as choose_series
    }
    double* A = c.Gu;
    for (int p = lane; p < nn; p += 32) A[p] *= scale;
    __syncwarp();
    double* M3 = c.M3;
    double* S2 = c.S2;
    // element (row 8*nt + 2q + j, column 8*ct + row8) of a swizzled row-major matrix sits at
    // lane_rc + 8*(ct ^ j) + (8*nt + j)*n : one runtime base per (column tile, j), the rest is immediate
    const int lane_rc = 2 * q * n + row8;
    double* jp = c.jac + (long long)b * P.nnz_jac_local;
    const long long own_off = jac_own_off(P, kk, I.doff, n);

    // phase 1: A^2 (kept as fragments in S2) and A^3 (row-major in M3)
#pragma unroll 1
    for (int cb = 0; cb < NCB; ++cb) {
        int cbase[ME][2];
#pragma unroll
        for (int mt = 0; mt < ME; ++mt) {
            cbase[mt][0] = lane_rc + 8 * (cb * ME + mt);
            cbase[mt][1] = lane_rc + 8 * ((cb * ME + mt) ^ SWZ);
        }
        double* S2b = S2 + cb * (ME * NT * 2 * 32) + lane;
        double V[ME][NT][2], O[ME][NT][2];
#pragma unroll
        for (int mt = 0; mt < ME; ++mt)
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                V[mt][t][0] = A[cbase[mt][0] + (8 * t) * n];
                V[mt][t][1] = A[cbase[mt][1] + (8 * t + 1) * n];
            }
        frag_zero(O);
        mma_apply<ME, NT, ME>(O, V, A, lane);  // columns of A*A
#pragma unroll
        for (int mt = 0; mt < ME; ++mt)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                S2b[((mt * NT + nt) * 2 + 0) * 32] = O[mt][nt][0];
                S2b[((mt * NT + nt) * 2 + 1) * 32] = O[mt][nt][1];
            }
        frag_zero(V);
        mma_apply<ME, NT, ME>(V, O, A, lane);  // columns of A*A^2
#pragma unroll
        for (int mt = 0; mt < ME; ++mt)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                M3[cbase[mt][0] + (8 * nt) * n] = V[mt][nt][0];
                M3[cbase[mt][1] + (8 * nt + 1) * n] = V[mt][nt][1];
            }
    }
    __syncwarp();

    const double cd = kInvFact[3 * nb];
    // phase 2: Horner in A^3.  The lane's fragments of A and A^2 are re-read from shared memory for every B_j
    // (registers hold only the running polynomial and the accumulator)
#pragma unroll 1
    for (int cb = 0; cb < NCB; ++cb) {
        int cbase[ME][2];
#pragma unroll
        for (int mt = 0; mt < ME; ++mt) {
            cbase[mt][0] = lane_rc + 8 * (cb * ME + mt);
            cbase[mt][1] = lane_rc + 8 * ((cb * ME + mt) ^ SWZ);
        }
        double* S2b = S2 + cb * (ME * NT * 2 * 32) + lane;
        double Pm[ME][NT][2];
        {
            const double c0 = kInvFact[3 * (nb - 1)], c1 = kInvFact[3 * (nb - 1) + 1], c2 = kInvFact[3 * (nb - 1) + 2];
#pragma unroll
            for (int mt = 0; mt < ME; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const bool diag = (8 * nt + 2 * q + j) == 8 * (cb * ME + mt) + row8;
                        const double v1 = A[cbase[mt][j] + (8 * nt + j) * n];
                        const double v2 = S2b[((mt * NT + nt) * 2 + j) * 32];
                        const double v3 = M3[cbase[mt][j] + (8 * nt + j) * n];
                        Pm[mt][nt][j] = fma(cd, v3, fma(c2, v2, fma(c1, v1, diag ? c0 : 0.0)));
                    }
        }
#pragma unroll 1
        for (int j3 = nb - 2; j3 >= 0; --j3) {
            const double c0 = kInvFact[3 * j3], c1 = kInvFact[3 * j3 + 1], c2 = kInvFact[3 * j3 + 2];
            asm volatile("" ::: "memory");  // re-read the fragments: hoisting them out of the loop costs 4*ME*NT registers
            double O[ME][NT][2];
#pragma unroll
            for (int mt = 0; mt < ME; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const bool diag = (8 * nt + 2 * q + j) == 8 * (cb * ME + mt) + row8;
                        const double v1 = A[cbase[mt][j] + (8 * nt + j) * n];
                        const double v2 = S2b[((mt * NT + nt) * 2 + j) * 32];
                        O[mt][nt][j] = fma(c2, v2, fma(c1, v1, diag ? c0 : 0.0));
                    }
            mma_apply<ME, NT, ME>(O, Pm, M3, lane);  // O = B_j + A^3 * P
#pragma unroll
            for (int mt = 0; mt < ME; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    Pm[mt][nt][0] = O[mt][nt][0];
                    Pm[mt][nt][1] = O[mt][nt][1];
                }
        }
        if (sq == 0) {
#pragma unroll
            for (int mt = 0; mt < ME; ++mt) {
                const int col = 8 * (cb * ME + mt) + row8;
                double* cp = jp + jac_col(P, kk, I.x_off + col) + own_off;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    cp[8 * nt + 2 * q] = -Pm[mt][nt][0];
                    cp[8 * nt + 2 * q + 1] = -Pm[mt][nt][1];
                }
            }
        } else {
#pragma unroll
            for (int mt = 0; mt < ME; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    S2b[((mt * NT + nt) * 2 + 0) * 32] = Pm[mt][nt][0];
                    S2b[((mt * NT + nt) * 2 + 1) * 32] = Pm[mt][nt][1];
                }
        }
    }
    // squarings: M3 <- current matrix (row-major), every column block times M3
#pragma unroll 1
    for (int it = 0; it < sq; ++it) {
        __syncwarp();
#pragma unroll 1
        for (int cb = 0; cb < NCB; ++cb) {
            const double* S2b = S2 + cb * (ME * NT * 2 * 32) + lane;
#pragma unroll
            for (int mt = 0; mt < ME; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    M3[lane_rc + 8 * (cb * ME + mt) + (8 * nt) * n] = S2b[((mt * NT + nt) * 2 + 0) * 32];
                    M3[lane_rc + 8 * ((cb * ME + mt) ^ SWZ) + (8 * nt + 1) * n] = S2b[((mt * NT + nt) * 2 + 1) * 32];
                }
        }
        __syncwarp();
#pragma unroll 1
        for (int cb = 0; cb < NCB; ++cb) {
            double* S2b = S2 + cb * (ME * NT * 2 * 32) + lane;
            double V[ME][NT][2], O[ME][NT][2];
#pragma unroll
            for (int mt = 0; mt < ME; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    V[mt][nt][0] = S2b[((mt * NT + nt) * 2 + 0) * 32];
                    V[mt][nt][1] = S2b[((mt * NT + nt) * 2 + 1) * 32];
                }
            frag_zero(O);
            mma_apply<ME, NT, ME>(O, V, M3, lane);
            if (it == sq - 1) {
#pragma unroll
                for (int mt = 0; mt < ME; ++mt) {
                    const int col = 8 * (cb * ME + mt) + row8;
                    double* cp = jp + jac_col(P, kk, I.x_off + col) + own_off;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        cp[8 * nt + 2 * q] = -O[mt][nt][0];
                        cp[8 * nt + 2 * q + 1] = -O[mt][nt][1];
                    }
                }
            } else {
#pragma unroll
                for (int mt = 0; mt < ME; ++mt)
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        S2b[((mt * NT + nt) * 2 + 0) * 32] = O[mt][nt][0];
                        S2b[((mt * NT + nt) * 2 + 1) * 32] = O[mt][nt][1];
                    }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// ADJ: rows 0 -> mu, 1+i -> d/du_i, through G(u)' (Gu holds the transpose)
// ------------------------------------------------------------------------------------------------------------------
template <int NT>
__device__ __forceinline__ void role_adjoint(const Ctx<NT>& c, int b, int kk) {
    constexpr int n = 8 * NT, nn = n * n;
    const DProb& P = *c.P;
    const DInt& I = *c.I;
    const int m = I.m, z = P.z, lane = c.lane, q = lane & 3, row8 = lane >> 2;
    const double* zk = c.Z + (long long)b * P.n_vars_local + (long long)kk * z;
    const double dt = zk[P.dt_off];
    double uu[kMaxDrives];
#pragma unroll
    for (int i = 0; i < kMaxDrives; ++i) uu[i] = i < m ? zk[I.u_off + i] : 0.0;
    // ||G(u)||_1 with the arithmetic of build_generator (same series length as the forward role), then G(u)'
    Series ser;
    if (c.plan != nullptr) {
        ser = choose_series(c.plan[(long long)b * P.nI + kk]);
    } else {
        double cmax = 0.0;
        for (int k = lane; k < n; k += 32) {
            double s1 = 0.0;
            for (int s = 0; s < n; ++s) {
                const int p = sw<NT>(s, k);
                double v = c.Gs[p];
#pragma unroll
                for (int i = 0; i < kMaxDrives; ++i)
                    if (i < m) v = fma(uu[i], c.Gs[(1 + i) * nn + p], v);
                s1 += fabs(v);
            }
            cmax = fmax(cmax, s1);
        }
        ser = choose_series(fabs(dt) * warp_max(cmax));
    }
    for (int e = lane; e < nn; e += 32) {
        const int r = e / n, col = e % n;  // G(r, col) -> G'(col, r)
        const int p = sw<NT>(r, col);
        double v = c.Gs[p];
#pragma unroll
        for (int i = 0; i < kMaxDrives; ++i)
            if (i < m) v = fma(uu[i], c.Gs[(1 + i) * nn + p], v);
        c.Gu[sw<NT>(col, r)] = v;
    }
    __syncwarp();
    const long long mu_off = (long long)b * P.n_cons_local + I.row_off + (long long)kk * n;
    double* avec = c.vbuf;      // n
    double* ybuf = c.vbuf + n;  // m*n
    double F[1][NT][2], term[1][NT][2];
    frag_zero(F);
    if (row8 == 0) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            F[0][nt][0] = c.mu[mu_off + 8 * nt + 2 * q];
            F[0][nt][1] = c.mu[mu_off + 8 * nt + 2 * q + 1];
        }
    }
    for (int st = 0; st < ser.stages; ++st) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            term[0][nt][0] = F[0][nt][0];
            term[0][nt][1] = F[0][nt][1];
        }
        for (int t = 1; t <= ser.terms; ++t) {
            const double cf = dt * ser.inv_stages * kInv[t];
            // y_i = G_i' a on the FP64 pipe: lane s reads column s of G_i (row-major rows, conflict-free)
            if (row8 == 0) {
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    avec[8 * nt + 2 * q] = term[0][nt][0];
                    avec[8 * nt + 2 * q + 1] = term[0][nt][1];
                }
            }
            __syncwarp();
            adjoint_drive_products<NT>(c.Gs, avec, ybuf, m, lane);
            double nw[1][NT][2];
            frag_zero(nw);
            mma_apply<1, NT, 1>(nw, term, c.Gu, lane);
            __syncwarp();
            if (row8 >= 1 && row8 <= m) {
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    nw[0][nt][0] += ybuf[(row8 - 1) * n + 8 * nt + 2 * q];
                    nw[0][nt][1] += ybuf[(row8 - 1) * n + 8 * nt + 2 * q + 1];
                }
            }
            __syncwarp();
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                term[0][nt][0] = cf * nw[0][nt][0];
                term[0][nt][1] = cf * nw[0][nt][1];
                F[0][nt][0] += term[0][nt][0];
                F[0][nt][1] += term[0][nt][1];
            }
        }
    }
    double GY[1][NT][2];
    frag_zero(GY);
    mma_apply<1, NT, 1>(GY, F, c.Gu, lane);
    double* hx = I.hs + ((long long)b * P.nI + kk) * I.hs_stride;
    if (row8 >= 1 && row8 <= m) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            hx[(row8 - 1) * n + 8 * nt + 2 * q] = -F[0][nt][0];
            hx[(row8 - 1) * n + 8 * nt + 2 * q + 1] = -F[0][nt][1];
        }
    }
    if (row8 == 0) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            hx[m * n + 8 * nt + 2 * q] = -GY[0][nt][0];
            hx[m * n + 8 * nt + 2 * q + 1] = -GY[0][nt][1];
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// the persistent kernel
// ------------------------------------------------------------------------------------------------------------------
// warps per CTA the register file allows: 24 x 80 registers at n = 8, 16 x 128 at n = 16, 12 x 168 above
template <int NT>
constexpr int max_warps() {
    return NT == 1 ? 24 : (NT == 2 ? 16 : kMaxWarps);
}

template <int NT, int MT>
__global__ void __launch_bounds__(max_warps<NT>() * 32, 1)
    bilinear_persistent_kernel(DProb P, int ii, const double* __restrict__ Z, const double* __restrict__ mu, double* __restrict__ g,
                               double* __restrict__ jac, int want_jac, int want_hess, unsigned long long* __restrict__ wq, int nE,
                               int fetch, int jets) {
    extern __shared__ __align__(16) double sm[];
    constexpr int n = 8 * NT, nn = n * n;
    const DInt& I = P.in[ii];
    const int m = I.m;
    const int W = blockDim.x >> 5;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = lane & 3, row8 = lane >> 2;
    constexpr int slot = nn + (1 + kMaxDrives) * n;

    double* Gs = sm;
    if (I.Gsw != nullptr) {  // the swizzled copy made at construction, moved by the bulk-copy engine
        __shared__ __align__(8) unsigned long long bar;
        bulk_stage(Gs, I.Gsw, (unsigned)((m + 1) * nn * sizeof(double)), &bar);
    } else {
        for (int e = threadIdx.x; e < (m + 1) * nn; e += blockDim.x) {
            const int i = e / nn, r = e % nn;
            Gs[i * nn + sw<NT>(r / n, r % n)] = I.Grm[e];  // coalesced read, rows stay contiguous in shared memory
        }
        __syncthreads();
    }

    Ctx<NT> c;
    c.P = &P;
    c.I = &I;
    c.Z = Z;
    c.mu = mu;
    c.g = g;
    c.jac = jac;
    c.Gs = Gs;
    c.Gu = Gs + (size_t)(m + 1) * nn + (size_t)warp * slot;
    c.vbuf = c.Gu + nn;
    c.M3 = Gs + (size_t)(m + 1) * nn + (size_t)W * slot + (size_t)warp * 2 * nn;
    c.S2 = c.M3 + nn;
    c.lane = lane;
    c.want_jac = want_jac;
    c.want_hess = want_hess;
    c.jets = jets;
    c.plan = I.plan;
    const bool ps = warp < nE;  // this warp owns the two spare matrices of the Paterson-Stockmeyer propagator

    // forward rows: r = mt*8 + row8 : 0 -> x, 1+i -> d/du_i, 1+m+p -> d2/(du_i du_j); where the drive products go
    int src[kMaxDrives][MT];
    double coef[kMaxDrives][MT];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
        const int r = mt * 8 + row8;
        int pa = -1, pb = -1;
        if (r >= 1 + m) {
            int p = r - 1 - m, a = 0;
            while (a < m && p >= m - a) {
                p -= m - a;
                ++a;
            }
            if (a < m) {
                pa = a;
                pb = a + p;
            }
        }
#pragma unroll
        for (int i = 0; i < kMaxDrives; ++i) {
            int s_row = 0;
            double cc = 0.0;
            if (i < m) {
                if (r == 1 + i) { s_row = 0; cc = 1.0; }
                else if (pa == i && pb == i) { s_row = 1 + i; cc = 2.0; }
                else if (pa == i) { s_row = 1 + pb; cc = 1.0; }
                else if (pb == i) { s_row = 1 + pa; cc = 1.0; }
            }
            src[i][mt] = s_row * 4 + q;
            coef[i][mt] = cc;
        }
    }

    const int nIc = min(P.kc1, P.nI) - P.kc0;  // intervals of the active range
    const unsigned long long nItems = (unsigned long long)P.batch * (unsigned long long)nIc;
    // Paterson-Stockmeyer warps clear the propagators first and then join the others; when no warp has
    // spare matrices (nE == 0) the propagators run in series mode on every warp, after the forward items
    int order[3];
    int nroles = 0;
    if (ps && want_jac) order[nroles++] = ROLE_EXP;
    if (jets != DTO_JETS_USE) order[nroles++] = ROLE_FWD;
    if (nE == 0 && want_jac) order[nroles++] = ROLE_EXP;
    if (want_hess) order[nroles++] = ROLE_ADJ;
    for (int ri = 0; ri < nroles; ++ri) {
        const int role = order[ri];
        while (true) {
            unsigned long long id0 = 0;
            if (lane == 0) id0 = atomicAdd(&wq[role], (unsigned long long)fetch);  // `fetch` consecutive items per round trip
            id0 = __shfl_sync(0xffffffffu, id0, 0);
            if (id0 >= nItems) break;
            for (unsigned long long id = id0; id < id0 + fetch && id < nItems; ++id) {
            const int b = (int)(id / (unsigned long long)nIc), kk = P.kc0 + (int)(id % (unsigned long long)nIc);
            __syncwarp();
#ifndef DTO_SKIP_FWD
            if (role == ROLE_FWD) role_forward<NT, MT>(c, b, kk, src, coef);
#endif
#ifndef DTO_SKIP_ADJ
            if (role == ROLE_ADJ) role_adjoint<NT>(c, b, kk);
#endif
#ifndef DTO_SKIP_PS
            if (role == ROLE_EXP && ps) role_exp_ps<NT>(c, b, kk);
#endif
#ifndef DTO_SKIP_SER
            if (role == ROLE_EXP && !ps) role_exp_series<NT, (NT <= 2 ? 2 : 1)>(c, b, kk);
#endif
            __syncwarp();
            }
        }
    }
    // the CTA that leaves last zeroes the queue for the next launch (no memset node between the launches of a stream)
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&wq[3], 1ull) == (unsigned long long)gridDim.x - 1) {
            wq[0] = wq[1] = wq[2] = wq[3] = 0ull;
            __threadfence();
        }
    }
}

// ------------------------------------------------------------------------------------------------------------------
// Matrix-free Jacobian products (evaluator.jl:406-456 materialises all Jacobian values first; here the products come
// straight from the series).  J w: rows [x; w_x; d] with d the directional derivative of exp(dt G(u)) x along
// (w_u, w_dt): one extra tile product with G_w = sum_i w_ui G_i per term.  J' w: the adjoint rows of role ADJ with
// mu := w, contracted with x.  No propagator, no second-order rows.
// ------------------------------------------------------------------------------------------------------------------
template <int NT>
__device__ __forceinline__ void product_forward(const Ctx<NT>& c, double* Gw, const double* __restrict__ w, double* __restrict__ y, int b,
                                                int kk) {
    constexpr int n = 8 * NT, nn = n * n;
    const DProb& P = *c.P;
    const DInt& I = *c.I;
    const int m = I.m, z = P.z, lane = c.lane, q = lane & 3, row8 = lane >> 2;
    const double* zk = c.Z + (long long)b * P.n_vars_local + (long long)kk * z;
    const double* wk = w + (long long)b * P.n_vars_local + (long long)kk * z;
    const double dt = zk[P.dt_off], wdt = wk[P.dt_off];
    double uu[kMaxDrives], wu[kMaxDrives];
#pragma unroll
    for (int i = 0; i < kMaxDrives; ++i) {
        uu[i] = i < m ? zk[I.u_off + i] : 0.0;
        wu[i] = i < m ? wk[I.u_off + i] : 0.0;
    }
    const Series ser = choose_series(fabs(dt) * build_generator<NT>(c, uu, m));
    for (int p = lane; p < nn; p += 32) {
        double v = 0.0;
#pragma unroll
        for (int i = 0; i < kMaxDrives; ++i)
            if (i < m) v = fma(wu[i], c.Gs[(1 + i) * nn + p], v);
        Gw[p] = v;
    }
    __syncwarp();
    double F[1][NT][2], term[1][NT][2];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int s = 8 * nt + 2 * q + j;
            F[0][nt][j] = row8 == 0 ? zk[I.x_off + s] : (row8 == 1 ? wk[I.x_off + s] : 0.0);
        }
    for (int st = 0; st < ser.stages; ++st) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            term[0][nt][0] = F[0][nt][0];
            term[0][nt][1] = F[0][nt][1];
        }
        for (int t = 1; t <= ser.terms; ++t) {
            const double cf = dt * ser.inv_stages * kInv[t];
            double nw[1][NT][2], tmp[1][NT][2];
            frag_zero(nw);
            frag_zero(tmp);
            mma_apply<1, NT, 1>(nw, term, c.Gu, lane);
            mma_apply<1, NT, 1>(tmp, term, Gw, lane);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                const double v0 = __shfl_sync(0xffffffffu, tmp[0][nt][0], q);  // row 0 (x) feeds row 2 (d)
                const double v1 = __shfl_sync(0xffffffffu, tmp[0][nt][1], q);
                if (row8 == 2) {
                    nw[0][nt][0] += v0;
                    nw[0][nt][1] += v1;
                }
                term[0][nt][0] = cf * nw[0][nt][0];
                term[0][nt][1] = cf * nw[0][nt][1];
                F[0][nt][0] += term[0][nt][0];
                F[0][nt][1] += term[0][nt][1];
            }
        }
    }
    double GF[1][NT][2];
    frag_zero(GF);
    mma_apply<1, NT, 1>(GF, F, c.Gu, lane);  // row 0: G E x
    const double* wk1 = wk + z;
    double* yp = y + (long long)b * P.n_cons_local + I.row_off + (long long)kk * n;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const double f1 = __shfl_sync(0xffffffffu, F[0][nt][j], 4 + q);
            const double f2 = __shfl_sync(0xffffffffu, F[0][nt][j], 8 + q);
            if (row8 == 0) {
                const int s = 8 * nt + 2 * q + j;
                yp[s] = wk1[I.x_off + s] - (f1 + f2 + wdt * GF[0][nt][j]);
            }
        }
}

template <int NT>
__device__ __forceinline__ void product_adjoint(const Ctx<NT>& c, const double* __restrict__ w, double* __restrict__ y, int b, int kk) {
    constexpr int n = 8 * NT, nn = n * n;
    const DProb& P = *c.P;
    const DInt& I = *c.I;
    const int m = I.m, z = P.z, lane = c.lane, q = lane & 3, row8 = lane >> 2;
    const double* zk = c.Z + (long long)b * P.n_vars_local + (long long)kk * z;
    const double dt = zk[P.dt_off];
    double uu[kMaxDrives];
#pragma unroll
    for (int i = 0; i < kMaxDrives; ++i) uu[i] = i < m ? zk[I.u_off + i] : 0.0;
    double cmax = 0.0;
    for (int k = lane; k < n; k += 32) {
        double s1 = 0.0;
        for (int s = 0; s < n; ++s) {
            const int p = sw<NT>(s, k);
            double v = c.Gs[p];
#pragma unroll
            for (int i = 0; i < kMaxDrives; ++i)
                if (i < m) v = fma(uu[i], c.Gs[(1 + i) * nn + p], v);
            s1 += fabs(v);
        }
        cmax = fmax(cmax, s1);
    }
    const Series ser = choose_series(fabs(dt) * warp_max(cmax));
    for (int e = lane; e < nn; e += 32) {
        const int r = e / n, col = e % n;
        const int p = sw<NT>(r, col);
        double v = c.Gs[p];
#pragma unroll
        for (int i = 0; i < kMaxDrives; ++i)
            if (i < m) v = fma(uu[i], c.Gs[(1 + i) * nn + p], v);
        c.Gu[sw<NT>(col, r)] = v;
    }
    __syncwarp();
    const double* wr = w + (long long)b * P.n_cons_local + I.row_off + (long long)kk * n;
    double* avec = c.vbuf;
    double* ybuf = c.vbuf + n;
    double F[1][NT][2], term[1][NT][2];
    frag_zero(F);
    if (row8 == 0) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            F[0][nt][0] = wr[8 * nt + 2 * q];
            F[0][nt][1] = wr[8 * nt + 2 * q + 1];
        }
    }
    for (int st = 0; st < ser.stages; ++st) {
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            term[0][nt][0] = F[0][nt][0];
            term[0][nt][1] = F[0][nt][1];
        }
        for (int t = 1; t <= ser.terms; ++t) {
            const double cf = dt * ser.inv_stages * kInv[t];
            if (row8 == 0) {
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    avec[8 * nt + 2 * q] = term[0][nt][0];
                    avec[8 * nt + 2 * q + 1] = term[0][nt][1];
                }
            }
            __syncwarp();
            adjoint_drive_products<NT>(c.Gs, avec, ybuf, m, lane);
            double nw[1][NT][2];
            frag_zero(nw);
            mma_apply<1, NT, 1>(nw, term, c.Gu, lane);
            __syncwarp();
            if (row8 >= 1 && row8 <= m) {
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    nw[0][nt][0] += ybuf[(row8 - 1) * n + 8 * nt + 2 * q];
                    nw[0][nt][1] += ybuf[(row8 - 1) * n + 8 * nt + 2 * q + 1];
                }
            }
            __syncwarp();
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                term[0][nt][0] = cf * nw[0][nt][0];
                term[0][nt][1] = cf * nw[0][nt][1];
                F[0][nt][0] += term[0][nt][0];
                F[0][nt][1] += term[0][nt][1];
            }
        }
    }
    double GY[1][NT][2];
    frag_zero(GY);
    mma_apply<1, NT, 1>(GY, F, c.Gu, lane);  // row 0: G' E' w
    // x-columns of this knot: -E'w ; of the next knot: +w ; u_i: -x'(L_i' w) ; dt: -x'(G'E'w)
    double* yk = y + (long long)b * P.n_vars_local + (long long)kk * z;
    double dx = 0.0, dg = 0.0;  // x . F[row], x . GY[row 0]
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int s = 8 * nt + 2 * q + j;
            const double xs = zk[I.x_off + s];
            dx = fma(xs, F[0][nt][j], dx);
            dg = fma(xs, GY[0][nt][j], dg);
            if (row8 == 0) {
                atomicAdd(yk + I.x_off + s, -F[0][nt][j]);
                atomicAdd(yk + z + I.x_off + s, wr[s]);
            }
        }
    dx = quad_sum(dx);
    dg = quad_sum(dg);
    if (q == 0 && row8 >= 1 && row8 <= m) atomicAdd(yk + I.u_off + (row8 - 1), -dx);
    if (lane == 0) atomicAdd(yk + P.dt_off, -dg);
}

template <int NT>
__global__ void __launch_bounds__(max_warps<NT>() * 32, 1)
    bilinear_product_kernel(DProb P, int ii, const double* __restrict__ Z, const double* __restrict__ w, double* __restrict__ y,
                            int transpose, unsigned long long* __restrict__ wq, int fetch) {
    extern __shared__ __align__(16) double sm[];
    constexpr int n = 8 * NT, nn = n * n;
    const DInt& I = P.in[ii];
    const int m = I.m;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int slot = 2 * nn + (1 + kMaxDrives) * n;
    double* Gs = sm;
    for (int e = threadIdx.x; e < (m + 1) * nn; e += blockDim.x) {
        const int i = e / nn, r = e % nn;
        Gs[i * nn + sw<NT>(r / n, r % n)] = I.Grm[e];
    }
    __syncthreads();
    Ctx<NT> c;
    c.P = &P;
    c.I = &I;
    c.Z = Z;
    c.mu = nullptr;
    c.g = nullptr;
    c.jac = nullptr;
    c.Gs = Gs;
    c.Gu = Gs + (size_t)(m + 1) * nn + (size_t)warp * slot;
    double* Gw = c.Gu + nn;
    c.vbuf = Gw + nn;
    c.M3 = c.S2 = nullptr;
    c.lane = lane;
    c.want_jac = c.want_hess = 0;
    c.jets = DTO_JETS_NONE;
    c.plan = nullptr;  // the products are called on their own: no plan of this iterate
    const unsigned long long nItems = (unsigned long long)P.batch * (unsigned long long)P.nI;
    while (true) {
        unsigned long long id0 = 0;
        if (lane == 0) id0 = atomicAdd(&wq[0], (unsigned long long)fetch);
        id0 = __shfl_sync(0xffffffffu, id0, 0);
        if (id0 >= nItems) break;
        for (unsigned long long id = id0; id < id0 + fetch && id < nItems; ++id) {
            const int b = (int)(id / (unsigned long long)P.nI), kk = (int)(id % (unsigned long long)P.nI);
            __syncwarp();
            if (transpose) product_adjoint<NT>(c, w, y, b, kk);
            else product_forward<NT>(c, Gw, w, y, b, kk);
            __syncwarp();
        }
    }
}

constexpr size_t kSmemBudget = 227 * 1024 - 1024;  // dynamic shared memory the persistent kernel launches with at most

template <int NT>
void launch_product_nt(const DProb& P, int ii, const double* Z, const double* w, double* y, bool transpose, cudaStream_t st,
                       long long* launches) {
    const DInt& I = P.in[ii];
    constexpr int n = 8 * NT;
    const size_t mat = sizeof(double) * (size_t)n * n;
    const size_t slot = 2 * mat + sizeof(double) * (1 + kMaxDrives) * n;
    const size_t shared_part = (size_t)(I.m + 1) * mat;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int W = (int)std::min<size_t>(max_warps<NT>(), (kSmemBudget - shared_part) / slot);
    const size_t smem = shared_part + (size_t)W * slot;
    auto kern = bilinear_product_kernel<NT>;
    const long long items = (long long)P.batch * P.nI;
    const int grid = (int)std::max<long long>(1, std::min<long long>(sms, (items + W - 1) / W));
    const long long per_warp = items / ((long long)grid * W);
    const int fetch = (NT <= 2) ? (int)std::max<long long>(1, std::min<long long>(8, per_warp / 8)) : 1;
    kern<<<grid, W * 32, smem, st>>>(P, ii, Z, w, y, transpose ? 1 : 0, I.wq, fetch);
    cudaMemsetAsync(I.wq, 0, 4 * sizeof(unsigned long long), st);  // zero between launches
    ++*launches;
}

template <int NT, int MT>
void launch_variant(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, int ne_cap,
                    cudaStream_t st, long long* launches) {
    const DInt& I = P.in[ii];
    constexpr int n = 8 * NT;
    const size_t mat = sizeof(double) * (size_t)n * n;
    const size_t slot = mat + sizeof(double) * (1 + kMaxDrives) * n;
    const size_t shared_part = (size_t)(I.m + 1) * mat;  // with one slot at most 194.5 KB (n = 64, m = 4)
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // warps per CTA and how many of them carry the two spare matrices: prefer full occupancy, then
    // one Paterson-Stockmeyer warp per three
    int W = (int)std::min<size_t>(max_warps<NT>(), (kSmemBudget - shared_part) / slot);
    int nE = 0;
    if (f.want_jac) {
        int bestW = W, bestE = 0;
        for (int w = W; w >= std::max(2, W - 4); --w) {
            const size_t left = kSmemBudget - shared_part - (size_t)w * slot;
            const int e = (int)std::min<size_t>((size_t)w, left / (2 * mat));
            if (e >= (w + 2) / 3) {
                bestW = w;
                bestE = std::min(e, (w + 2) / 3);
                break;
            }
            if (e > bestE && w >= W - 2) {
                bestW = w;
                bestE = e;
            }
        }
        W = bestW;
        nE = std::min(bestE, ne_cap);
    }
    const size_t smem = shared_part + (size_t)W * slot + (size_t)nE * 2 * mat;
    auto kern = bilinear_persistent_kernel<NT, MT>;
    const long long items = (long long)P.batch * (std::min(P.kc1, P.nI) - P.kc0);
    const long long roles = (f.jets != DTO_JETS_USE ? 1 : 0) + (f.want_jac ? 1 : 0) + (f.want_hess ? 1 : 0);
    const long long want_ctas = (items * roles + W - 1) / W;
    const int grid = (int)std::max<long long>(1, std::min<long long>(std::max(1, sms - P.reserve_sms), want_ctas));
    // (the queue counters are zero between launches: the kernel's last CTA resets them)
    // small items (n <= 16) are fetched several at a time: the atomic's round trip is as long as the item itself
    const long long per_warp = items / ((long long)grid * W);
    const int fetch = (NT <= 2) ? (int)std::max<long long>(1, std::min<long long>(8, per_warp / 8)) : 1;
    kern<<<grid, W * 32, smem, st>>>(P, ii, Z, mu, f.want_g ? g : nullptr, jac, f.want_jac ? 1 : 0, f.want_hess ? 1 : 0, I.wq, nE, fetch, f.jets);
    ++*launches;
}

}  // namespace

bool bilinear_persistent_supported(int n, int m) {
    if (m < 0 || m > kMaxDrives) return false;
    return n == 8 || n == 16 || n == 24 || n == 32 || n == 48 || n == 64;
}

// the product kernel's m + 1 generators and one warp's slot: they exceed kSmemBudget at n = 64, m = 4
bool bilinear_product_supported(int n, int m) {
    const size_t mat = sizeof(double) * (size_t)n * n;
    return (size_t)(m + 1) * mat + 2 * mat + sizeof(double) * (1 + kMaxDrives) * n <= kSmemBudget;
}

bool bilinear_persistent_configure(int n, bool interval, bool product, std::string& err) {
    return with_nt(n, [&](auto nt) {
        constexpr int NT = decltype(nt)::value;
        const std::string s = std::to_string(NT);
        return (!interval || (opt_in_smem(bilinear_persistent_kernel<NT, 1>, kSmemBudget, "bilinear_persistent_kernel<" + s + ", 1>", err) &&
                              opt_in_smem(bilinear_persistent_kernel<NT, 2>, kSmemBudget, "bilinear_persistent_kernel<" + s + ", 2>", err))) &&
               (!product || opt_in_smem(bilinear_product_kernel<NT>, 227 * 1024, "bilinear_product_kernel<" + s + ">", err));
    });
}

void launch_bilinear_persistent(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f,
                                int ne_cap, cudaStream_t st, long long* launches) {
    const DInt& I = P.in[ii];
    if (std::min(P.kc1, P.nI) - P.kc0 <= 0) return;
    const bool second = (f.want_hess && f.jets == DTO_JETS_NONE) || f.jets == DTO_JETS_STORE;  // forward role carries d2/du du
    const int nrows = second ? 1 + I.m + I.m * (I.m + 1) / 2 : 1 + I.m;
    with_nt(I.n, [&](auto nt) {
        if (nrows > 8) launch_variant<decltype(nt)::value, 2>(P, ii, Z, mu, g, jac, f, ne_cap, st, launches);
        else launch_variant<decltype(nt)::value, 1>(P, ii, Z, mu, g, jac, f, ne_cap, st, launches);
    });
}

// y (+)= the rows / columns of integrator ii in J w (transpose = false: rows are assigned) or J' w (atomically added)
void launch_bilinear_product(const DProb& P, int ii, const double* Z, const double* w, double* y, bool transpose, cudaStream_t st,
                             long long* launches) {
    if (P.nI <= 0) return;
    with_nt(P.in[ii].n, [&](auto nt) { launch_product_nt<decltype(nt)::value>(P, ii, Z, w, y, transpose, st, launches); });
}

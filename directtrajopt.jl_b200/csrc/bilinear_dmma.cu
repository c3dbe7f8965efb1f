// K1 (DMMA variant): BilinearIntegrator interval kernel on the FP64 tensor cores (mma.sync m8n8k4 ->
// SASS DMMA.8x8x4) for state dimensions that are multiples of 8 (8..64) and up to 4 drives.
//
// One warp per (problem, interval); three roles per interval, selected by blockIdx.y so that one
// launch fills the 148 SMs with 3x the warps:
//   role FWD  propagates the rows [x; dx/du_i; d2x/du_i du_j] (<= 16 rows = 2 m-tiles) through the scaled
//             Taylor series of exp(dt*G(u)); writes the residual, the d/du and d/ddt Jacobian columns, the
//             identity / zero columns and the (u,dt)x(u,dt) block of the compact Hessian scratch
//   role EXP  propagates the columns of the identity, 16 at a time, and writes the -E Jacobian block
//   role ADJ  propagates [mu; dmu/du_i] through the transposed generator and writes the (x,u), (x,dt)
//             rows of the compact Hessian scratch
//
// Layout trick: vectors are the ROWS of the A operand (Out[vec][s] = sum_k V[vec][k] * M[s][k]), so the
// C fragment of one Taylor term (lane holds row lane/4, columns 2*(lane%4)+{0,1} of each 8-wide tile) is
// *already* the A fragment of the next term if k-step 2t contracts over the even and k-step 2t+1 over the
// odd states of tile t -- the matching B fragments are one 16-byte LDS (M row-major, k contiguous).
// The whole series therefore stays in registers; shared memory only feeds B fragments (conflict-free
// with the row stride chosen == 8 mod 16 doubles).
#include "dto_internal.h"

namespace {

constexpr int kMaxDrives = 4;

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

__host__ __device__ inline int dmma_ld(int n) { return (n % 16 == 8) ? n : n + 8; }

// out[mt][nt] += V[mt] * M'   (M row-major [s][k], leading dimension ld): out[vec][s] += sum_k V[vec][k] M[s][k]
// MT = tiles used, MD = tiles the source array is declared with (MT <= MD)
template <int MT, int NT, int MD>
__device__ __forceinline__ void mma_apply(double (&out)[MT][NT][2], const double (&v)[MD][NT][2], const double* __restrict__ M,
                                          int ld, int lane) {
    const double* base = M + (lane >> 2) * ld + 2 * (lane & 3);
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        double2 b[NT];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) b[nt] = *reinterpret_cast<const double2*>(base + 8 * nt * ld + 8 * t);
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

struct Series {
    int stages, terms;
    double poison;  // 1, or NaN for a generator norm that is not finite or absurd (>= 1e8): the interval's outputs become NaN
};

__device__ __forceinline__ Series choose_series(double theta) {
    Series s{1, 2, __longlong_as_double(0x7ff8000000000000LL)};
    if (theta < 1e8) {
        s.poison = 1.0;
        s.stages = theta > 4.0 ? (int)ceil(theta * 0.25) : 1;  // one stage up to ||dt G||_1 = 4 (e^4 round-off amplification)
        const double ths = theta / s.stages;
        double term = ths;
        int T = 1;
        while (term > 1.1102230246251565e-16 && T < 60) {  // 2^-53, as series_tables.cuh
            ++T;
            term *= ths / T;
        }
        s.terms = T + 2;
    }
    return s;
}

enum { ROLE_FWD = 0, ROLE_EXP = 1, ROLE_ADJ = 2 };

template <int NT, int MT>
__global__ void __launch_bounds__(128) bilinear_dmma_kernel(DProb P, int ii, const double* __restrict__ Z,
                                                              const double* __restrict__ mu, double* __restrict__ g,
                                                              double* __restrict__ jac, int want_jac, int want_hess, int W,
                                                              int ctas_per_problem) {
    extern __shared__ __align__(16) double sm[];
    constexpr int n = 8 * NT;
    const DInt& I = P.in[ii];
    const int m = I.m, z = P.z;
    const int ld = dmma_ld(n);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = lane & 3, row8 = lane >> 2;
    const int b = blockIdx.x / ctas_per_problem;
    const int kl = (blockIdx.x % ctas_per_problem) * W + warp;
    int role = blockIdx.y;
    if (role == 1 && !want_jac) role = ROLE_ADJ;
    const bool active = kl < P.nI;
    const double* Gg = I.G + (long long)b * I.G_stride;    // column-major matrices: Gg[i][k*n + s] = G_i(s,k)
    const double* Gr = I.Grm + (long long)b * I.G_stride;  // row-major copies:      Gr[i][s*n + k] = G_i(s,k)

    double* Gs = sm;                                  // m matrices, row-major G_i(s,k) at [s*ld + k]
    double* Gu = Gs + (size_t)m * n * ld + (size_t)warp * (n * ld + (1 + kMaxDrives) * n);  // per warp
    double* vbuf = Gu + n * ld;                       // per warp: n + kMaxDrives*n doubles of exchange space

    for (int e = threadIdx.x; e < m * n * n; e += blockDim.x) {
        const int i = e / (n * n), r = e % (n * n), s = r / n, k = r % n;
        Gs[(size_t)i * n * ld + s * ld + k] = Gr[(size_t)(1 + i) * n * n + r];  // coalesced read, conflict-free store
    }
    __syncthreads();
    if (!active) return;

    const int kk = kl;
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kk * z;
    const double* zk1 = zk + z;
    if (P.halo != nullptr && kk + 1 == P.nK - 1) zk1 = P.halo;
    const double dt = zk[P.dt_off];
    double uu[kMaxDrives];
#pragma unroll
    for (int i = 0; i < kMaxDrives; ++i) uu[i] = i < m ? zk[I.u_off + i] : 0.0;

    // per-warp generator G(u) (ADJ: its transpose), built from global (coalesced) into smem
    {
        // FWD/EXP want G(u) row-major, ADJ wants its transpose: read whichever global copy makes both the
        // global read coalesced and the shared store conflict-free
        const double* Gsrc = role == ROLE_ADJ ? Gg : Gr;
        for (int e = lane; e < n * n; e += 32) {
            double v = Gsrc[e];
#pragma unroll
            for (int i = 0; i < kMaxDrives; ++i)
                if (i < m) v = fma(uu[i], Gsrc[(size_t)(1 + i) * n * n + e], v);
            Gu[(e / n) * ld + (e % n)] = v;
        }
    }
    __syncwarp();
    // theta = |dt| * ||G(u)||_1 (max column abs sum), identical summation order in every role
    double cmax = 0.0;
    for (int k = lane; k < n; k += 32) {
        double s1 = 0.0;
        for (int s = 0; s < n; ++s) s1 += fabs(role == ROLE_ADJ ? Gu[k * ld + s] : Gu[s * ld + k]);
        cmax = fmax(cmax, s1);
    }
    const Series ser = choose_series(fabs(dt) * warp_max(cmax));

    const long long mu_off = (long long)b * P.n_cons_local + I.row_off + (long long)kk * n;

    if (role == ROLE_FWD) {
        // ---------------- forward rows: r = mt*8 + row8 : 0 -> x, 1+i -> d/du_i, 1+m+p -> d2/(du_i du_j) -------------
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
                double c = 0.0;
                if (i < m) {
                    if (r == 1 + i) { s_row = 0; c = 1.0; }
                    else if (pa == i && pb == i) { s_row = 1 + i; c = 2.0; }
                    else if (pa == i) { s_row = 1 + pb; c = 1.0; }
                    else if (pb == i) { s_row = 1 + pa; c = 1.0; }
                }
                src[i][mt] = s_row * 4 + q;
                coef[i][mt] = c;
            }
        }
        const bool deriv = want_jac || want_hess;
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
                const double c = ser.poison * dt / ((double)t * (double)ser.stages);
                double nw[MT][NT][2];
                frag_zero(nw);
                mma_apply<MT, NT, MT>(nw, term, Gu, ld, lane);
#pragma unroll
                for (int i = 0; i < kMaxDrives; ++i) {
                    if (i < m && deriv) {
                        double tmp[1][NT][2];
                        frag_zero(tmp);
                        mma_apply<1, NT, MT>(tmp, term, Gs + (size_t)i * n * ld, ld, lane);
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
                        term[mt][nt][0] = c * nw[mt][nt][0];
                        term[mt][nt][1] = c * nw[mt][nt][1];
                        F[mt][nt][0] += term[mt][nt][0];
                        F[mt][nt][1] += term[mt][nt][1];
                    }
            }
        }
        // ---- epilogue: GF = G(u) * rows of tile 0 (row 0: G F, rows 1+i: G dF/du_i) ----
        double GF[1][NT][2];
        frag_zero(GF);
        mma_apply<1, NT, MT>(GF, F, Gu, ld, lane);
        if (g != nullptr && row8 == 0) {
            double* gp = g + mu_off;
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                gp[8 * nt + 2 * q] = zk1[I.x_off + 8 * nt + 2 * q] - F[0][nt][0];
                gp[8 * nt + 2 * q + 1] = zk1[I.x_off + 8 * nt + 2 * q + 1] - F[0][nt][1];
            }
        }
        if (want_jac) {
            double* jp = jac + (long long)b * P.nnz_jac_local;
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
        if (want_hess) {
            // hpp[p][q] over parameters [u_1..u_m, dt]; hs = hx[np][n] | hpp[np][np]
            const int np = m + 1;
            double* hpp = I.hs + ((long long)b * P.nI + kk) * I.hs_stride + (long long)np * n;
            double muf[NT][2];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                muf[nt][0] = mu[mu_off + 8 * nt + 2 * q];
                muf[nt][1] = mu[mu_off + 8 * nt + 2 * q + 1];
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
            double dB = 0.0;  // mu' (G dF/du_i) in quad 1+i; mu' G F unused in quad 0
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) dB = fma(muf[nt][0], GF[0][nt][0], fma(muf[nt][1], GF[0][nt][1], dB));
            dB = quad_sum(dB);
            double GGF[1][NT][2];
            frag_zero(GGF);
            mma_apply<1, NT, 1>(GGF, GF, Gu, ld, lane);
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
                    mma_apply<1, NT, MT>(GiF, F, Gs + (size_t)i * n * ld, ld, lane);
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
    } else if (role == ROLE_EXP) {
        // ---------------- propagator columns, MT*8 at a time; V[c][s] = E(s,c) -----------------------------------------
        double* jp = jac + (long long)b * P.nnz_jac_local;
        const long long own_off = jac_own_off(P, kk, I.doff, n);
        for (int c0 = 0; c0 < n; c0 += 8 * MT) {
            double F[MT][NT][2], term[MT][NT][2];
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    const int c = c0 + mt * 8 + row8;
                    F[mt][nt][0] = (8 * nt + 2 * q == c) ? 1.0 : 0.0;
                    F[mt][nt][1] = (8 * nt + 2 * q + 1 == c) ? 1.0 : 0.0;
                }
            for (int st = 0; st < ser.stages; ++st) {
#pragma unroll
                for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        term[mt][nt][0] = F[mt][nt][0];
                        term[mt][nt][1] = F[mt][nt][1];
                    }
                for (int t = 1; t <= ser.terms - 2; ++t) {  // value series only: two terms fewer than the derivative rows
                    const double c = ser.poison * dt / ((double)t * (double)ser.stages);
                    double nw[MT][NT][2];
                    frag_zero(nw);
                    mma_apply<MT, NT, MT>(nw, term, Gu, ld, lane);
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            term[mt][nt][0] = c * nw[mt][nt][0];
                            term[mt][nt][1] = c * nw[mt][nt][1];
                            F[mt][nt][0] += term[mt][nt][0];
                            F[mt][nt][1] += term[mt][nt][1];
                        }
                }
            }
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                const int c = c0 + mt * 8 + row8;
                if (c < n) {
                    double* col = jp + jac_col(P, kk, I.x_off + c) + own_off;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        col[8 * nt + 2 * q] = -F[mt][nt][0];
                        col[8 * nt + 2 * q + 1] = -F[mt][nt][1];
                    }
                }
            }
        }
    } else {
        // ---------------- adjoint rows: 0 -> mu, 1+i -> d/du_i, through G(u)' (Gu holds the transpose) ------------------
        double* avec = vbuf;       // n
        double* ybuf = vbuf + n;   // m*n
        double F[1][NT][2], term[1][NT][2];
        frag_zero(F);
        if (row8 == 0) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                F[0][nt][0] = mu[mu_off + 8 * nt + 2 * q];
                F[0][nt][1] = mu[mu_off + 8 * nt + 2 * q + 1];
            }
        }
        for (int st = 0; st < ser.stages; ++st) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                term[0][nt][0] = F[0][nt][0];
                term[0][nt][1] = F[0][nt][1];
            }
            for (int t = 1; t <= ser.terms; ++t) {
                const double c = ser.poison * dt / ((double)t * (double)ser.stages);
                // y_i = G_i' a on the FP64 pipe: lane s reads column s of G_i (row-major, conflict-free)
                if (row8 == 0) {
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        avec[8 * nt + 2 * q] = term[0][nt][0];
                        avec[8 * nt + 2 * q + 1] = term[0][nt][1];
                    }
                }
                __syncwarp();
                for (int s = lane; s < n; s += 32) {
                    double y[kMaxDrives] = {0.0, 0.0, 0.0, 0.0};
                    for (int k = 0; k < n; k += 2) {
                        const double2 a2 = *reinterpret_cast<const double2*>(avec + k);
#pragma unroll
                        for (int i = 0; i < kMaxDrives; ++i)
                            if (i < m) {
                                y[i] = fma(Gs[(size_t)i * n * ld + k * ld + s], a2.x, y[i]);
                                y[i] = fma(Gs[(size_t)i * n * ld + (k + 1) * ld + s], a2.y, y[i]);
                            }
                    }
#pragma unroll
                    for (int i = 0; i < kMaxDrives; ++i)
                        if (i < m) ybuf[i * n + s] = y[i];
                }
                double nw[1][NT][2];
                frag_zero(nw);
                mma_apply<1, NT, 1>(nw, term, Gu, ld, lane);
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
                    term[0][nt][0] = c * nw[0][nt][0];
                    term[0][nt][1] = c * nw[0][nt][1];
                    F[0][nt][0] += term[0][nt][0];
                    F[0][nt][1] += term[0][nt][1];
                }
            }
        }
        double GY[1][NT][2];
        frag_zero(GY);
        mma_apply<1, NT, 1>(GY, F, Gu, ld, lane);
        const int np = m + 1;
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
        (void)np;
    }
}

template <int NT, int MT>
void launch_variant(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, cudaStream_t st,
                    long long* launches) {
    const DInt& I = P.in[ii];
    const int n = 8 * NT, ld = dmma_ld(n);
    const size_t per_warp = sizeof(double) * ((size_t)n * ld + (1 + kMaxDrives) * n);
    const size_t shared_part = sizeof(double) * (size_t)I.m * n * ld;
    int W = 4;
    while (W > 1 && shared_part + W * per_warp > 100 * 1024) W >>= 1;
    const size_t smem = shared_part + W * per_warp;  // at most 182.5 KB (n = 64, m = 4, W = 1)
    auto kern = bilinear_dmma_kernel<NT, MT>;
    const int cpp = (P.nI + W - 1) / W;
    dim3 grid((unsigned)(cpp * P.batch), 1 + (f.want_jac ? 1 : 0) + (f.want_hess ? 1 : 0));
    kern<<<grid, W * 32, smem, st>>>(P, ii, Z, mu, f.want_g ? g : nullptr, jac, f.want_jac ? 1 : 0, f.want_hess ? 1 : 0, W, cpp);
    ++*launches;
}

}  // namespace

bool bilinear_dmma_supported(int n, int m) {
    if (m < 0 || m > kMaxDrives) return false;
    return n == 8 || n == 16 || n == 24 || n == 32 || n == 48 || n == 64;
}

bool bilinear_dmma_configure(int n, std::string& err) {
    return with_nt(n, [&](auto nt) {
        constexpr int NT = decltype(nt)::value;
        return opt_in_smem(bilinear_dmma_kernel<NT, 1>, 227 * 1024, "bilinear_dmma_kernel<" + std::to_string(NT) + ", 1>", err) &&
               opt_in_smem(bilinear_dmma_kernel<NT, 2>, 227 * 1024, "bilinear_dmma_kernel<" + std::to_string(NT) + ", 2>", err);
    });
}

void launch_bilinear_dmma(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f,
                          cudaStream_t st, long long* launches) {
    const DInt& I = P.in[ii];
    if (P.nI <= 0) return;
    const int nrows = f.want_hess ? 1 + I.m + I.m * (I.m + 1) / 2 : 1 + I.m;
    // MT is the number of 8-row tiles of the forward role; the EXP role uses the same MT per chunk
    with_nt(I.n, [&](auto nt) {
        if (nrows > 8) launch_variant<decltype(nt)::value, 2>(P, ii, Z, mu, g, jac, f, st, launches);
        else launch_variant<decltype(nt)::value, 1>(P, ii, Z, mu, g, jac, f, st, launches);
    });
}

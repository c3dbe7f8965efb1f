// K1 (octet variant): BilinearIntegrator interval kernel for SMALL states (n = 8, 16) on the FP64 tensor pipe.
//
// At n = 8 a jet of one interval ([x; dx/du_i; d2x/du_i du_j] = 6 rows at m = 2) fills 6 of the 8 rows of a DMMA tile,
// its drive products 3 of 8, and the row-to-row couplings between them (G_i x feeds dx/du_i, ...) cost shuffles and
// shared-memory round trips: the persistent kernel spends ~27 other instructions per DMMA there and is issue- and
// latency-bound (profiles/r01_ncu_summary_c5.json).  This variant turns the tile around:
//
//   a warp owns EIGHT intervals; tile row r = interval r.  One tile per jet component (X, D_i, D_ij): every row of a
//   tile is the same component of a different interval.  The generators are shared by all intervals, so the B
//   operands are the constant matrices G_0, G_1, .., G_m and  G(u_r) V = G_0 V + sum_i u_{r,i} G_i V  is formed with the
//   row's own drives as lane-local FMAs (a lane holds row lane/4).  The products G_i X, G_i D_j that this needs are
//   exactly the coupling terms of the jet recurrence, and they land in the row they are added to:
//   no shuffles, no padding rows, no per-interval generator assembly, no shared-memory traffic besides the B fragments.
//
// Per term and octet at m = 2: 18 tile products (36 DMMA at n = 8) and ~60 lane-local FP64 instructions, against
// 48 DMMA + ~1300 other instructions for eight intervals of the persistent kernel.
//
// Roles: FWD (residual, d/du, d/ddt, identity/zero columns, (u,dt)x(u,dt) block of the compact Hessian) and
// ADJ ((x,u), (x,dt) rows of the compact Hessian) for all eight intervals; EXP (the -E block) per interval with the
// interval's own G(u) as B operand, assembled lane-locally from the same fragments.
// Every row keeps its own series plan (terms, stages): a row stops accumulating after its own number of terms, so
// the result of an interval does not depend on which other intervals share its octet (batches, knot ranges and shards
// stay bit-identical to the single-problem evaluation).
//
// Math as in bilinear_persistent.cu (SURVEY.md section 8a): jet recurrence of the scaled Taylor series of
// exp(dt G(u)) x, reference: src/integrators/bilinear_integrator.jl:81 differentiated by ForwardDiff (:111-161).
#include <math.h>
#include <stdlib.h>

#include "dto_internal.h"
#include "analytic_block.cuh"
#include "series_tables.cuh"

namespace {

__device__ __forceinline__ void dmma(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ double quad_sum(double v) {
    v += __shfl_xor_sync(0xffffffffu, v, 1);
    v += __shfl_xor_sync(0xffffffffu, v, 2);
    return v;
}
__device__ __forceinline__ double quad_max(double v) {
    v = fmax(v, __shfl_xor_sync(0xffffffffu, v, 1));
    v = fmax(v, __shfl_xor_sync(0xffffffffu, v, 2));
    return v;
}

// One tile: 8 rows (intervals) x n states; the lane holds row lane/4, states 8*nt + 2*(lane%4) + {0,1}.
template <int NT>
struct Tile {
    double v[NT][2];
};
template <int NT>
__device__ __forceinline__ void tzero(Tile<NT>& t) {
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) t.v[nt][0] = t.v[nt][1] = 0.0;
}

// B fragments of matrix `mat` in shared memory, fragment order: [(mat*NT + t)*NT + nt][lane] (double2): conflict-free
// LDS.128.  out[r][s] += sum_k V[r][k] M[s][k]
template <int NT>
__device__ __forceinline__ void tmma(Tile<NT>& out, const Tile<NT>& v, const double2* __restrict__ bf, int mat, int lane) {
#pragma unroll
    for (int t = 0; t < NT; ++t) {
        double2 b[NT];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) b[nt] = bf[((mat * NT + t) * NT + nt) * 32 + lane];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) dmma(out.v[nt][0], out.v[nt][1], v.v[t][0], b[nt].x);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) dmma(out.v[nt][0], out.v[nt][1], v.v[t][1], b[nt].y);
    }
}

// index of the second-order tile (a <= b)
template <int M>
__host__ __device__ constexpr int idx2(int a, int b) {
    return 1 + M + a * M - a * (a - 1) / 2 + (b - a);
}

// G(u_r) V = G_0 V + sum_i u_i (G_i V); the drive products are returned for the couplings
template <int NT, int M>
__device__ __forceinline__ void apply_all(Tile<NT>& gu, Tile<NT> (&pi)[M], const Tile<NT>& v, const double (&u)[M], const double2* bf,
                                          int mat0, int lane) {
    tzero(gu);
    tmma<NT>(gu, v, bf, mat0, lane);
#pragma unroll
    for (int i = 0; i < M; ++i) {
        tzero(pi[i]);
        tmma<NT>(pi[i], v, bf, mat0 + 1 + i, lane);
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) {
            gu.v[nt][0] = fma(u[i], pi[i].v[nt][0], gu.v[nt][0]);
            gu.v[nt][1] = fma(u[i], pi[i].v[nt][1], gu.v[nt][1]);
        }
    }
}
template <int NT, int M>
__device__ __forceinline__ void apply_gu(Tile<NT>& gu, const Tile<NT>& v, const double (&u)[M], const double2* bf, int mat0, int lane) {
    Tile<NT> pi[M];
    apply_all<NT, M>(gu, pi, v, u, bf, mat0, lane);
}

template <int NT>
__device__ __forceinline__ double tdot(const double (&muf)[NT][2], const Tile<NT>& t) {
    double s = 0.0;
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) s = fma(muf[nt][0], t.v[nt][0], fma(muf[nt][1], t.v[nt][1], s));
    return quad_sum(s);
}

// An n x n matrix in fragment form: r[mt] holds rows 8*mt .. 8*mt+7 (lane: row 8*mt + lane/4, columns 8*t + 2*(lane%4) + {0,1}).
// The C fragment of a tile is at the same time the B fragment of that tile's matrix: out = V * W' needs no data movement
// (out[i][s] = sum_k V[i][k] W[s][k]; for k-step (t, e) the B operand of lane (s', q) is W[8*nt + s'][8*t + 2q + e] = W.r[nt].v[t][e]).
template <int NT>
struct Mat {
    Tile<NT> r[NT];
};
template <int NT>
__device__ __forceinline__ void mul_t(Mat<NT>& out, const Mat<NT>& V, const Mat<NT>& W) {
#pragma unroll
    for (int mt = 0; mt < NT; ++mt) {
        tzero(out.r[mt]);
#pragma unroll
        for (int t = 0; t < NT; ++t) {
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) dmma(out.r[mt].v[nt][0], out.r[mt].v[nt][1], V.r[mt].v[t][0], W.r[nt].v[t][0]);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) dmma(out.r[mt].v[nt][0], out.r[mt].v[nt][1], V.r[mt].v[t][1], W.r[nt].v[t][1]);
        }
    }
}

// PP: every problem of the batch has its own generators (dto_integrator_desc::G_batch_stride != 0).  An octet then holds
// intervals of ONE problem (the last octet of a problem may be partial) and reads that problem's fragment-ordered
// generators straight from global memory (DInt::bfrag, 2 (M+1) NT^2 KB-sized blocks that stay in L1/L2) instead of the
// CTA's shared copy.
template <int NT, int M, bool PP>
__global__ void __launch_bounds__(NT == 1 ? 256 : 128, (NT == 1 && M <= 2) ? 2 : 1)  // n = 8, m <= 2: 128 registers, two CTAs of 8 warps per SM
    bilinear_octet_kernel(DProb P, int ii, const double* __restrict__ Z, const double* __restrict__ mu, double* __restrict__ g,
                          double* __restrict__ jac, int want_jac, int want_hess, int jets, long long n_whole) {
    constexpr int n = 8 * NT, nn = n * n, J = 1 + M + M * (M + 1) / 2;
    extern __shared__ __align__(16) double sm[];
    const DInt& I = P.in[ii];
    const int lane = threadIdx.x & 31, q = lane & 3, row8 = lane >> 2;
    const int z = P.z;

    // ---- stage once per CTA: the matrices row-major (for the 1-norms) and the B fragments of G_j and G_j' ----
    const double* Gs = sm;                                                  // (M+1) * nn
    const double2* bf = reinterpret_cast<const double2*>(sm + (M + 1) * nn);  // 2 (M+1) NT NT 32 double2: [G_0..G_M | G_0'..G_M']
    constexpr int kFrag = 2 * (M + 1) * NT * NT * 32;
    if constexpr (!PP) {
    double* Gw = sm;
    double2* bw = reinterpret_cast<double2*>(sm + (M + 1) * nn);
    for (int e = threadIdx.x; e < (M + 1) * nn; e += blockDim.x) Gw[e] = I.Grm[e];
    for (int e = threadIdx.x; e < kFrag; e += blockDim.x) {
        const int l = e & 31, f = e >> 5;
        const int nt = f % NT, t = (f / NT) % NT, mat = f / (NT * NT);
        const int s = 8 * nt + (l >> 2), k = 8 * t + 2 * (l & 3);
        double2 b;
        if (mat <= M) {  // M[s][k] = G[s][k]: row-major copy
            b.x = I.Grm[mat * nn + s * n + k];
            b.y = I.Grm[mat * nn + s * n + k + 1];
        } else {         // M[s][k] = G'[s][k] = G[k][s]: column-major copy, element (row k, col s) at s*n + k
            b.x = I.G[(mat - M - 1) * nn + s * n + k];
            b.y = I.G[(mat - M - 1) * nn + s * n + k + 1];
        }
        bw[e] = b;
    }
    __syncthreads();
    }

    const int nIc = min(P.kc1, P.nI) - P.kc0;  // intervals of the active range
    const long long nItems = (long long)P.batch * nIc;
    const long long opp = (nIc + 7) / 8;       // PP: octets per problem
    const long long nOct = PP ? opp * P.batch : (nItems + 7) / 8;
    // (problem, local interval) of row r of octet `oct`; false for the padding rows of a partial octet
    auto locate = [&](long long oct, int r, int& b, int& kk) -> bool {
        if constexpr (PP) {
            b = (int)(oct / opp);
            const long long id = (oct % opp) * 8 + r;
            kk = P.kc0 + (int)(id < nIc ? id : nIc - 1);
            return id < nIc;
        } else {
            const long long id = oct * 8 + r;
            const long long idc = id < nItems ? id : nItems - 1;
            b = (int)(idc / nIc);
            kk = P.kc0 + (int)(idc % nIc);
            return id < nItems;
        }
    };
    // CTA-major numbering: the warps of a CTA work on neighbouring octets (a CTA-minor numbering, which would spread a partial
    // last round over all SMs, costs 20 % at c5: the writes of one SM then scatter over the whole output)
    const long long warp0 = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long nWarps = (long long)gridDim.x * (blockDim.x >> 5);

    // Work units.  Normally one octet = one unit (forward, adjoint and propagator phases back to back in one warp).  When a
    // launch has only a few rounds of octets per warp (a knot-range shard on eight GPUs: 1.3 rounds), the duration of one
    // unit -- latency-bound, the same with two or eight warps on the SM -- quantises the kernel time; the octets from
    // `n_whole` on are therefore cut into their phases, each its own unit (longest first), a third of the granularity:
    // whole rounds of whole octets (the faster form), then the remainder in phases.
    int phases[3], nPh = 0;
    if (jets != DTO_JETS_USE) phases[nPh++] = 0;  // forward
    if (want_jac) phases[nPh++] = 1;              // propagator + constant columns (+ derivative integrators)
    if (want_hess) phases[nPh++] = 2;             // adjoint
    const long long nSplit = nOct - n_whole, nUnits = n_whole + nSplit * nPh;
    for (long long unit = warp0; unit < nUnits; unit += nWarps) {
        const bool whole = unit < n_whole;
        const long long oct = whole ? unit : n_whole + (unit - n_whole) % nSplit;
        const int ph = whole ? -1 : phases[(unit - n_whole) / nSplit];
        const bool do_fwd = ph < 0 || ph == 0, do_exp = ph < 0 || ph == 1, do_adj = ph < 0 || ph == 2;
        int b, kk;
        const bool valid = locate(oct, row8, b, kk);
        if constexpr (PP) {  // this problem's generators
            Gs = I.Grm + (long long)b * I.G_stride;
            bf = reinterpret_cast<const double2*>(I.bfrag) + (long long)b * kFrag;
        }
        const double* zk = Z + (long long)b * P.n_vars_local + (long long)kk * z;
        const double* zk1 = zk + z;
        if (P.halo != nullptr && kk + 1 == P.nK - 1) zk1 = P.halo;
        const double dt = zk[P.dt_off];
        double u[M];
#pragma unroll
        for (int i = 0; i < M; ++i) u[i] = zk[I.u_off + i];

        // ---- series plan of the row's interval from ||G(u_r)||_1: the lane sums its 2 NT columns over all rows, the quad
        // takes the maximum ----
        double cmax = 0.0;
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            double s0 = 0.0, s1 = 0.0;
            // m = 3: unrolled in full, the loads of this sum make the n = 8 knot-program form spill
#pragma unroll(M == 3 ? 4 : n)
            for (int s = 0; s < n; ++s) {
                const double2 g0 = *reinterpret_cast<const double2*>(Gs + s * n + 8 * t + 2 * q);
                double v0 = g0.x, v1 = g0.y;
#pragma unroll
                for (int i = 0; i < M; ++i) {
                    const double2 gi = *reinterpret_cast<const double2*>(Gs + (1 + i) * nn + s * n + 8 * t + 2 * q);
                    v0 = fma(u[i], gi.x, v0);
                    v1 = fma(u[i], gi.y, v1);
                }
                s0 += fabs(v0);
                s1 += fabs(v1);
            }
            cmax = fmax(cmax, fmax(s0, s1));
        }
        const Series ser = choose_series(fabs(dt) * quad_max(cmax));
        const int Tmax = __reduce_max_sync(0xffffffffu, ser.terms), Smax = __reduce_max_sync(0xffffffffu, ser.stages);
        const double cdt = dt * ser.inv_stages;
        const long long mu_off = (long long)b * P.n_cons_local + I.row_off + (long long)kk * n;
        double* jp = jac + (long long)b * P.nnz_jac_local;
        const long long own_off = jac_own_off(P, kk, I.doff, n);
        const bool store = jets == DTO_JETS_STORE;       // keep the second-order vectors for a later Hessian pass
        const bool second = store || (want_hess && jets == DTO_JETS_NONE);
        const bool deriv = want_jac || second;

        // =========================== FWD ===========================
        if (jets != DTO_JETS_USE && do_fwd) {
            Tile<NT> F[J], term[J];
#pragma unroll
            for (int j = 0; j < J; ++j) tzero(F[j]);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                F[0].v[nt][0] = zk[I.x_off + 8 * nt + 2 * q];  // knots are not 16-byte aligned (odd z)
                F[0].v[nt][1] = zk[I.x_off + 8 * nt + 2 * q + 1];
            }
            const int JJ = deriv ? (second ? J : 1 + M) : 1;  // tiles carried (uniform)
            for (int st = 0; st < Smax; ++st) {
                const bool act_s = st < ser.stages;
#pragma unroll
                for (int j = 0; j < J; ++j) term[j] = F[j];
                for (int t = 1; t <= Tmax; ++t) {
                    const double cf = cdt * kInv[t];
                    const bool acc = act_s && t <= ser.terms;
                    // products of the value and first-order tiles (old terms), cached for the couplings
                    Tile<NT> gu[1 + M], pi[1 + M][M];
                    apply_all<NT, M>(gu[0], pi[0], term[0], u, bf, 0, lane);
                    if (JJ > 1) {
#pragma unroll
                        for (int j = 1; j <= M; ++j) apply_all<NT, M>(gu[j], pi[j], term[j], u, bf, 0, lane);
                    }
                    if (JJ > 1 + M) {
                        // second-order tiles, in place: new = G(u) D_ab + G_a D_b + G_b D_a  (2 G_a D_a on the diagonal)
#pragma unroll
                        for (int a = 0; a < M; ++a)
#pragma unroll
                            for (int c = a; c < M; ++c) {
                                Tile<NT> w;
                                apply_gu<NT, M>(w, term[idx2<M>(a, c)], u, bf, 0, lane);
#pragma unroll
                                for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                                    for (int e = 0; e < 2; ++e) {
                                        const double cpl = (a == c) ? 2.0 * pi[1 + a][a].v[nt][e] : pi[1 + c][a].v[nt][e] + pi[1 + a][c].v[nt][e];
                                        const double tv = cf * (w.v[nt][e] + cpl);
                                        term[idx2<M>(a, c)].v[nt][e] = tv;
                                        if (acc) F[idx2<M>(a, c)].v[nt][e] += tv;
                                    }
                            }
                    }
                    if (JJ > 1) {
#pragma unroll
                        for (int i = 0; i < M; ++i)
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                                for (int e = 0; e < 2; ++e) {
                                    const double tv = cf * (gu[1 + i].v[nt][e] + pi[0][i].v[nt][e]);
                                    term[1 + i].v[nt][e] = tv;
                                    if (acc) F[1 + i].v[nt][e] += tv;
                                }
                    }
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const double tv = cf * gu[0].v[nt][e];
                            term[0].v[nt][e] = tv;
                            if (acc) F[0].v[nt][e] += tv;
                        }
                }
            }
            // ---- epilogue ----
            if (g != nullptr && valid) {
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    double* gp = g + mu_off + 8 * nt + 2 * q;
                    gp[0] = zk1[I.x_off + 8 * nt + 2 * q] - F[0].v[nt][0];
                    gp[1] = zk1[I.x_off + 8 * nt + 2 * q + 1] - F[0].v[nt][1];
                }
            }
            if (deriv) {
                Tile<NT> GF0, GiF0[M];
                apply_all<NT, M>(GF0, GiF0, F[0], u, bf, 0, lane);  // G(u) F and G_i F
                if (want_jac && valid) {
#pragma unroll
                    for (int i = 0; i < M; ++i) {
                        double* col = jp + jac_col(P, kk, I.u_off + i) + own_off;
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            col[8 * nt + 2 * q] = -F[1 + i].v[nt][0];
                            col[8 * nt + 2 * q + 1] = -F[1 + i].v[nt][1];
                        }
                    }
                    double* col = jp + jac_col(P, kk, P.dt_off) + own_off;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        col[8 * nt + 2 * q] = -GF0.v[nt][0];
                        col[8 * nt + 2 * q + 1] = -GF0.v[nt][1];
                    }
                }
                if (store && valid) {
                    // the vectors the (parameter, parameter) entries are contractions of (launch_hpp_contract)
                    constexpr int J2 = M * (M + 1) / 2;
                    double* W = I.jets + ((long long)b * P.nI + kk) * I.jet_stride;
                    auto put = [&](int slot, const Tile<NT>& t) {
                        double* w = W + (long long)slot * n;
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            w[8 * nt + 2 * q] = t.v[nt][0];
                            w[8 * nt + 2 * q + 1] = t.v[nt][1];
                        }
                    };
#pragma unroll
                    for (int a = 0; a < M; ++a)
#pragma unroll
                        for (int c = a; c < M; ++c) put(idx2<M>(a, c) - 1 - M, F[idx2<M>(a, c)]);
                }
                if (store) {
                    constexpr int J2 = M * (M + 1) / 2;
                    double* W = I.jets + ((long long)b * P.nI + kk) * I.jet_stride;
                    Tile<NT> GGF;
                    apply_gu<NT, M>(GGF, GF0, u, bf, 0, lane);
#pragma unroll
                    for (int i = 0; i < M; ++i) {
                        Tile<NT> GFi;
                        apply_gu<NT, M>(GFi, F[1 + i], u, bf, 0, lane);
                        if (valid) {
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt) {
                                W[(long long)(J2 + 1 + i) * n + 8 * nt + 2 * q] = GiF0[i].v[nt][0];
                                W[(long long)(J2 + 1 + i) * n + 8 * nt + 2 * q + 1] = GiF0[i].v[nt][1];
                                W[(long long)(J2 + 1 + M + i) * n + 8 * nt + 2 * q] = GFi.v[nt][0];
                                W[(long long)(J2 + 1 + M + i) * n + 8 * nt + 2 * q + 1] = GFi.v[nt][1];
                            }
                        }
                    }
                    if (valid) {
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            W[(long long)J2 * n + 8 * nt + 2 * q] = GGF.v[nt][0];
                            W[(long long)J2 * n + 8 * nt + 2 * q + 1] = GGF.v[nt][1];
                        }
                    }
                }
                if (want_hess && jets == DTO_JETS_NONE) {
                    // hpp[p][q] over parameters [u_1..u_M, dt]; hs = hx[np][n] | hpp[np][np]
                    constexpr int np = M + 1;
                    double* hpp = I.hs + ((long long)b * P.nI + kk) * I.hs_stride + (long long)np * n;
                    double muf[NT][2];
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        muf[nt][0] = mu[mu_off + 8 * nt + 2 * q];
                        muf[nt][1] = mu[mu_off + 8 * nt + 2 * q + 1];
                    }
                    const bool wr = valid && q == 0;
#pragma unroll
                    for (int a = 0; a < M; ++a)
#pragma unroll
                        for (int c = a; c < M; ++c) {
                            const double s1 = tdot<NT>(muf, F[idx2<M>(a, c)]);
                            if (wr) {
                                hpp[a * np + c] = -s1;
                                hpp[c * np + a] = -s1;
                            }
                        }
                    Tile<NT> GGF;
                    apply_gu<NT, M>(GGF, GF0, u, bf, 0, lane);
                    const double dtt = tdot<NT>(muf, GGF);
                    if (wr) hpp[M * np + M] = -dtt;
#pragma unroll
                    for (int i = 0; i < M; ++i) {
                        Tile<NT> GFi;
                        apply_gu<NT, M>(GFi, F[1 + i], u, bf, 0, lane);
                        const double dA = tdot<NT>(muf, GiF0[i]), dB = tdot<NT>(muf, GFi);
                        if (wr) {
                            hpp[i * np + M] = -(dA + dB);
                            hpp[M * np + i] = -(dA + dB);
                        }
                    }
                }
            }
        }

        // =========================== ADJ ===========================
        if (want_hess && do_adj) {
            Tile<NT> F[1 + M], term[1 + M];
#pragma unroll
            for (int j = 0; j <= M; ++j) tzero(F[j]);
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                F[0].v[nt][0] = mu[mu_off + 8 * nt + 2 * q];
                F[0].v[nt][1] = mu[mu_off + 8 * nt + 2 * q + 1];
            }
            for (int st = 0; st < Smax; ++st) {
                const bool act_s = st < ser.stages;
#pragma unroll
                for (int j = 0; j <= M; ++j) term[j] = F[j];
                for (int t = 1; t <= Tmax; ++t) {
                    const double cf = cdt * kInv[t];
                    const bool acc = act_s && t <= ser.terms;
                    Tile<NT> gu0, pi0[M];
                    apply_all<NT, M>(gu0, pi0, term[0], u, bf, M + 1, lane);  // G(u)' a and G_i' a
#pragma unroll
                    for (int i = 0; i < M; ++i) {
                        Tile<NT> w;
                        apply_gu<NT, M>(w, term[1 + i], u, bf, M + 1, lane);
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const double tv = cf * (w.v[nt][e] + pi0[i].v[nt][e]);
                                term[1 + i].v[nt][e] = tv;
                                if (acc) F[1 + i].v[nt][e] += tv;
                            }
                    }
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const double tv = cf * gu0.v[nt][e];
                            term[0].v[nt][e] = tv;
                            if (acc) F[0].v[nt][e] += tv;
                        }
                }
            }
            Tile<NT> GY;
            apply_gu<NT, M>(GY, F[0], u, bf, M + 1, lane);
            if (valid) {
                double* hx = I.hs + ((long long)b * P.nI + kk) * I.hs_stride;
#pragma unroll
                for (int i = 0; i < M; ++i)
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        hx[i * n + 8 * nt + 2 * q] = -F[1 + i].v[nt][0];
                        hx[i * n + 8 * nt + 2 * q + 1] = -F[1 + i].v[nt][1];
                    }
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    hx[M * n + 8 * nt + 2 * q] = -GY.v[nt][0];
                    hx[M * n + 8 * nt + 2 * q + 1] = -GY.v[nt][1];
                }
            }
        }

        // =========================== EXP: -E block, one interval at a time (rows = columns of E) ===========================
        // zero and identity columns (everything except the x, u, dt columns of the own knot), all eight intervals at once:
        // the four lanes of a row write the 8 NT rows of their interval's column
        if (want_jac && valid && do_exp) {
            const long long prev_off = jac_prev_off(P, kk + 1, I.doff);
            for (int l = 0; l < 2 * z; ++l) {
                if (l < z) {
                    if ((l >= I.x_off && l < I.x_off + n) || (l >= I.u_off && l < I.u_off + M) || l == P.dt_off) continue;
                    double* c = jp + jac_col(P, kk, l) + own_off;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) c[8 * nt + 2 * q] = c[8 * nt + 2 * q + 1] = 0.0;
                } else {
                    double* c = jp + jac_col(P, kk + 1, l - z) + prev_off;
                    const int dg = l - z - I.x_off;  // the row that holds the 1 of d x_{k+1} / d x_{k+1}
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        c[8 * nt + 2 * q] = (dg == 8 * nt + 2 * q) ? 1.0 : 0.0;
                        c[8 * nt + 2 * q + 1] = (dg == 8 * nt + 2 * q + 1) ? 1.0 : 0.0;
                    }
                }
            }
        }
        const bool fused = P.analytic_fused == ii + 1;  // this kernel also writes the derivative integrators' rows
        if (fused && !want_jac && g != nullptr && do_fwd) {
            for (int r = 0; r < 8; ++r) {
                int br, kr;
                if (locate(oct, r, br, kr)) analytic_interval(P, Z, g, nullptr, br, kr, lane, 32);
            }
        }
        if (want_jac && do_exp) {
            for (int r = 0; r < 8; ++r) {
                int br, kr;
                if (!locate(oct, r, br, kr)) break;
                if (fused) analytic_interval(P, Z, g, jac, br, kr, lane, 32);
                // the interval's own scalars, broadcast from the lanes of row r
                const double cdt_r = __shfl_sync(0xffffffffu, cdt, 4 * r);
                const int terms_r = __shfl_sync(0xffffffffu, ser.terms, 4 * r), stages_r = __shfl_sync(0xffffffffu, ser.stages, 4 * r);
                double ur[M];
#pragma unroll
                for (int i = 0; i < M; ++i) ur[i] = __shfl_sync(0xffffffffu, u[i], 4 * r);
                // B fragments of G(u_r), assembled lane-locally from the constant fragments
                double2 bu[NT][NT];
#pragma unroll
                for (int t = 0; t < NT; ++t)
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        double2 v = bf[((0 * NT + t) * NT + nt) * 32 + lane];
#pragma unroll
                        for (int i = 0; i < M; ++i) {
                            const double2 gi = bf[(((1 + i) * NT + t) * NT + nt) * 32 + lane];
                            v.x = fma(ur[i], gi.x, v.x);
                            v.y = fma(ur[i], gi.y, v.y);
                        }
                        bu[t][nt] = v;
                    }
                double* jr = jac + (long long)br * P.nnz_jac_local;
                const long long own_r = jac_own_off(P, kr, I.doff, n);
                if (stages_r == 1) {
                    // Paterson-Stockmeyer in A^3 on fragments.  Wanted: tile rows = columns of E, i.e. R = exp(B), B = A' (A = dt G(u_r)).
                    // With mul_t(V, W) = V W':  B^2 = mul_t(B, A),  A^2 = mul_t(A, B),  A^3 = mul_t(A^2, B),  R B^3 = mul_t(R, A^3).
                    // exp(B) ~ sum_{j < nb} (c_3j I + c_3j+1 B + c_3j+2 B^2) (B^3)^j: 3 + (nb - 1) products instead of `terms` tile sweeps.
                    Mat<NT> A, B;
#pragma unroll
                    for (int mt = 0; mt < NT; ++mt)
#pragma unroll
                        for (int t = 0; t < NT; ++t) {
                            double2 v = bf[(((M + 1) * NT + t) * NT + mt) * 32 + lane];  // G_0'
#pragma unroll
                            for (int i = 0; i < M; ++i) {
                                const double2 gi = bf[(((M + 2 + i) * NT + t) * NT + mt) * 32 + lane];
                                v.x = fma(ur[i], gi.x, v.x);
                                v.y = fma(ur[i], gi.y, v.y);
                            }
                            B.r[mt].v[t][0] = cdt_r * v.x;
                            B.r[mt].v[t][1] = cdt_r * v.y;
                            A.r[mt].v[t][0] = cdt_r * bu[t][mt].x;
                            A.r[mt].v[t][1] = cdt_r * bu[t][mt].y;
                        }
                    Mat<NT> B2, A3, R;
                    mul_t<NT>(B2, B, A);
                    {
                        Mat<NT> A2;
                        mul_t<NT>(A2, A, B);
                        mul_t<NT>(A3, A2, B);
                    }
                    const int nb = (terms_r - 2 + 3) / 3;  // degree 3 nb - 1 >= terms - 2 (value series only)
#pragma unroll 1
                    for (int j3 = nb - 1; j3 >= 0; --j3) {
                        const double c0 = kInvFact[3 * j3], c1 = kInvFact[3 * j3 + 1], c2 = kInvFact[3 * j3 + 2];
                        Mat<NT> Rn;
                        if (j3 == nb - 1) {
#pragma unroll
                            for (int mt = 0; mt < NT; ++mt) tzero(Rn.r[mt]);
                        } else {
                            mul_t<NT>(Rn, R, A3);
                        }
#pragma unroll
                        for (int mt = 0; mt < NT; ++mt)
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                                for (int e = 0; e < 2; ++e) {
                                    const bool diag = (8 * nt + 2 * q + e) == (8 * mt + row8);
                                    R.r[mt].v[nt][e] = Rn.r[mt].v[nt][e] + fma(c2, B2.r[mt].v[nt][e], fma(c1, B.r[mt].v[nt][e], diag ? c0 : 0.0));
                                }
                    }
#pragma unroll
                    for (int mt = 0; mt < NT; ++mt) {
                        double* cp = jr + jac_col(P, kr, I.x_off + 8 * mt + row8) + own_r;
#pragma unroll
                        for (int nt = 0; nt < NT; ++nt) {
                            cp[8 * nt + 2 * q] = -R.r[mt].v[nt][0];
                            cp[8 * nt + 2 * q + 1] = -R.r[mt].v[nt][1];
                        }
                    }
                } else {
#pragma unroll 1
                for (int mt = 0; mt < NT; ++mt) {  // several stages: 8 columns of E at a time through the series
                    Tile<NT> F, term;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        F.v[nt][0] = (8 * nt + 2 * q == 8 * mt + row8) ? 1.0 : 0.0;
                        F.v[nt][1] = (8 * nt + 2 * q + 1 == 8 * mt + row8) ? 1.0 : 0.0;
                    }
                    for (int st = 0; st < stages_r; ++st) {
                        term = F;
                        for (int t = 1; t <= terms_r - 2; ++t) {  // value series only
                            const double cf = cdt_r * kInv[t];
                            Tile<NT> w;
                            tzero(w);
#pragma unroll
                            for (int tt = 0; tt < NT; ++tt) {
#pragma unroll
                                for (int nt = 0; nt < NT; ++nt) dmma(w.v[nt][0], w.v[nt][1], term.v[tt][0], bu[tt][nt].x);
#pragma unroll
                                for (int nt = 0; nt < NT; ++nt) dmma(w.v[nt][0], w.v[nt][1], term.v[tt][1], bu[tt][nt].y);
                            }
#pragma unroll
                            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                                for (int e = 0; e < 2; ++e) {
                                    term.v[nt][e] = cf * w.v[nt][e];
                                    F.v[nt][e] += term.v[nt][e];
                                }
                        }
                    }
                    double* cp = jr + jac_col(P, kr, I.x_off + 8 * mt + row8) + own_r;
#pragma unroll
                    for (int nt = 0; nt < NT; ++nt) {
                        cp[8 * nt + 2 * q] = -F.v[nt][0];
                        cp[8 * nt + 2 * q + 1] = -F.v[nt][1];
                    }
                }
                }
            }
        }
    }
}

template <int NT, int M, bool PP>
bool launch_octet_pp(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, cudaStream_t st,
                     long long* launches) {
    constexpr int n = 8 * NT;
    const size_t smem = PP ? 0 : sizeof(double) * (size_t)(M + 1) * n * n + sizeof(double2) * (size_t)2 * (M + 1) * NT * NT * 32;
    auto kern = bilinear_octet_kernel<NT, M, PP>;
    static PerDeviceOnce configured;
    if (smem > 48 * 1024 && configured.first()) {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return false;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int threads = NT == 1 ? 256 : 128;
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
    const long long nIc = std::min(P.kc1, P.nI) - P.kc0, items = (long long)P.batch * nIc;
    const long long octs = PP ? (long long)P.batch * ((nIc + 7) / 8) : (items + 7) / 8, wpc = threads / 32;
    const int nPh = (f.jets != DTO_JETS_USE ? 1 : 0) + (f.want_jac ? 1 : 0) + (f.want_hess ? 1 : 0);
    const long long resident = (long long)std::max(1, sms - P.reserve_sms) * per_sm * wpc;  // warps in flight
    const char* env = getenv("DTO_B200_OCTET_SPLIT");           // A/B switch: 0 = whole octets only, 1 = every octet in phases
    // Three forms: whole octets only; every octet in phases (a third of the granularity, but ~8 % (n = 16) / ~20 % (n = 8)
    // slower per octet); whole rounds of whole octets and the remainder in phases.  Measured (tools/c4_size_sweep.py,
    // tools/c5_batch_sweep.py): with two or more complete rounds the third form wins or ties everywhere (c5 on one to
    // eight GPUs 4-6 %, a c4 shard on two GPUs 4 %); below that the phases of the last round are too unequal for it, and
    // cutting every octet pays once it recovers more than a tenth of the launch (a c4 shard on eight GPUs: 1.33 rounds,
    // 256 -> 172 us).
    auto idle = [&](double r) { return (ceil(r) - r) / ceil(r); };
    const double rounds = (double)octs / (double)resident;
    const long long full = (long long)floor(rounds) * resident;  // octets of the complete rounds
    long long n_whole = octs;
    if (nPh > 1) {
        if (env) n_whole = env[0] == '1' ? 0 : octs;
        else if (rounds >= 2.0) n_whole = full < octs ? full : octs;
        else if (idle(rounds) - idle(rounds * nPh) > 0.1) n_whole = 0;
    }
    const long long units = n_whole + (octs - n_whole) * nPh;
    const int grid = (int)std::max<long long>(1, std::min<long long>((long long)std::max(1, sms - P.reserve_sms) * per_sm, (units + wpc - 1) / wpc));
    kern<<<grid, threads, smem, st>>>(P, ii, Z, mu, f.want_g ? g : nullptr, jac, f.want_jac ? 1 : 0, f.want_hess ? 1 : 0, f.jets, n_whole);
    ++*launches;
    return true;
}

template <int NT, int M>
bool launch_octet(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f, cudaStream_t st,
                  long long* launches) {
    if (P.in[ii].G_stride != 0) {
        if (P.in[ii].bfrag == nullptr) return false;
        return launch_octet_pp<NT, M, true>(P, ii, Z, mu, g, jac, f, st, launches);
    }
    return launch_octet_pp<NT, M, false>(P, ii, Z, mu, g, jac, f, st, launches);
}

}  // namespace

// fragment-ordered copy of one problem's generators [G_0..G_m | G_0'..G_m'] (the layout the kernel stages in shared memory)
void bilinear_octet_fragments(int n, int m, const double* Gcm /* (m+1) column-major matrices */, double* out) {
    const int NT = n / 8, nn = n * n;
    for (int mat = 0; mat < 2 * (m + 1); ++mat)
        for (int t = 0; t < NT; ++t)
            for (int nt = 0; nt < NT; ++nt)
                for (int l = 0; l < 32; ++l) {
                    const int s = 8 * nt + (l >> 2), k = 8 * t + 2 * (l & 3);
                    double* o = out + ((((size_t)mat * NT + t) * NT + nt) * 32 + l) * 2;
                    for (int e = 0; e < 2; ++e)  // G[s][k] = Gcm[k*n + s];  G'[s][k] = G[k][s] = Gcm[s*n + k]
                        o[e] = mat <= m ? Gcm[(size_t)mat * nn + (size_t)(k + e) * n + s] : Gcm[(size_t)(mat - m - 1) * nn + (size_t)s * n + k + e];
                }
}
size_t bilinear_octet_fragment_doubles(int n, int m) { return (size_t)2 * (m + 1) * (n / 8) * (n / 8) * 32 * 2; }

bool bilinear_octet_supported(int n, int m) {
    if (n == 8) return m >= 1 && m <= 4;
    if (n == 16) return m >= 1 && m <= 2;
    return false;
}

bool launch_bilinear_octet(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f,
                           cudaStream_t st, long long* launches) {
    const DInt& I = P.in[ii];
    if (std::min(P.kc1, P.nI) - P.kc0 <= 0) return true;
    if (!bilinear_octet_supported(I.n, I.m)) return false;
    if (f.jets != DTO_JETS_NONE && I.jets == nullptr) return false;
    if (I.n == 8) {
        switch (I.m) {
            case 1: return launch_octet<1, 1>(P, ii, Z, mu, g, jac, f, st, launches);
            case 2: return launch_octet<1, 2>(P, ii, Z, mu, g, jac, f, st, launches);
            case 3: return launch_octet<1, 3>(P, ii, Z, mu, g, jac, f, st, launches);
            case 4: return launch_octet<1, 4>(P, ii, Z, mu, g, jac, f, st, launches);
        }
    } else if (I.n == 16) {
        switch (I.m) {
            case 1: return launch_octet<2, 1>(P, ii, Z, mu, g, jac, f, st, launches);
            case 2: return launch_octet<2, 2>(P, ii, Z, mu, g, jac, f, st, launches);
        }
    }
    return false;
}

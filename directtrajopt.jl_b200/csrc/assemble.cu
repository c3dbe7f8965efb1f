// K2/K3/K4/K5/K6: the HBM-bound kernels around the interval kernels.
//   analytic_kernel      DerivativeIntegrator residual + dense Jacobian block          (derivative_integrator.jl:45-86)
//   constraint_kernel    NonlinearKnotPointConstraint values + Jacobian (hyper-duals)   (knot_point_constraint.jl:235-268)
//   knot_program_kernel  the same for a constraint given as a knot program, one thread per seed
//   hessian_assemble     per-knot upper-triangle Hessian of the Lagrangian in COO order (evaluator.jl:560-647)
//   objective_kernel     objective value + dense gradient, warp-shuffle reductions       (_objectives.jl:111-128)
//   violation_kernel     max-norm constraint violation
//   jac_product_kernel   y = J w / J' w from the COO values                              (evaluator.jl:406-456)
#include "dto_internal.h"
#include "analytic_block.cuh"
#include "knotfun.cuh"

namespace {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block-wide sum, result valid in thread 0 (and broadcast through smem slot)
__device__ double block_sum(double v, double* red) {
    v = warp_sum(v);
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (l == 0) red[w] = v;
    __syncthreads();
    if (w == 0) {
        double t = (l < nw) ? red[l] : 0.0;
        t = warp_sum(t);
        if (l == 0) red[0] = t;
    }
    __syncthreads();
    return red[0];
}

// ------------------------------------------------------------------------------------------------
// K2: DerivativeIntegrator  f = x+ - x - dt*xdot : residual and full d x 2z block (zeros included)
// ------------------------------------------------------------------------------------------------
template <int GS>
__global__ void analytic_kernel(DProb P, const double* __restrict__ Z, double* __restrict__ g, double* __restrict__ jac,
                                long long total) {
    // one group of GS lanes per (problem, interval)
    const long long item = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / GS;
    if (item >= total) return;
    const int nIc = min(P.kc1, P.nI) - P.kc0;  // intervals of the active range
    const int b = (int)(item / nIc), kl = P.kc0 + (int)(item % nIc);
    analytic_interval(P, Z, g, jac, b, kl, threadIdx.x % GS, GS);
}

// ------------------------------------------------------------------------------------------------
// K5: knot constraints, one thread per (problem, owned time entry)
// ------------------------------------------------------------------------------------------------
__global__ void constraint_kernel(DProb P, int ci, const double* __restrict__ Z, double* __restrict__ g, double* __restrict__ jac,
                                  double* __restrict__ dense_probe) {
    const DCon& C = P.co[ci];
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)P.batch * C.nt_own) return;
    const int b = (int)(t / C.nt_own), j = (int)(t % C.nt_own);
    const int kl = C.own_knot[j];
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * P.z;
    const double* gp = Z + (long long)b * P.n_vars_local + (long long)P.nK * P.z;  // global variables
    const double* p = C.params + (long long)C.own_ti[j] * C.np;
    const int nv = C.nv, gd = C.gd;
    if (g != nullptr) {
        double out[16];
        knot_cfun<false, double>(C.fn, C.prog, ValueVars{zk, gp, C.var_offs, C.nvk}, nv, p, out, gd);
        double* gp = g + (long long)b * P.n_cons_local + C.row_off + (long long)j * gd;
        for (int a = 0; a < gd; ++a) gp[a] = out[a];
    }
    if (jac != nullptr || dense_probe != nullptr) {
        HDual out[16];
        for (int i = 0; i < nv; ++i) {
            knot_cfun<false, HDual>(C.fn, C.prog, SeededVars{zk, gp, C.var_offs, C.nvk, i, -1}, nv, p, out, gd);
            for (int a = 0; a < gd; ++a) {
                const long long e = ((long long)j * gd + a) * nv + i;
                if (dense_probe != nullptr) {
                    if (b == 0) dense_probe[e] = out[a].d1;
                } else {
                    const long long pos = C.jac_pos[e];
                    if (pos >= 0) jac[(long long)b * P.nnz_jac_local + pos] = out[a].d1;
                }
            }
        }
    }
}

// K5 for knot programs: one thread per (problem, owned time entry, seed).  Seed 0 evaluates the values, seed 1 + i the
// Jacobian column of variable i.  A program of 100 operations costs a few thousand instructions per seed; the catalogue
// kernel's loop over the nv seeds in one thread would leave most of the GPU idle.
__global__ void knot_program_kernel(DProb P, int ci, const double* __restrict__ Z, double* __restrict__ g, double* __restrict__ jac,
                                    double* __restrict__ dense_probe, int seed0, int seeds, long long total) {
    const DCon& C = P.co[ci];
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int seed = seed0 + (int)(t % seeds);
    const long long r = t / seeds;
    const int b = (int)(r / C.nt_own), j = (int)(r % C.nt_own);
    const int kl = C.own_knot[j];
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * P.z;
    const double* gp = Z + (long long)b * P.n_vars_local + (long long)P.nK * P.z;  // global variables
    const double* p = C.params + (long long)C.own_ti[j] * C.np;
    const int nv = C.nv, gd = C.gd;
    if (seed == 0) {
        double out[16];
        run_knot_program<double, ValueVars>(C.prog.code, C.prog.n_code, ValueVars{zk, gp, C.var_offs, C.nvk}, p, out);
        double* gr = g + (long long)b * P.n_cons_local + C.row_off + (long long)j * gd;
        for (int a = 0; a < gd; ++a) gr[a] = out[a];
        return;
    }
    const int i = seed - 1;
    HDual out[16];
    run_knot_program<HDual, SeededVars>(C.prog.code, C.prog.n_code, SeededVars{zk, gp, C.var_offs, C.nvk, i, -1}, p, out);
    for (int a = 0; a < gd; ++a) {
        const long long e = ((long long)j * gd + a) * nv + i;
        if (dense_probe != nullptr) {
            if (b == 0) dense_probe[e] = out[a].d1;
        } else {
            const long long pos = C.jac_pos[e];
            if (pos >= 0) jac[(long long)b * P.nnz_jac_local + pos] = out[a].d1;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// K3: Hessian of the Lagrangian, one CTA per (problem, owned knot)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void sym_add(double* diag, int z, int i, int j, double v) {
    if (i <= j) diag[i * z + j] += v;
    else diag[j * z + i] += v;
}

// parameter p of integrator I -> (0: own knot, 1: next knot, component offset)
__device__ __forceinline__ void int_param(const DInt& I, int dt_off, int p, int& next, int& comp) {
    if (I.kind == DTO_INT_BILINEAR) {
        next = 0;
        comp = p < I.m ? I.u_off + p : dt_off;
    } else {  // tdbilinear: [u0 (m), u1 (m, order 1), dt, t]
        const int nu = I.order == 1 ? 2 * I.m : I.m;
        if (p < I.m) { next = 0; comp = I.u_off + p; }
        else if (p < nu) { next = 1; comp = I.u_off + (p - I.m); }
        else if (p == nu) { next = 0; comp = dt_off; }
        else { next = 0; comp = I.t_off; }
    }
}
__device__ __forceinline__ int int_nparam(const DInt& I) {
    return I.kind == DTO_INT_BILINEAR ? I.m + 1 : (I.order == 1 ? 2 * I.m : I.m) + 2;
}

// One group of GS lanes per (problem, owned knot) -- a whole warp for wide knots, 16 or 8 lanes for narrow ones
// (z <= 24 / z <= 16: a warp would idle most of its lanes and the kernel is latency-bound); several knots per
// CTA, each with its own z x z tile(s) in shared memory.
template <int GS>
__device__ __forceinline__ double group_sum(double v, unsigned gmask) {
#pragma unroll
    for (int o = GS / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o);
    return v;
}

// Narrow knots are register-limited at the compiler's own allocation (68 registers: 3 CTAs of 256 threads per SM, a third
// of the warp slots, too few loads in flight for a latency-bound stream-out): capped to 5 (GS = 8) / 4 (GS = 16) CTAs per SM
// (c5: 560 -> 477 us, 0.62 of the measured HBM copy rate).
// Left: the launch covers only local knot 0 of a linked shard that starts after knot 1 (hessian_assemble_left_kernel); the
// previous interval's rows were received from the left neighbour into the leading row of DInt::hs (shard_link.cu).
template <int GS, bool Prog, bool Left>
__device__ __forceinline__ void hessian_assemble_body(const DProb& P, const double* __restrict__ Z, double sigma,
                                                      const double* __restrict__ mu, double* __restrict__ hess, int warps_per_cta,
                                                      long long total) {
    extern __shared__ double sm[];
    constexpr int GPW = 32 / GS;  // groups per warp
    const int z = P.z, lane = threadIdx.x & 31, tid = lane % GS, nt = GS;
    const int warp = (threadIdx.x >> 5) * GPW + lane / GS;  // group index inside the CTA
    const unsigned gmask = GS == 32 ? 0xffffffffu : (((1u << GS) - 1u) << ((lane / GS) * GS));
    const long long item = (long long)blockIdx.x * warps_per_cta * GPW + warp;
    const int tiles = P.any_cross ? 2 : 1;
    // gather table of the stream-out, built once per CTA: entry e of a knot's region (column-major upper triangle with the
    // z cross rows in front of every column) -> index into the knot's [diag | cross] tiles, 0xFFFFFFFF = structural zero
    // (only for narrow knots, GS < 32: many knots share a CTA and the table; a wide knot has a CTA almost to itself and
    // decodes its entries incrementally instead)
    unsigned int* tab = reinterpret_cast<unsigned int*>(sm + (size_t)warps_per_cta * GPW * tiles * z * z);
    if constexpr (GS < 32) {
        const int region_c = z * z + z * (z + 1) / 2;
        for (int e = threadIdx.x; e < region_c; e += blockDim.x) {
            int l = 0, i = e;
            while (i >= z + l + 1) {
                i -= z + l + 1;
                ++l;
            }
            tab[e] = i < z ? (P.any_cross ? (unsigned int)(z * z + i * z + l) : 0xFFFFFFFFu) : (unsigned int)((i - z) * z + l);
        }
        __syncthreads();
    }
    if (item >= total) return;
    const int nKc = min(P.kc1, P.nOwn) - P.kc0;  // owned knots of the active range
    const int b = (int)(item / nKc), kl = P.kc0 + (int)(item % nKc);
    double* diag = sm + (size_t)warp * tiles * z * z;  // z*z, entries (i<=l) used
    double* cross = diag + z * z;                      // z*z if any_cross: cross[i*z + l] = H[knot kl-1 comp i][knot kl comp l]
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * z;
    const double* gpz = Z + (long long)b * P.n_vars_local + (long long)P.nK * z;  // global variables
    const double* mub = mu + (long long)b * P.n_cons_local;
    const bool has_cross = hess_knot_has_cross(P, kl);
    for (int e = tid; e < tiles * z * z; e += nt) diag[e] = 0.0;
    __syncwarp(gmask);

    for (int ii = 0; ii < P.n_int; ++ii) {
        const DInt& I = P.in[ii];
        if (I.kind == DTO_INT_DERIVATIVE) {
            if (kl < P.nI) {
                const double* mup = mub + I.row_off + (long long)kl * I.n;
                for (int a = tid; a < I.n; a += nt) sym_add(diag, z, I.u_off + a, P.dt_off, -mup[a]);
            }
            __syncwarp(gmask);
            continue;
        }
        const int np = int_nparam(I), n = I.n;
        if (kl < P.nI) {  // own interval: entries among this knot's variables
            const double* hs = I.hs + ((long long)b * P.nI + kl) * I.hs_stride;
            const double* hpp = hs + (long long)np * n;
            for (int e = tid; e < np * n; e += nt) {
                const int p = e / n, a = e % n;
                int nx, comp;
                int_param(I, P.dt_off, p, nx, comp);
                if (!nx) sym_add(diag, z, I.x_off + a, comp, hs[e]);
            }
            __syncwarp(gmask);
            for (int e = tid; e < np * np; e += nt) {
                const int p = e / np, q = e % np;
                if (p > q) continue;
                int nxp, cp, nxq, cq;
                int_param(I, P.dt_off, p, nxp, cp);
                int_param(I, P.dt_off, q, nxq, cq);
                if (!nxp && !nxq) sym_add(diag, z, cp, cq, hpp[e]);
            }
            __syncwarp(gmask);
        }
        if (I.kind == DTO_INT_TDBILINEAR && I.order == 1 && (kl >= 1 || Left)) {
            // previous interval: (next,next) -> this knot's diagonal block; (own,next) -> cross block (Left: row -1)
            const double* hs = I.hs + ((long long)b * P.nI + (kl - 1)) * I.hs_stride;
            const double* hpp = hs + (long long)np * n;
            for (int e = tid; e < np * n; e += nt) {
                const int p = e / n, a = e % n;
                int nx, comp;
                int_param(I, P.dt_off, p, nx, comp);
                if (nx) cross[(I.x_off + a) * z + comp] += hs[e];
            }
            __syncwarp(gmask);
            for (int e = tid; e < np * np; e += nt) {
                const int p = e / np, q = e % np;
                int nxp, cp, nxq, cq;
                int_param(I, P.dt_off, p, nxp, cp);
                int_param(I, P.dt_off, q, nxq, cq);
                if (nxp && nxq) {
                    if (p <= q) sym_add(diag, z, cp, cq, hpp[e]);
                } else if (!nxp && nxq) {
                    cross[cp * z + cq] += hpp[e];
                }
            }
            __syncwarp(gmask);
        }
    }

    // knot constraints at this knot: sum_a mu_a * Hess g_a  (hyper-dual pairs)
    for (int ci = 0; ci < P.n_con; ++ci) {
        const DCon& C = P.co[ci];
        const int j = C.knot_to_own[kl];
        if (j >= 0) {
            const int nv = C.nv, nvk = C.nvk, gd = C.gd;  // (knot, global) and (global, global) entries: launch_global_hessian
            const double* p = C.params + (long long)C.own_ti[j] * C.np;
            const double* mup = mub + C.row_off + (long long)j * gd;
            for (int e = tid; e < nvk * nvk; e += nt) {
                const int a = e / nvk, c = e % nvk;
                if (a > c) continue;
                HDual out[16];
                knot_cfun<Prog, HDual>(C.fn, C.prog, SeededVars{zk, gpz, C.var_offs, nvk, a, c}, nv, p, out, gd);
                double s = 0.0;
                for (int q = 0; q < gd; ++q) s = fma(mup[q], out[q].d12, s);
                sym_add(diag, z, C.var_offs[a], C.var_offs[c], s);
            }
        }
        __syncwarp(gmask);
    }

    // objective: sigma * sum_i w_i Hess J_i   (skipped entirely when sigma == 0, evaluator.jl:626)
    if (sigma != 0.0) {
        for (int oi = 0; oi < P.n_obj; ++oi) {
            const DObj& O = P.ob[oi];
            if (O.kind == DTO_OBJ_QUADREG) {
                if (O.knot_to_own[kl] >= 0) {
                    const double dt = zk[P.dt_off], sw = sigma * O.weight;
                    const long long kg = (long long)P.kb - 1 + kl;  // global 0-based knot
                    double part = 0.0;
                    for (int a = tid; a < O.nv; a += nt) {
                        const int va = O.var_offs[a];
                        const double dv = zk[va] - (O.baseline ? O.baseline[kg * O.nv + a] : 0.0);
                        diag[va * z + va] += sw * dt * dt * O.R[a];
                        // written only at (row v, col dt): survives the upper-triangle filter iff v <= dt
                        // (regularizers.jl:160, evaluator.jl:637)
                        if (va <= P.dt_off && va != P.dt_off) diag[va * z + P.dt_off] += sw * 2.0 * dt * O.R[a] * dv;
                        part += O.R[a] * dv * dv;
                    }
                    const double q = group_sum<GS>(part, gmask);
                    __syncwarp(gmask);
                    if (tid == 0) diag[P.dt_off * z + P.dt_off] += sw * q;
                }
                __syncwarp(gmask);
            }
            if (O.kind == DTO_OBJ_LINREG) {
                // d2J/(dv ddt) = R, written at (row v, col dt) only (regularizers.jl:287-313): kept iff v precedes dt
                if (O.knot_to_own[kl] >= 0)
                    for (int a = tid; a < O.nv; a += nt) {
                        const int va = O.var_offs[a];
                        if (va < P.dt_off) diag[va * z + P.dt_off] += sigma * O.weight * O.R[a];
                    }
                __syncwarp(gmask);
            }
            if ((O.kind == DTO_OBJ_KNOT || O.kind == DTO_OBJ_GLOBAL_KNOT) && O.nvk > 0 && P.knot_side != nullptr) {
                // the pairs w Q d2l/dv_a dv_c of a listed knot were evaluated by knot_objective_pairs_kernel (one thread per
                // hyper-dual pair, beside the interval kernels); lane-private (a, c - a) cursor over the packed upper triangle
                const int j = O.knot_to_own[kl];
                if (j >= 0) {
                    const int nv = O.nvk, npairs = nv * (nv + 1) / 2;
                    const double* sd = P.knot_side + (long long)b * P.side_stride + O.side_off + (long long)j * npairs;
                    int a = 0, p = tid;
                    while (a < nv && p >= nv - a) {
                        p -= nv - a;
                        ++a;
                    }
                    for (int e = tid; e < npairs; e += nt) {
                        sym_add(diag, z, O.var_offs[a], O.var_offs[a + p], sigma * sd[e]);
                        p += nt;
                        while (a < nv && p >= nv - a) {
                            p -= nv - a;
                            ++a;
                        }
                    }
                }
                __syncwarp(gmask);
            }
        }
    }

    // stream the knot's region out in COO order: per column l: [z cross rows][l+1 diagonal rows]; the region is
    // contiguous, so the warp walks it linearly (coalesced) and decodes (column, row) incrementally
    double* hp = hess + (long long)b * P.nnz_hess_local + hess_knot_base(P, kl);
    const int ncross = has_cross ? z : 0;
    const int region = ncross * z + z * (z + 1) / 2;
    if (GS < 32 && has_cross) {
        for (int e = tid; e < region; e += GS) {
            const unsigned t = tab[e];
            hp[e] = t == 0xFFFFFFFFu ? 0.0 : diag[t];
        }
    } else if (has_cross && P.hess_tab != nullptr) {
        // wide knots: the same table, built once at construction, read from global memory (L2-resident, coalesced) --
        // the incremental (column, row) decode below costs ~500 cycles per 32 entries
#pragma unroll 4
        for (int e = tid; e < region; e += GS) {
            const unsigned t = __ldg(P.hess_tab + e);
            hp[e] = t == 0xFFFFFFFFu ? 0.0 : diag[t];
        }
    } else {
        // wide knots, and the first knot of the trajectory (no cross rows): lane-private (column l, row-in-column i) cursor advanced by GS entries
        int l = 0, i = tid;
        while (l < z && i >= ncross + l + 1) {
            i -= ncross + l + 1;
            ++l;
        }
        for (int e = tid; e < region; e += GS) {
            double v;
            if (i < ncross) v = P.any_cross ? cross[i * z + l] : 0.0;
            else v = diag[(i - ncross) * z + l];
            hp[e] = v;
            i += GS;
            while (l < z && i >= ncross + l + 1) {
                i -= ncross + l + 1;
                ++l;
            }
        }
    }
}

template <int GS, bool Prog>
__global__ void __launch_bounds__(256, GS == 8 ? 5 : (GS == 16 ? 4 : 1))
hessian_assemble_kernel(DProb P, const double* __restrict__ Z, double sigma, const double* __restrict__ mu, double* __restrict__ hess,
                        int warps_per_cta, long long total) {
    hessian_assemble_body<GS, Prog, false>(P, Z, sigma, mu, hess, warps_per_cta, total);
}

template <int GS, bool Prog>
__global__ void __launch_bounds__(256, GS == 8 ? 5 : (GS == 16 ? 4 : 1))
hessian_assemble_left_kernel(DProb P, const double* __restrict__ Z, double sigma, const double* __restrict__ mu,
                             double* __restrict__ hess, int warps_per_cta, long long total) {
    hessian_assemble_body<GS, Prog, true>(P, Z, sigma, mu, hess, warps_per_cta, total);
}

// Knot-objective Hessians: w * Q * Hess l, one thread per (problem, listed knot, variable pair), into DProb::knot_side (a
// terminal cost on a 32- or 64-dimensional state is one knot with ~500-2000 hyper-dual evaluations, which would serialise
// inside the per-knot warp of the assembler).  Depends on Z only: it runs beside the interval kernels on the second stream
// and the assembler adds sigma times the pairs to the knot's tile.
template <bool Prog>
__global__ void knot_objective_pairs_kernel(DProb P, int oi, const double* __restrict__ Z, long long total) {
    const DObj& O = P.ob[oi];
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const int nv = O.nvk, npairs = nv * (nv + 1) / 2, z = P.z;  // pairs of knot variables
    const int pair = (int)(t % npairs);
    const long long r = t / npairs;
    const int j = (int)(r % O.nt_own), b = (int)(r / O.nt_own);
    int a = 0, p = pair;
    while (p >= nv - a) {
        p -= nv - a;
        ++a;
    }
    const int c = a + p;
    const int kl = O.own_knot[j];
    if (kl < P.kc0 || kl >= P.kc1) return;  // assembled by another launch of the pipeline
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * z;
    const double* prm = O.params + (long long)O.own_ti[j] * O.np;
    const double* gp = Z + (long long)b * P.n_vars_local + (long long)P.nK * z;
    const HDual res = knot_lfun<Prog, HDual>(O.fn, O.prog, SeededVars{zk, gp, O.var_offs, nv, a, c}, O.nv, prm);
    P.knot_side[(long long)b * P.side_stride + O.side_off + (long long)j * npairs + pair] = O.weight * O.Qs[O.own_ti[j]] * res.d12;
}

// ------------------------------------------------------------------------------------------------
// K6: objective value + gradient, one WARP per (problem, owned knot); partial sums reduced in a
// second, deterministic pass.
// ------------------------------------------------------------------------------------------------
template <int GS, bool Prog>
__global__ void objective_kernel(DProb P, const double* __restrict__ Z, double* __restrict__ grad, double* __restrict__ partials,
                                 int warps_per_cta, long long total) {
    extern __shared__ double sm[];
    constexpr int GPW = 32 / GS;
    const int z = P.z, lane = threadIdx.x & 31, tid = lane % GS, nt = GS;
    const int warp = (threadIdx.x >> 5) * GPW + lane / GS;  // group index inside the CTA
    const unsigned gmask = GS == 32 ? 0xffffffffu : (((1u << GS) - 1u) << ((lane / GS) * GS));
    const long long item = (long long)blockIdx.x * warps_per_cta * GPW + warp;
    if (item >= total) return;
    const int b = (int)(item / P.nOwn), kl = (int)(item % P.nOwn);
    double* gz = sm + (size_t)warp * z;
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * z;
    const double* gp = Z + (long long)b * P.n_vars_local + (long long)P.nK * z;  // global variables
    const long long kg = (long long)P.kb - 1 + kl;  // global 0-based knot
    for (int e = tid; e < z; e += nt) gz[e] = 0.0;
    __syncwarp(gmask);
    double Jk = 0.0;  // meaningful in lane 0 only
    for (int oi = 0; oi < P.n_obj; ++oi) {
        const DObj& O = P.ob[oi];
        if (O.kind == DTO_OBJ_QUADREG) {
            if (O.knot_to_own[kl] >= 0) {
                const double dt = zk[P.dt_off];
                double part = 0.0;
                for (int a = tid; a < O.nv; a += nt) {
                    const double dv = zk[O.var_offs[a]] - (O.baseline ? O.baseline[kg * O.nv + a] : 0.0);
                    gz[O.var_offs[a]] += O.weight * dt * dt * O.R[a] * dv;
                    part += O.R[a] * dv * dv;
                }
                const double q = group_sum<GS>(part, gmask);
                __syncwarp(gmask);
                if (tid == 0) {
                    Jk += O.weight * 0.5 * dt * dt * q;
                    gz[P.dt_off] += O.weight * q * dt;
                }
            }
            __syncwarp(gmask);
        } else if (O.kind == DTO_OBJ_LINREG) {
            // J = sum_t dt_t R'v_t (regularizers.jl:241-270)
            if (O.knot_to_own[kl] >= 0) {
                const double dt = zk[P.dt_off];
                double part = 0.0;
                for (int a = tid; a < O.nv; a += nt) {
                    gz[O.var_offs[a]] += O.weight * dt * O.R[a];
                    part += O.R[a] * zk[O.var_offs[a]];
                }
                const double q = group_sum<GS>(part, gmask);
                __syncwarp(gmask);
                if (tid == 0) {
                    Jk += O.weight * dt * q;
                    gz[P.dt_off] += O.weight * q;
                }
            }
            __syncwarp(gmask);
        } else if (O.kind == DTO_OBJ_MINTIME) {
            if (tid == 0 && kg < P.N - 1) {
                Jk += O.weight * O.D * zk[P.dt_off];
                gz[P.dt_off] += O.weight * O.D;
            }
            __syncwarp(gmask);
        } else if (O.kind == DTO_OBJ_KNOT || O.kind == DTO_OBJ_GLOBAL_KNOT) {
            // knot part of the gradient; the global part is launch_global_gradient's
            const int j = O.knot_to_own[kl];
            if (j >= 0) {
                const int nv = O.nv, nvk = O.nvk;
                const double* p = O.params + (long long)O.own_ti[j] * O.np;
                const double w = O.weight * O.Qs[O.own_ti[j]];
                if (tid == 0) Jk += w * knot_lfun<Prog, double>(O.fn, O.prog, ValueVars{zk, gp, O.var_offs, nvk}, nv, p);
                if (grad != nullptr)
                    for (int a = tid; a < nvk; a += nt) {
                        const HDual r = knot_lfun<Prog, HDual>(O.fn, O.prog, SeededVars{zk, gp, O.var_offs, nvk, a, -1}, nv, p);
                        gz[O.var_offs[a]] += w * r.d1;
                    }
            }
            __syncwarp(gmask);
        }
    }
    if (grad != nullptr)
        for (int e = tid; e < z; e += nt) grad[(long long)b * P.n_grad_local + (long long)kl * z + e] = gz[e];
    if (tid == 0 && partials != nullptr) partials[(long long)b * P.nOwn + kl] = Jk;
}

// deterministic two-level sum: fixed chunking, fixed tree
__global__ void objective_chunk_kernel(int nOwn, int chunk, const double* __restrict__ partials, double* __restrict__ chunks) {
    const int b = blockIdx.y, c = blockIdx.x;
    const int k0 = c * chunk, k1 = min(nOwn, k0 + chunk);
    double s = 0.0;
    for (int k = k0 + threadIdx.x; k < k1; k += blockDim.x) s += partials[(long long)b * nOwn + k];
    __shared__ double red[32];
    s = block_sum(s, red);
    if (threadIdx.x == 0) chunks[(long long)b * gridDim.x + c] = s;
}

__global__ void objective_reduce_kernel(int nOwn, const double* __restrict__ partials, double* __restrict__ J) {
    const int b = blockIdx.x;
    double s = 0.0;
    for (int k = threadIdx.x; k < nOwn; k += blockDim.x) s += partials[(long long)b * nOwn + k];
    __shared__ double red[32];
    s = block_sum(s, red);
    if (threadIdx.x == 0) J[b] = s;
}

// ------------------------------------------------------------------------------------------------
__global__ void violation_kernel(long long n_cons, const double* __restrict__ g, const int* __restrict__ row_is_eq,
                                 double* __restrict__ viol) {
    const int b = blockIdx.y;
    double m = 0.0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n_cons; r += (long long)gridDim.x * blockDim.x) {
        const double v = g[(long long)b * n_cons + r];
        m = nan_max(m, row_is_eq[r] ? fabs(v) : nan_max(0.0, v));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = nan_max(m, __shfl_xor_sync(0xffffffffu, m, o));
    // non-negative doubles order like their bit patterns, and every NaN above +inf
    if ((threadIdx.x & 31) == 0) atomicMax((unsigned long long*)(viol + b), (unsigned long long)__double_as_longlong(m));
}

__global__ void jac_product_kernel(long long nnz, long long n_rows, long long n_cols, const double* __restrict__ jac,
                                   const long long* __restrict__ rows0, const long long* __restrict__ cols0,
                                   const double* __restrict__ w, double* __restrict__ y, int transpose) {
    const int b = blockIdx.y;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (long long)gridDim.x * blockDim.x) {
        const double v = jac[(long long)b * nnz + e];
        if (!transpose) atomicAdd(y + (long long)b * n_rows + rows0[e], v * w[(long long)b * n_cols + cols0[e]]);
        else atomicAdd(y + (long long)b * n_cols + cols0[e], v * w[(long long)b * n_rows + rows0[e]]);
    }
}

// Matrix-free J w / J' w of the analytic parts: DerivativeIntegrator rows (one warp per interval) and the stored
// knot-constraint entries (one thread per listed knot).  J w assigns its rows; J' w adds atomically (several
// integrators and constraints touch the same variable).
__global__ void analytic_product_kernel(DProb P, const double* __restrict__ Z, const double* __restrict__ w, double* __restrict__ y,
                                        int transpose, long long total) {
    const long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= total) return;
    const int b = (int)(item / P.nI), kl = (int)(item % P.nI), z = P.z, lane = threadIdx.x & 31;
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * z;
    const double dt = zk[P.dt_off];
    for (int ii = 0; ii < P.n_int; ++ii) {
        const DInt& I = P.in[ii];
        if (I.kind != DTO_INT_DERIVATIVE) continue;
        const int d = I.n;
        const long long row0 = (long long)b * P.n_cons_local + I.row_off + (long long)kl * d;
        if (!transpose) {
            const double* wk = w + (long long)b * P.n_vars_local + (long long)kl * z;
            for (int a = lane; a < d; a += 32)
                y[row0 + a] = wk[z + I.x_off + a] - wk[I.x_off + a] - dt * wk[I.u_off + a] - zk[I.u_off + a] * wk[P.dt_off];
        } else {
            double* yk = y + (long long)b * P.n_vars_local + (long long)kl * z;
            double part = 0.0;
            for (int a = lane; a < d; a += 32) {
                const double wa = w[row0 + a];
                atomicAdd(yk + I.x_off + a, -wa);
                atomicAdd(yk + I.u_off + a, -dt * wa);
                atomicAdd(yk + z + I.x_off + a, wa);
                part = fma(zk[I.u_off + a], wa, part);
            }
            part = warp_sum(part);
            if (lane == 0) atomicAdd(yk + P.dt_off, -part);
        }
    }
}

template <bool Prog>
__global__ void constraint_product_kernel(DProb P, int ci, const double* __restrict__ Z, const double* __restrict__ w,
                                          double* __restrict__ y, int transpose) {
    const DCon& C = P.co[ci];
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)P.batch * C.nt_own) return;
    const int b = (int)(t / C.nt_own), j = (int)(t % C.nt_own);
    const int kl = C.own_knot[j];
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * P.z;
    const double* gp = Z + (long long)b * P.n_vars_local + (long long)P.nK * P.z;
    const double* p = C.params + (long long)C.own_ti[j] * C.np;
    const int nv = C.nv, gd = C.gd;
    const long long row0 = (long long)b * P.n_cons_local + C.row_off + (long long)j * gd;
    const long long col0 = (long long)b * P.n_vars_local + (long long)kl * P.z;
    const long long gcol0 = (long long)b * P.n_vars_local + (long long)P.nK * P.z;
    double acc[16];
    for (int a = 0; a < gd; ++a) acc[a] = 0.0;
    HDual out[16];
    for (int i = 0; i < nv; ++i) {
        knot_cfun<Prog, HDual>(C.fn, C.prog, SeededVars{zk, gp, C.var_offs, C.nvk, i, -1}, nv, p, out, gd);
        double col = 0.0;
        for (int a = 0; a < gd; ++a) {
            if (C.jac_pos[((long long)j * gd + a) * nv + i] < 0) continue;  // never stored by the reference: not part of J
            if (!transpose) acc[a] = fma(out[a].d1, w[(i < C.nvk ? col0 : gcol0) + C.var_offs[i]], acc[a]);
            else col = fma(out[a].d1, w[row0 + a], col);
        }
        if (transpose) atomicAdd(y + (i < C.nvk ? col0 : gcol0) + C.var_offs[i], col);
    }
    if (!transpose)
        for (int a = 0; a < gd; ++a) y[row0 + a] = acc[a];
}


// (parameter, parameter) block of the compact Hessian of a bilinear integrator from the stored second-order vectors of
// the forward jet (DInt::jets, written by the mu-independent pass over the iterate): hpp = -mu' W.  One quad per
// entry; the lane owns elements 8 nt + 2 q + {0,1} and the sums run in the order of the interval kernels
// (fma chain over nt, then the two xor-shuffles), so the two-pass result has the bits of the single pass.
__global__ void hpp_contract_kernel(DProb P, int ii, const double* __restrict__ mu) {
    const DInt& I = P.in[ii];
    const int n = I.n, m = I.m, np = m + 1, J2 = m * (m + 1) / 2, nout = J2 + 1 + m, NT = n / 8;
    const int q = threadIdx.x & 3;
    const long long nIc = min(P.kc1, P.nI) - P.kc0;
    const long long total = (long long)P.batch * nIc * nout;
    const long long quad = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    const bool valid = quad < total;
    const long long qd = valid ? quad : total - 1;
    const int o = (int)(qd % nout);
    const long long item = qd / nout;
    const int b = (int)(item / nIc), kk = P.kc0 + (int)(item % nIc);
    const double* mup = mu + (long long)b * P.n_cons_local + I.row_off + (long long)kk * n;
    const double* W = I.jets + ((long long)b * P.nI + kk) * I.jet_stride;
    auto dot = [&](int v) {
        const double* w = W + (long long)v * n;
        double s = 0.0;
        for (int nt = 0; nt < NT; ++nt) s = fma(mup[8 * nt + 2 * q], w[8 * nt + 2 * q], fma(mup[8 * nt + 2 * q + 1], w[8 * nt + 2 * q + 1], s));
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        return s;
    };
    double* hpp = I.hs + ((long long)b * P.nI + kk) * I.hs_stride + (long long)np * n;
    if (o < J2) {
        const double s1 = dot(o);
        int p = o, a = 0;
        while (p >= m - a) {
            p -= m - a;
            ++a;
        }
        const int bb = a + p;
        if (valid && q == 0) {
            hpp[a * np + bb] = -s1;
            hpp[bb * np + a] = -s1;
        }
    } else if (o == J2) {
        const double dtt = dot(J2);
        if (valid && q == 0) hpp[m * np + m] = -dtt;
    } else {
        const int i = o - J2 - 1;
        const double dA = dot(J2 + 1 + i), dB = dot(J2 + 1 + m + i);
        if (valid && q == 0) {
            hpp[i * np + m] = -(dA + dB);
            hpp[m * np + i] = -(dA + dB);
        }
    }
}

bool any_program_constraint(const DProb& P) {
    for (int ci = 0; ci < P.n_con; ++ci)
        if (P.co[ci].fn == DTO_G_PROGRAM) return true;
    return false;
}

}  // namespace

void launch_hpp_contract(const DProb& P, int ii, const double* mu, cudaStream_t st, long long* launches) {
    const DInt& I = P.in[ii];
    const long long nIc = std::min(P.kc1, P.nI) - P.kc0;
    if (nIc <= 0 || I.jets == nullptr || I.hs == nullptr) return;
    const long long quads = (long long)P.batch * nIc * (I.m * (I.m + 1) / 2 + 1 + I.m);
    const int threads = 256;
    hpp_contract_kernel<<<(unsigned)((quads * 4 + threads - 1) / threads), threads, 0, st>>>(P, ii, mu);
    ++*launches;
}

void launch_analytic(const DProb& P, const double* Z, double* g, double* jac, EvalFlags f, cudaStream_t st, long long* launches) {
    bool any_deriv = false;
    for (int i = 0; i < P.n_int; ++i) any_deriv |= P.in[i].kind == DTO_INT_DERIVATIVE;
    const int nIc = std::min(P.kc1, P.nI) - P.kc0;
    if (P.analytic_fused) return;  // written by the bilinear kernel together with its own columns (bilinear_octet.cu)
    if (any_deriv && nIc > 0) {
        const long long total = (long long)nIc * P.batch;
        int dmax = 0;
        for (int i = 0; i < P.n_int; ++i)
            if (P.in[i].kind == DTO_INT_DERIVATIVE) dmax = std::max(dmax, P.in[i].n);
        if (2 * P.z * dmax <= 64)  // a handful of entries per interval: 8 lanes each
            analytic_kernel<8><<<(unsigned)((total + 31) / 32), 256, 0, st>>>(P, Z, f.want_g ? g : nullptr, f.want_jac ? jac : nullptr, total);
        else
            analytic_kernel<32><<<(unsigned)((total + 7) / 8), 256, 0, st>>>(P, Z, f.want_g ? g : nullptr, f.want_jac ? jac : nullptr, total);
        ++*launches;
    }
}

void launch_knot_program(const DProb& P, int ci, const double* Z, double* g, double* jac, double* dense_probe, cudaStream_t st,
                         long long* launches) {
    const DCon& C = P.co[ci];
    const bool want_jac = jac != nullptr || dense_probe != nullptr;
    const int seed0 = g != nullptr ? 0 : 1, seeds = (g != nullptr ? 1 : 0) + (want_jac ? C.nv : 0);
    const long long tot = (long long)P.batch * C.nt_own * seeds;
    if (tot == 0) return;
    knot_program_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(P, ci, Z, g, jac, dense_probe, seed0, seeds, tot);
    ++*launches;
}

void launch_constraints(const DProb& P, const double* Z, double* g, double* jac, EvalFlags f, cudaStream_t st, long long* launches) {
    for (int ci = 0; ci < P.n_con; ++ci) {
        const long long tot = (long long)P.batch * P.co[ci].nt_own;
        if (tot == 0) continue;
        if (P.co[ci].fn == DTO_G_PROGRAM) {
            launch_knot_program(P, ci, Z, f.want_g ? g : nullptr, f.want_jac ? jac : nullptr, nullptr, st, launches);
            continue;
        }
        constraint_kernel<<<(unsigned)((tot + 63) / 64), 64, 0, st>>>(P, ci, Z, f.want_g ? g : nullptr, f.want_jac ? jac : nullptr,
                                                                       nullptr);
        ++*launches;
    }
}

void launch_constraint_pattern_probe(const DProb& P, const double* Z, double* dense, cudaStream_t st, long long* launches) {
    long long off = 0;
    for (int ci = 0; ci < P.n_con; ++ci) {
        const DCon& C = P.co[ci];
        const long long tot = (long long)P.batch * C.nt_own;
        if (tot && C.fn == DTO_G_PROGRAM) {
            launch_knot_program(P, ci, Z, nullptr, nullptr, dense + off, st, launches);
        } else if (tot) {
            constraint_kernel<<<(unsigned)((tot + 63) / 64), 64, 0, st>>>(P, ci, Z, nullptr, nullptr, dense + off);
            ++*launches;
        }
        off += (long long)C.nt_own * C.gd * C.nv;
    }
}

// warps per CTA of the Hessian assembler and its dynamic shared memory: every knot group stages its z x z diagonal tile
// (and the cross tile when some integrator couples neighbouring knots)
static size_t hessian_assemble_plan(const DProb& P, int& W) {
    const size_t per_group = sizeof(double) * (size_t)P.z * P.z * (P.any_cross ? 2 : 1);
    const int GS = P.z <= 16 ? 8 : (P.z <= 24 ? 16 : 32), GPW = 32 / GS;
    W = 8;
    while (W > 1 && W * GPW * per_group > 64 * 1024) W >>= 1;
    const size_t tab_bytes = (sizeof(unsigned int) * ((size_t)P.z * P.z + (size_t)P.z * (P.z + 1) / 2) + 15) / 16 * 16;
    return W * GPW * per_group + (GS < 32 ? tab_bytes : 0);
}

size_t hessian_assemble_smem_bytes(const DProb& P) {
    int W;
    return hessian_assemble_plan(P, W);
}

template <int GS, bool PROG>
static bool configure_assemble(bool left_block, std::string& err) {
    const std::string args = "<" + std::to_string(GS) + (PROG ? ", true>" : ", false>");
    return opt_in_smem(hessian_assemble_kernel<GS, PROG>, 227 * 1024, "hessian_assemble_kernel" + args, err) &&
           (!left_block || opt_in_smem(hessian_assemble_left_kernel<GS, PROG>, 227 * 1024, "hessian_assemble_left_kernel" + args, err));
}

// the form launch_hessian_assemble picks for this problem, and its left-knot form if the handle launches it
bool hessian_assemble_configure(const DProb& P, bool left_block, std::string& err) {
    if (hessian_assemble_smem_bytes(P) <= 48 * 1024) return true;
    const int GS = P.z <= 16 ? 8 : (P.z <= 24 ? 16 : 32);
    if (any_program_constraint(P))
        return GS == 8 ? configure_assemble<8, true>(left_block, err)
                       : (GS == 16 ? configure_assemble<16, true>(left_block, err) : configure_assemble<32, true>(left_block, err));
    return GS == 8 ? configure_assemble<8, false>(left_block, err)
                   : (GS == 16 ? configure_assemble<16, false>(left_block, err) : configure_assemble<32, false>(left_block, err));
}

void launch_hessian_assemble(const DProb& P, const double* Z, double sigma, const double* mu, double* hess, cudaStream_t st,
                             long long* launches, bool left_block) {
    const int nKc = std::min(P.kc1, P.nOwn) - P.kc0;
    if (nKc <= 0) return;
    const int GS = P.z <= 16 ? 8 : (P.z <= 24 ? 16 : 32), GPW = 32 / GS;
    int W;
    const size_t smem = hessian_assemble_plan(P, W);
    const long long total = (long long)nKc * P.batch;
    const unsigned grid = (unsigned)((total + (long long)W * GPW - 1) / ((long long)W * GPW));
    if (left_block) {  // local knot 0 only (kc0 = 0, kc1 = 1)
        const bool prog = any_program_constraint(P);
        if (GS == 8) (prog ? hessian_assemble_left_kernel<8, true> : hessian_assemble_left_kernel<8, false>)<<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
        else if (GS == 16) (prog ? hessian_assemble_left_kernel<16, true> : hessian_assemble_left_kernel<16, false>)<<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
        else (prog ? hessian_assemble_left_kernel<32, true> : hessian_assemble_left_kernel<32, false>)<<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
    } else if (any_program_constraint(P)) {
        if (GS == 8) hessian_assemble_kernel<8, true><<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
        else if (GS == 16) hessian_assemble_kernel<16, true><<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
        else hessian_assemble_kernel<32, true><<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
    } else {
        if (GS == 8) hessian_assemble_kernel<8, false><<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
        else if (GS == 16) hessian_assemble_kernel<16, false><<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
        else hessian_assemble_kernel<32, false><<<grid, W * 32, smem, st>>>(P, Z, sigma, mu, hess, W, total);
    }
    ++*launches;
}

// the knot-objective pairs of the active range (nothing to do without knot objectives there)
bool launch_knot_objective_pairs(const DProb& P, const double* Z, cudaStream_t st, long long* launches) {
    if (P.knot_side == nullptr) return false;
    bool any = false;
    for (int oi = 0; oi < P.n_obj; ++oi) {
        const DObj& O = P.ob[oi];
        if ((O.kind != DTO_OBJ_KNOT && O.kind != DTO_OBJ_GLOBAL_KNOT) || O.nt_own == 0 || O.nvk == 0) continue;
        if (O.own_kmax < P.kc0 || O.own_kmin >= P.kc1) continue;  // no listed knot in the active range
        const long long tot = (long long)P.batch * O.nt_own * (O.nvk * (O.nvk + 1) / 2);
        if (O.fn == DTO_L_PROGRAM) knot_objective_pairs_kernel<true><<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(P, oi, Z, tot);
        else knot_objective_pairs_kernel<false><<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(P, oi, Z, tot);
        ++*launches;
        any = true;
    }
    return any;
}

void launch_objective(const DProb& P, const double* Z, double* J, double* grad, double* partials, cudaStream_t st,
                      long long* launches) {
    if (P.nOwn <= 0) return;
    const int W = 8;
    const int GS = P.z <= 16 ? 8 : (P.z <= 24 ? 16 : 32), GPW = 32 / GS;
    const size_t smem = sizeof(double) * (size_t)P.z * W * GPW;
    const long long total = (long long)P.nOwn * P.batch;
    const unsigned grid = (unsigned)((total + (long long)W * GPW - 1) / ((long long)W * GPW));
    bool prog = false;
    for (int oi = 0; oi < P.n_obj; ++oi) prog |= P.ob[oi].fn == DTO_L_PROGRAM && (P.ob[oi].kind == DTO_OBJ_KNOT || P.ob[oi].kind == DTO_OBJ_GLOBAL_KNOT);
    if (prog) {
        if (GS == 8) objective_kernel<8, true><<<grid, W * 32, smem, st>>>(P, Z, grad, J ? partials : nullptr, W, total);
        else if (GS == 16) objective_kernel<16, true><<<grid, W * 32, smem, st>>>(P, Z, grad, J ? partials : nullptr, W, total);
        else objective_kernel<32, true><<<grid, W * 32, smem, st>>>(P, Z, grad, J ? partials : nullptr, W, total);
    } else {
        if (GS == 8) objective_kernel<8, false><<<grid, W * 32, smem, st>>>(P, Z, grad, J ? partials : nullptr, W, total);
        else if (GS == 16) objective_kernel<16, false><<<grid, W * 32, smem, st>>>(P, Z, grad, J ? partials : nullptr, W, total);
        else objective_kernel<32, false><<<grid, W * 32, smem, st>>>(P, Z, grad, J ? partials : nullptr, W, total);
    }
    ++*launches;
    if (J) {
        // partials layout: [batch][nOwn] followed by [batch][nchunks] of scratch
        const int chunk = 2048;
        const int nchunks = (P.nOwn + chunk - 1) / chunk;
        if (nchunks > 1) {
            double* chunks = partials + (long long)P.batch * P.nOwn;
            objective_chunk_kernel<<<dim3(nchunks, P.batch), 256, 0, st>>>(P.nOwn, chunk, partials, chunks);
            objective_reduce_kernel<<<P.batch, 256, 0, st>>>(nchunks, chunks, J);
            *launches += 2;
        } else {
            objective_reduce_kernel<<<P.batch, 256, 0, st>>>(P.nOwn, partials, J);
            ++*launches;
        }
    }
}

void launch_violation(const DProb& P, const double* g, const int* row_is_eq, double* viol, cudaStream_t st, long long* launches) {
    cudaMemsetAsync(viol, 0, sizeof(double) * P.batch, st);
    if (P.n_cons_local == 0) return;
    dim3 grid((unsigned)((P.n_cons_local + 255) / 256 > 1184 ? 1184 : (P.n_cons_local + 255) / 256), P.batch);
    violation_kernel<<<grid, 256, 0, st>>>(P.n_cons_local, g, row_is_eq, viol);
    ++*launches;
}

void launch_jac_product(const DProb& P, const double* jac, const long long* rows0, const long long* cols0, const double* w,
                        double* y, bool transpose, cudaStream_t st, long long* launches) {
    const long long n_rows = P.n_cons_local, n_cols = P.n_vars_local;
    cudaMemsetAsync(y, 0, sizeof(double) * (transpose ? n_cols : n_rows) * P.batch, st);
    if (P.nnz_jac_local == 0) return;
    dim3 grid((unsigned)((P.nnz_jac_local + 255) / 256 > 2368 ? 2368 : (P.nnz_jac_local + 255) / 256), P.batch);
    jac_product_kernel<<<grid, 256, 0, st>>>(P.nnz_jac_local, n_rows, n_cols, jac, rows0, cols0, w, y, transpose ? 1 : 0);
    ++*launches;
}

void launch_analytic_product(const DProb& P, const double* Z, const double* w, double* y, bool transpose, cudaStream_t st,
                             long long* launches) {
    bool any_deriv = false;
    for (int i = 0; i < P.n_int; ++i) any_deriv |= P.in[i].kind == DTO_INT_DERIVATIVE;
    if (any_deriv && P.nI > 0) {
        const long long total = (long long)P.nI * P.batch;
        analytic_product_kernel<<<(unsigned)((total + 7) / 8), 256, 0, st>>>(P, Z, w, y, transpose ? 1 : 0, total);
        ++*launches;
    }
    for (int ci = 0; ci < P.n_con; ++ci) {
        const long long tot = (long long)P.batch * P.co[ci].nt_own;
        if (tot == 0) continue;
        if (P.co[ci].fn == DTO_G_PROGRAM)
            constraint_product_kernel<true><<<(unsigned)((tot + 63) / 64), 64, 0, st>>>(P, ci, Z, w, y, transpose ? 1 : 0);
        else
            constraint_product_kernel<false><<<(unsigned)((tot + 63) / 64), 64, 0, st>>>(P, ci, Z, w, y, transpose ? 1 : 0);
        ++*launches;
    }
}

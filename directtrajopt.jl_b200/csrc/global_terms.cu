// K8: terms that read global (non-time-varying) variables -- GlobalObjective / GlobalKnotPointObjective
// (src/objectives/global_objectives.jl:35-341), NonlinearGlobalConstraint (src/constraints/nonlinear/global_constraint.jl:24-159)
// and NonlinearGlobalKnotPointConstraint (src/constraints/nonlinear/global_knot_point_constraint.jl:30-256).
//
// A term evaluates a catalogue function on [knot variables at times[i]; global variables].  Values, the knot part of
// the gradient, the Jacobian (all columns, through the precomputed scatter map) and the (knot, knot) Hessian entries
// come out of the ordinary knot kernels of assemble.cu, whose variable accessors read both segments.  What is left
// couples every listed knot to the SAME few global variables, i.e. reductions over the knots:
//   global part of the gradient      g[zN + gi]   = sum_slots w Q dl/dg_gi            (global_objectives.jl:262-266)
//   (global, global) Hessian entries H[gi, gj]    = sum_slots factor d2/(dg_gi dg_gj)  (global_objectives.jl:334-337,
//                                                                                       global_knot_point_constraint.jl:243-245)
//   (knot, global) Hessian entries   H[(k,a), gi] = factor d2/(dv_a dg_gi)             (one slot each)
// One "slot" = (term, listed time).  Each slot writes its contribution to a slot-major scratch row; a second kernel sums
// the columns in a fixed order (bit-reproducible).  All of them live in the tail of the Hessian value array: the global
// columns come after every knot column in the column-major upper triangle (evaluator.jl:199-203).
#include "dto_internal.h"
#include "knotfun.cuh"

namespace {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// thread per (problem, objective slot, global variable)
template <bool Prog>
__global__ void global_grad_kernel(DProb P, const double* __restrict__ Z, long long total) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const DGlob& L = P.gl;
    const int gi = (int)(t % L.G);
    const long long r = t / L.G;
    const int s = (int)(r % L.S_obj), b = (int)(r / L.S_obj);
    const DObj& O = P.ob[L.slot_term[s]];
    const int j = L.slot_j[s];
    const int v = O.g2l[gi];
    double val = 0.0;
    if (v >= 0) {
        const double* zk = Z + (long long)b * P.n_vars_local + (long long)O.own_knot[j] * P.z;
        const double* gp = Z + (long long)b * P.n_vars_local + (long long)P.nK * P.z;
        const double* prm = O.params + (long long)O.own_ti[j] * O.np;
        const HDual res = knot_lfun<Prog, HDual>(O.fn, O.prog, SeededVars{zk, gp, O.var_offs, O.nvk, v, -1}, O.nv, prm);
        val = O.weight * O.Qs[O.own_ti[j]] * res.d1;
    }
    L.scratchG[((long long)b * L.S_obj + s) * L.G + gi] = val;
}

// thread per (problem, slot, item): item < Gtri -> (gi <= gj) pair into the scratch; then (knot variable a, global gi)
template <bool Prog>
__global__ void global_hess_kernel(DProb P, const double* __restrict__ Z, double sigma, const double* __restrict__ mu,
                                   double* __restrict__ hess, double* __restrict__ kg_probe, long long total) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= total) return;
    const DGlob& L = P.gl;
    const int G = L.G, gtri = G * (G + 1) / 2, items = gtri + L.KV * G;
    const int item = (int)(t % items);
    const long long r = t / items;
    const int s = (int)(r % L.S), b = (int)(r / L.S);
    const bool is_obj = s < L.S_obj;
    const int j = L.slot_j[s];
    const double* gp = Z + (long long)b * P.n_vars_local + (long long)P.nK * P.z;

    // local variable indices (a <= c in the term's numbering: knot variables precede globals)
    int a, c, gi = 0, gj = 0;
    const int* g2l = is_obj ? P.ob[L.slot_term[s]].g2l : P.co[L.slot_term[s]].g2l;
    const int nvk = is_obj ? P.ob[L.slot_term[s]].nvk : P.co[L.slot_term[s]].nvk;
    if (item < gtri) {
        int p = item;
        while (p >= G - gi) {
            p -= G - gi;
            ++gi;
        }
        gj = gi + p;
        a = g2l[gi];
        c = g2l[gj];
    } else {
        a = (item - gtri) / G;
        gi = (item - gtri) % G;
        c = g2l[gi];
        if (a >= nvk) a = -1;
    }
    double val = 0.0;
    if (a >= 0 && c >= 0) {
        if (is_obj) {
            if (sigma != 0.0) {  // evaluator.jl:626
                const DObj& O = P.ob[L.slot_term[s]];
                const double* zk = Z + (long long)b * P.n_vars_local + (long long)O.own_knot[j] * P.z;
                const double* prm = O.params + (long long)O.own_ti[j] * O.np;
                const HDual res = knot_lfun<Prog, HDual>(O.fn, O.prog, SeededVars{zk, gp, O.var_offs, O.nvk, a, c}, O.nv, prm);
                val = sigma * O.weight * O.Qs[O.own_ti[j]] * res.d12;
            }
        } else {
            const DCon& C = P.co[L.slot_term[s]];
            const double* zk = Z + (long long)b * P.n_vars_local + (long long)C.own_knot[j] * P.z;
            const double* prm = C.params + (long long)C.own_ti[j] * C.np;
            HDual out[16];
            knot_cfun<Prog, HDual>(C.fn, C.prog, SeededVars{zk, gp, C.var_offs, C.nvk, a, c}, C.nv, prm, out, C.gd);
            if (kg_probe != nullptr) {  // structure probe: mu = ones (evaluator.jl:170-171)
                for (int q = 0; q < C.gd; ++q) val += out[q].d12;
            } else {
                const double* mup = mu + (long long)b * P.n_cons_local + C.row_off + (long long)j * C.gd;
                for (int q = 0; q < C.gd; ++q) val = fma(mup[q], out[q].d12, val);
            }
        }
    }
    if (item < gtri) {
        L.scratchH[((long long)b * L.S + s) * gtri + item] = val;
    } else if (a >= 0 && c >= 0) {
        const long long e = ((long long)s * L.KV + a) * G + gi;
        if (kg_probe != nullptr) {
            if (b == 0) kg_probe[e] = val;
        } else {
            const long long pos = L.kg_pos[e];
            // several terms may couple the same (knot variable, global) pair: at most a handful of adds per entry
            if (pos >= 0) atomicAdd(hess + (long long)b * P.nnz_hess_local + L.hess_tail_off + pos, val);
        }
    }
}

// out[b*out_stride + out_off + pos[w]] = sum_s scratch[b][s][w]; one warp per (problem, column), fixed order
__global__ void column_sum_kernel(int batch, int S, int W, const double* __restrict__ scratch, const long long* __restrict__ pos,
                                  double* __restrict__ out, long long out_stride, long long out_off) {
    const long long item = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= (long long)batch * W) return;
    const int b = (int)(item / W), w = (int)(item % W), lane = threadIdx.x & 31;
    const long long p = pos ? pos[w] : w;
    if (p < 0) return;
    double acc = 0.0;
    for (int s = lane; s < S; s += 32) acc += scratch[((long long)b * S + s) * W + w];
    acc = warp_sum(acc);
    if (lane == 0) out[(long long)b * out_stride + out_off + p] = acc;
}

// some term with global variables is a knot program (objectives: obj = true, constraints: obj = false)
bool global_programs(const DProb& P, bool obj) {
    for (int i = 0; i < P.n_obj && obj; ++i)
        if (P.ob[i].kind == DTO_OBJ_GLOBAL_KNOT && P.ob[i].fn == DTO_L_PROGRAM) return true;
    for (int i = 0; i < P.n_con && !obj; ++i)
        if (P.co[i].nv > P.co[i].nvk && P.co[i].fn == DTO_G_PROGRAM) return true;
    return false;
}

}  // namespace

void launch_global_gradient(const DProb& P, const double* Z, double* grad, cudaStream_t st, long long* launches) {
    const DGlob& L = P.gl;
    if (L.G == 0 || grad == nullptr) return;
    if (L.S_obj > 0) {
        const long long total = (long long)P.batch * L.S_obj * L.G;
        if (global_programs(P, true)) global_grad_kernel<true><<<(unsigned)((total + 127) / 128), 128, 0, st>>>(P, Z, total);
        else global_grad_kernel<false><<<(unsigned)((total + 127) / 128), 128, 0, st>>>(P, Z, total);
        ++*launches;
    }
    const long long cols = (long long)P.batch * L.G;
    column_sum_kernel<<<(unsigned)((cols + 3) / 4), 128, 0, st>>>(P.batch, L.S_obj, L.G, L.scratchG, nullptr, grad, P.n_grad_local,
                                                                  (long long)P.nOwn * P.z);
    ++*launches;
}

void launch_global_hessian(const DProb& P, const double* Z, double sigma, const double* mu, double* hess, double* kg_probe,
                           cudaStream_t st, long long* launches) {
    const DGlob& L = P.gl;
    if (L.G == 0 || L.S == 0) return;
    const int gtri = L.G * (L.G + 1) / 2;
    if (kg_probe == nullptr) {
        if (L.n_hess_tail == 0) return;
        cudaMemset2DAsync(hess + L.hess_tail_off, sizeof(double) * P.nnz_hess_local, 0, sizeof(double) * L.n_hess_tail, P.batch, st);
    }
    const long long total = (long long)P.batch * L.S * (gtri + L.KV * L.G);
    if (global_programs(P, true) || global_programs(P, false))
        global_hess_kernel<true><<<(unsigned)((total + 127) / 128), 128, 0, st>>>(P, Z, sigma, mu, hess, kg_probe, total);
    else
        global_hess_kernel<false><<<(unsigned)((total + 127) / 128), 128, 0, st>>>(P, Z, sigma, mu, hess, kg_probe, total);
    ++*launches;
    if (kg_probe == nullptr) {
        const long long cols = (long long)P.batch * gtri;
        column_sum_kernel<<<(unsigned)((cols + 3) / 4), 128, 0, st>>>(P.batch, L.S, gtri, L.scratchH, L.gg_pos, hess, P.nnz_hess_local,
                                                                      L.hess_tail_off);
        ++*launches;
    }
}

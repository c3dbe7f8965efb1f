// K1 (generic variant): BilinearIntegrator interval kernel for state dimensions up to 96 whose block fits shared memory.
// A block holds the generator and every jet column of its interval (generic_smem_bytes): with the Hessian on a B200
// (227 KB per block) that is n <= 83 at one drive and n <= 76 at four; dto_create rejects larger shapes.
//
// One warp per (problem, interval).  Replaces `expv` + ForwardDiff through it
// (/root/reference/src/integrators/bilinear_integrator.jl:81,98-161): the warp propagates, through a
// scaled truncated Taylor series of exp(dt*G(u)), the state x together with its first and second
// directional derivatives w.r.t. the drives, the columns of the identity (giving the propagator E for
// the -E Jacobian block) and, for the Hessian, the multiplier mu with its first derivatives through
// the transposed generator.  Everything that depends on dt is closed-form on top of those
// (d/ddt exp(dt G) x = G exp(dt G) x).  The residual and the dense x_dim x 2z Jacobian block are
// written straight into the reference's COO order; the second derivatives go to a compact scratch
// that the Hessian assembler (K3) consumes.
//
// This is the correctness-first fallback (LDS-bound); state dimensions that are multiples of 8 take
// the DMMA tensor-core variant in bilinear_dmma.cu.
#include "dto_internal.h"

namespace {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_max(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

__global__ void __launch_bounds__(32) bilinear_generic_kernel(DProb P, int ii, const double* __restrict__ Z,
                                                               const double* __restrict__ mu, double* __restrict__ g,
                                                               double* __restrict__ jac, int want_jac, int want_hess) {
    extern __shared__ double sm[];
    const DInt I = P.in[ii];
    const int n = I.n, m = I.m, z = P.z;
    const int lane = threadIdx.x;
    const int b = blockIdx.x / P.nI, kl = blockIdx.x % P.nI;
    const double* zk = Z + (long long)b * P.n_vars_local + (long long)kl * z;
    const double* zk1 = zk + z;
    if (P.halo != nullptr && kl + 1 == P.nK - 1) zk1 = P.halo;
    const double* G = I.G + (long long)b * I.G_stride;
    const int ld = n | 1;  // odd leading dimension: conflict-free row and column access
    const int n2 = m * (m + 1) / 2;
    const int nfwd = want_hess ? 1 + m + n2 : (want_jac ? 1 + m : 1);
    const int colE = nfwd;
    const int nE = want_jac ? n : 0;
    const int colA = colE + nE;
    const int nadj = want_hess ? 1 + m : 0;
    const int ncol = colA + nadj;

    double* Gu = sm;                 // ld * n
    double* V = Gu + ld * n;         // ncol * n   accumulated series
    double* Ta = V + ncol * n;       // ncol * n   current term
    double* Tb = Ta + ncol * n;      // ncol * n   next term
    double* tmp = Tb + ncol * n;     // 3 * n

    const double dt = zk[P.dt_off];
    // Gu = G0 + sum u_i G_i
    for (int e = lane; e < n * n; e += 32) {
        int r = e % n, c = e / n;
        double s = G[e];
        for (int i = 0; i < m; ++i) s = fma(zk[I.u_off + i], G[(long long)(1 + i) * n * n + e], s);
        Gu[r + c * ld] = s;
    }
    __syncwarp();
    // theta = |dt| * ||Gu||_1
    double cmax = 0.0;
    for (int c = lane; c < n; c += 32) {
        double s = 0.0;
        for (int r = 0; r < n; ++r) s += fabs(Gu[r + c * ld]);
        cmax = fmax(cmax, s);
    }
    const double theta = fabs(dt) * warp_max(cmax);
    int s_stages = 1, T = 2;
    double poison = __longlong_as_double(0x7ff8000000000000LL);  // generator norm not finite or absurd: NaN out
    if (theta < 1e8) {
        poison = 1.0;
        s_stages = theta > 4.0 ? (int)ceil(theta * 0.25) : 1;
        double ths = theta / s_stages, term = ths;
        T = 1;
        while (term > 1.1102230246251565e-16 && T < 60) {  // 2^-53, as series_tables.cuh
            ++T;
            term *= ths / T;
        }
        T += 2;
    }
    // initial values
    for (int e = lane; e < ncol * n; e += 32) {
        int col = e / n, r = e % n;
        double v = 0.0;
        if (col == 0) v = zk[I.x_off + r];
        else if (col >= colE && col < colA) v = (col - colE == r) ? 1.0 : 0.0;
        else if (col == colA && nadj) v = mu[(long long)b * P.n_cons_local + I.row_off + (long long)kl * n + r];
        V[e] = v;
    }
    __syncwarp();
    for (int st = 0; st < s_stages; ++st) {
        for (int e = lane; e < ncol * n; e += 32) Ta[e] = V[e];
        __syncwarp();
        for (int q = 1; q <= T; ++q) {
            const double c = poison * dt / ((double)q * (double)s_stages);
            for (int e = lane; e < ncol * n; e += 32) {
                const int col = e / n, r = e % n;
                double acc = 0.0;
                if (col < colA) {
                    // forward family and E columns: Gu * t_col
                    const double* t = Ta + col * n;
                    for (int k = 0; k < n; ++k) acc = fma(Gu[r + k * ld], t[k], acc);
                    if (col >= 1 && col <= m) {
                        const double* Gi = G + (long long)col * n * n;  // drive col-1 is matrix index col
                        const double* t0 = Ta;
                        for (int k = 0; k < n; ++k) acc = fma(Gi[r + k * n], t0[k], acc);
                    } else if (col > m && col < colE) {
                        int p = col - 1 - m, i = 0;
                        while (p >= m - i) {
                            p -= m - i;
                            ++i;
                        }
                        const int j = i + p;
                        const double* Gi = G + (long long)(1 + i) * n * n;
                        const double* Gj = G + (long long)(1 + j) * n * n;
                        const double* ti = Ta + (1 + i) * n;
                        const double* tj = Ta + (1 + j) * n;
                        for (int k = 0; k < n; ++k) {
                            acc = fma(Gi[r + k * n], tj[k], acc);
                            acc = fma(Gj[r + k * n], ti[k], acc);
                        }
                    }
                } else {
                    // adjoint family: Gu' * a_col
                    const double* t = Ta + col * n;
                    for (int k = 0; k < n; ++k) acc = fma(Gu[k + r * ld], t[k], acc);
                    if (col > colA) {
                        const double* Gi = G + (long long)(col - colA) * n * n;
                        const double* a0 = Ta + colA * n;
                        for (int k = 0; k < n; ++k) acc = fma(Gi[k + r * n], a0[k], acc);
                    }
                }
                acc *= c;
                Tb[e] = acc;
                V[e] += acc;
            }
            __syncwarp();
            double* sw = Ta;
            Ta = Tb;
            Tb = sw;
        }
    }
    // ---- epilogue ----
    const double* F = V;
    double* gF = tmp;        // Gu F
    double* gTmu = tmp + n;  // Gu' mu
    double* hxt = tmp + 2 * n;  // Gu' Y
    for (int r = lane; r < n; r += 32) {
        double a = 0.0;
        for (int k = 0; k < n; ++k) a = fma(Gu[r + k * ld], F[k], a);
        gF[r] = a;
        if (want_hess) {
            const double* Y = V + colA * n;
            const double* mup = mu + (long long)b * P.n_cons_local + I.row_off + (long long)kl * n;
            double a2 = 0.0, a3 = 0.0;
            for (int k = 0; k < n; ++k) {
                a2 = fma(Gu[k + r * ld], mup[k], a2);
                a3 = fma(Gu[k + r * ld], Y[k], a3);
            }
            gTmu[r] = a2;
            hxt[r] = a3;
        }
    }
    __syncwarp();
    if (g != nullptr) {
        double* gp = g + (long long)b * P.n_cons_local + I.row_off + (long long)kl * n;
        for (int r = lane; r < n; r += 32) gp[r] = zk1[I.x_off + r] - F[r];
    }
    if (want_jac) {
        double* jp = jac + (long long)b * P.nnz_jac_local;
        const long long own_off = jac_own_off(P, kl, I.doff, n);
        const long long prev_off = jac_prev_off(P, kl + 1, I.doff);
        for (int e = lane; e < 2 * z * n; e += 32) {
            const int l = e / n, a = e % n;
            double v = 0.0;
            long long pos;
            if (l < z) {
                if (l >= I.x_off && l < I.x_off + n) v = -V[(colE + (l - I.x_off)) * n + a];
                else if (l >= I.u_off && l < I.u_off + m) v = -V[(1 + (l - I.u_off)) * n + a];
                else if (l == P.dt_off) v = -gF[a];
                pos = jac_col(P, kl, l) + own_off + a;
            } else {
                const int lp = l - z;
                if (lp - I.x_off == a) v = 1.0;
                pos = jac_col(P, (kl + 1), lp) + prev_off + a;
            }
            jp[pos] = v;
        }
    }
    if (want_hess) {
        // compact scratch, parameters p = [u_1..u_m, dt]:  hx[p][n] = d2(mu'r)/(dx dp) | hpp[p][q] = d2(mu'r)/(dp dq)
        const int np = m + 1;
        double* hs = I.hs + ((long long)b * P.nI + kl) * I.hs_stride;
        const double* mup = mu + (long long)b * P.n_cons_local + I.row_off + (long long)kl * n;
        for (int e = lane; e < m * n; e += 32) hs[e] = -V[(colA + 1) * n + e];
        for (int r = lane; r < n; r += 32) hs[m * n + r] = -hxt[r];
        double* hpp = hs + np * n;
        int p = 0;
        for (int i = 0; i < m; ++i)
            for (int j = i; j < m; ++j, ++p) {
                double s = 0.0;
                const double* w = V + (1 + m + p) * n;
                for (int r = lane; r < n; r += 32) s = fma(mup[r], w[r], s);
                s = warp_sum(s);
                if (lane == 0) {
                    hpp[i * np + j] = -s;
                    hpp[j * np + i] = -s;
                }
            }
        for (int i = 0; i < m; ++i) {
            const double* Gi = G + (long long)(1 + i) * n * n;
            const double* wi = V + (1 + i) * n;
            double s = 0.0;
            for (int r = lane; r < n; r += 32) {
                double a = 0.0;
                for (int k = 0; k < n; ++k) a = fma(Gi[r + k * n], F[k], a);
                s = fma(mup[r], a, s);
                s = fma(gTmu[r], wi[r], s);
            }
            s = warp_sum(s);
            if (lane == 0) {
                hpp[i * np + m] = -s;
                hpp[m * np + i] = -s;
            }
        }
        double s = 0.0;
        for (int r = lane; r < n; r += 32) s = fma(gTmu[r], gF[r], s);
        s = warp_sum(s);
        if (lane == 0) hpp[m * np + m] = -s;
    }
}

}  // namespace

size_t generic_smem_bytes(int n, int m, bool want_jac, bool want_hess) {
    int n2 = m * (m + 1) / 2;
    int nfwd = want_hess ? 1 + m + n2 : (want_jac ? 1 + m : 1);
    int ncol = nfwd + (want_jac ? n : 0) + (want_hess ? 1 + m : 0);
    return sizeof(double) * ((size_t)(n | 1) * n + 3 * (size_t)ncol * n + 3 * n);
}

void launch_bilinear_generic(const DProb& P, int ii, const double* Z, const double* mu, double* g, double* jac, EvalFlags f,
                             cudaStream_t st, long long* launches) {
    const DInt& I = P.in[ii];
    if (P.nI <= 0) return;
    size_t smem = generic_smem_bytes(I.n, I.m, f.want_jac, f.want_hess);
    static PerDeviceOnce configured;
    if (smem > 48 * 1024 && configured.first()) {
        cudaFuncSetAttribute(bilinear_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    }
    bilinear_generic_kernel<<<P.nI * P.batch, 32, smem, st>>>(P, ii, Z, mu, f.want_g ? g : nullptr, jac, f.want_jac ? 1 : 0,
                                                               f.want_hess ? 1 : 0);
    ++*launches;
}

// Series plan of the bilinear interval kernels: how many Taylor terms exp(dt G(u_k)) needs, per interval.
//
// The reference's `expv` (ExponentialAction.jl: Al-Mohy & Higham 2011) does not size its truncated Taylor series from
// ||A||_1 but from norms of POWERS of A, which bound ||A^k||^(1/k) far better for oscillatory or non-normal generators.
// Here: d2 = ||A^2||_1^(1/2).  Since ||A^(2j)|| <= ||A^2||^j and ||A^(2j+1)|| <= ||A^2||^j ||A||, the tail of the series is
// bounded by (||A||_1 / d2) sum_k d2^k / k!; one term beyond T(d2) absorbs the factor whenever ||A||_1 <= T(d2) + 1.
// At config c2 (n = 32): ||A||_1 = 1.0, d2 = 0.50 -- 16 terms instead of 19 for a 2^-53 tail.
//
// A = dt (G_0 + sum_i u_i G_i) is affine in u, so A^2 = dt^2 sum_{a<=b} w_a w_b S_ab with w = (1, u) and the symmetrised
// pair products S_ab = G_a G_b + G_b G_a (S_aa = G_a^2) formed ONCE at construction: a plan costs (npairs + m + 1) n^2
// multiply-adds per interval (half of ONE n^3 product at c2; < 1 % of an interval's work) instead of matrix products.
// The estimate needs a few digits only, so the matrices are kept and summed in FP32 (half the shared-memory traffic, which
// is what bounds this kernel: every interval reads all npairs + m + 1 matrices) and each warp carries T = 4 intervals per
// matrix element it loads; the FP32 rounding (<= 1e-5 of sum_a |w_a| ||G_a||_1, resp. its square) is ADDED to the norms
// before they are used, so the plan stays an upper bound.
// One CTA per SM stages the matrices; lane = column, sums |.| down its columns.  plan = { alpha, theta1 = ||A||_1 }: the
// kernels take the stages from theta1 (round-off of e^|A|) and the terms per stage from alpha / stages, where alpha is
// the argument that makes T(alpha) = min(T(theta1), T(d2) + 1).
// Every variant, pass, range, batch member and shard reads the same plan: their results stay bit-identical to each other.
#include "dto_internal.h"
#include "series_tables.cuh"
#include "bulk_copy.cuh"
#include <algorithm>
#include <cmath>
#include <vector>

namespace {

// (per-problem generator sets get no plan: the kernels keep ||dt G||_1 for them)
// NM = m + 1 matrices; GS lanes share T consecutive intervals (GS = n when n divides 32: 32 / n groups per warp, else 32)
template <int NM, int T>
__global__ void __launch_bounds__(512) series_plan_kernel(DProb P, int ii, const double* __restrict__ Z, double2* __restrict__ plan, int gs) {
    extern __shared__ __align__(128) float smf[];
    constexpr int NP = NM * (NM + 1) / 2;
    const DInt& I = P.in[ii];
    const int n = I.n, nn = n * n;
    const int lane = threadIdx.x & 31, wic = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    {   // stage [G_0..G_m | S_pairs] with the bulk-copy engine: per-thread loads made this copy 56 % of the kernel's time
        __shared__ __align__(8) unsigned long long bar;
        bulk_stage(smf, I.planmat, (unsigned)((NM + NP) * nn * sizeof(float)), &bar);  // a multiple of 16 bytes: n is even
    }
    const float *G = smf, *S = smf + NM * nn;
    const float* gnorm = I.planmat + (size_t)(NM + NP) * nn;  // ||G_a||_1, rounded up
    const int per_warp = 32 / gs, sub = lane / gs, c0 = lane % gs;
    const long long nIc = min(P.kc1, P.nI) - P.kc0, items = (long long)P.batch * nIc;
    const long long groups = (items + T - 1) / T, tasks = (groups + per_warp - 1) / per_warp;
    for (long long task = (long long)blockIdx.x * wpc + wic; task < tasks; task += (long long)gridDim.x * wpc) {
        const long long item0 = (task * per_warp + sub) * T;
        float w[T][NM], wp[T][NP];  // (1, u) and its pair products
        double dt[T], gsum[T];
#pragma unroll
        for (int t = 0; t < T; ++t) {
            const long long it = min(item0 + t, items - 1);
            const int b = (int)(it / nIc), kk = P.kc0 + (int)(it % nIc);
            const double* zk = Z + (long long)b * P.n_vars_local + (long long)kk * P.z;
            dt[t] = fabs(zk[P.dt_off]);
            w[t][0] = 1.0f;
            gsum[t] = (double)gnorm[0];
#pragma unroll
            for (int a = 1; a < NM; ++a) {
                const double u = zk[I.u_off + a - 1];
                w[t][a] = (float)u;
                gsum[t] += fabs(u) * (double)gnorm[a];
            }
            int p = 0;
#pragma unroll
            for (int a = 0; a < NM; ++a)
#pragma unroll
                for (int bb = a; bb < NM; ++bb, ++p) wp[t][p] = w[t][a] * w[t][bb];
        }
        float c1[T], c2[T];  // largest column sums of |G(u)| and |G(u)^2|
#pragma unroll
        for (int t = 0; t < T; ++t) c1[t] = c2[t] = 0.0f;
        for (int c = c0; c < n; c += gs) {
            float s1[T], s2[T];
#pragma unroll
            for (int t = 0; t < T; ++t) s1[t] = s2[t] = 0.0f;
            for (int r = 0; r < n; ++r) {
                const int e = r * n + c;
                float v1[T], v2[T];
#pragma unroll
                for (int t = 0; t < T; ++t) v1[t] = v2[t] = 0.0f;
#pragma unroll
                for (int a = 0; a < NM; ++a) {
                    const float ga = G[a * nn + e];
#pragma unroll
                    for (int t = 0; t < T; ++t) v1[t] = fmaf(w[t][a], ga, v1[t]);
                }
#pragma unroll
                for (int p = 0; p < NP; ++p) {
                    const float sp = S[p * nn + e];
#pragma unroll
                    for (int t = 0; t < T; ++t) v2[t] = fmaf(wp[t][p], sp, v2[t]);
                }
#pragma unroll
                for (int t = 0; t < T; ++t) {
                    s1[t] += fabsf(v1[t]);
                    s2[t] += fabsf(v2[t]);
                }
            }
#pragma unroll
            for (int t = 0; t < T; ++t) {
                c1[t] = fmaxf(c1[t], s1[t]);
                c2[t] = fmaxf(c2[t], s2[t]);
            }
        }
#pragma unroll
        for (int t = 0; t < T; ++t) {
            for (int o = gs >> 1; o > 0; o >>= 1) {
                c1[t] = fmaxf(c1[t], __shfl_xor_sync(0xffffffffu, c1[t], o));
                c2[t] = fmaxf(c2[t], __shfl_xor_sync(0xffffffffu, c2[t], o));
            }
        }
        if (c0 < T && item0 + c0 < items) {  // lane c0 of the group finishes interval item0 + c0
            double n1 = 0.0, n2 = 0.0, gs1 = 0.0, dtt = 0.0;
#pragma unroll
            for (int t = 0; t < T; ++t)
                if (t == c0) {
                    n1 = (double)c1[t];
                    n2 = (double)c2[t];
                    gs1 = gsum[t];
                    dtt = dt[t];
                }
            // FP32 rounding of the sums, added: the plan stays an upper bound
            double theta1 = dtt * (n1 + 1e-5 * gs1), d2 = dtt * sqrt(n2 + 1e-5 * gs1 * gs1);
            // an iterate whose crude bound dt sum_a |w_a| ||G_a||_1 is not finite or absurd may have overflowed the FP32 sums
            // (and fmaxf drops NaN): hand the crude bound on, the interval kernels turn it into NaN outputs (choose_series)
            if (!(dtt * gs1 < 1e7)) theta1 = d2 = dtt * gs1;
            // alpha: an argument with T(alpha) = min(T(theta1), T(d2) + 1)
            double alpha = theta1;
            if (theta1 < 1e8 && d2 < theta1) {
                const double inv_st = theta1 > 4.0 ? 1.0 / ceil(theta1 * 0.25) : 1.0;  // as choose_series
                const int t1 = taylor_terms(theta1 * inv_st), t2 = taylor_terms(d2 * inv_st) + 1;
                if (t2 < t1 && theta1 * inv_st <= (double)t2) alpha = kTermThr[t2] / inv_st;
            }
            const long long it = item0 + c0;
            const int b = (int)(it / nIc), kk = P.kc0 + (int)(it % nIc);
            plan[(long long)b * P.nI + kk] = make_double2(alpha, theta1);
        }
    }
}

}  // namespace

// shared memory the staged matrices need; 0: no plan (too many drives, odd n, or the matrices do not fit: the kernels fall
// back to ||dt G||_1)
size_t series_plan_smem(int n, int m) {
    if (m > 4 || (n & 1) || n < 4) return 0;
    const size_t nmat = m + 1, bytes = sizeof(float) * (nmat + nmat * (nmat + 1) / 2) * n * n;
    return bytes <= 200 * 1024 ? bytes : 0;
}

// the matrices the plan kernel stages, FP32: [G_0..G_m row-major | S_ab, a <= b, row-major | ||G_a||_1 rounded up]
void series_plan_matrices(int n, int m, const double* Gcm /* (m+1) column-major matrices */, std::vector<float>& out) {
    const int nmat = m + 1, npairs = nmat * (nmat + 1) / 2;
    const size_t nn = (size_t)n * n;
    out.assign((nmat + npairs) * nn + nmat, 0.0f);
    for (int a = 0; a < nmat; ++a) {
        double n1 = 0.0;
        for (int c = 0; c < n; ++c) {
            double sum = 0.0;
            for (int r = 0; r < n; ++r) {
                const double v = Gcm[a * nn + (size_t)c * n + r];
                out[a * nn + (size_t)r * n + c] = (float)v;
                sum += fabs(v);
            }
            n1 = std::max(n1, sum);
        }
        out[(nmat + npairs) * nn + a] = (float)(n1 * (1.0 + 1e-6));
    }
    int p = 0;
    for (int a = 0; a < nmat; ++a)
        for (int bb = a; bb < nmat; ++bb, ++p)
            for (int r = 0; r < n; ++r)
                for (int c = 0; c < n; ++c) {
                    double v = 0.0;
                    for (int k = 0; k < n; ++k) {
                        v += Gcm[a * nn + (size_t)k * n + r] * Gcm[bb * nn + (size_t)c * n + k];
                        if (bb != a) v += Gcm[bb * nn + (size_t)k * n + r] * Gcm[a * nn + (size_t)c * n + k];
                    }
                    out[(nmat + p) * nn + (size_t)r * n + c] = (float)v;
                }
}

template <int NM>
static void launch_plan_nm(const DProb& P, int ii, const double* Z, double2* out, long long items, int sms, cudaStream_t st) {
    constexpr int T = 4;
    const DInt& I = P.in[ii];
    const size_t smem = series_plan_smem(I.n, I.m);
    const int gs = (I.n <= 32 && 32 % I.n == 0) ? I.n : 32, per_warp = 32 / gs;
    const long long groups = (items + T - 1) / T, tasks = (groups + per_warp - 1) / per_warp;
    // every CTA stages the matrices once: as few warps per CTA as keep all SMs busy
    int threads = 512;
    while (threads > 128 && (tasks + threads / 32 - 1) / (threads / 32) < sms) threads >>= 1;
    const int wpc = threads / 32;
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(2048 / threads, (220 * 1024) / (smem + 1024)));
    const int grid = (int)std::min<long long>((tasks + wpc - 1) / wpc, (long long)sms * per_sm);
    series_plan_kernel<NM, T><<<grid, threads, smem, st>>>(P, ii, Z, out, gs);
}

bool series_plan_configure(int m, std::string& err) {
    void (*const kern[])(DProb, int, const double*, double2*, int) = {series_plan_kernel<1, 4>, series_plan_kernel<2, 4>, series_plan_kernel<3, 4>,
                                                                     series_plan_kernel<4, 4>, series_plan_kernel<5, 4>};
    return opt_in_smem(kern[m], 200 * 1024, "series_plan_kernel<" + std::to_string(m + 1) + ", 4>", err);
}

void launch_series_plan(const DProb& P, int ii, const double* Z, cudaStream_t st, long long* launches) {
    const DInt& I = P.in[ii];
    const long long items = (long long)P.batch * (std::min(P.kc1, P.nI) - P.kc0);
    if (items <= 0) return;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    double2* out = const_cast<double2*>(I.plan);
    switch (I.m) {
        case 0: launch_plan_nm<1>(P, ii, Z, out, items, sms, st); break;
        case 1: launch_plan_nm<2>(P, ii, Z, out, items, sms, st); break;
        case 2: launch_plan_nm<3>(P, ii, Z, out, items, sms, st); break;
        case 3: launch_plan_nm<4>(P, ii, Z, out, items, sms, st); break;
        case 4: launch_plan_nm<5>(P, ii, Z, out, items, sms, st); break;
    }
    ++*launches;
}

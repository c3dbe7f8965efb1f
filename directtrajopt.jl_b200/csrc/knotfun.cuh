// Device catalogue of knot-point functions and the forward-mode hyper-dual number they are
// differentiated with; user functions given as knot programs dispatch to the interpreter of knot_program.cuh.  This replaces the ForwardDiff closures of the reference
// (src/constraints/nonlinear/knot_point_constraint.jl:254-294, src/objectives/knot_point_objectives.jl:184-243):
// every catalogue function is written once as a template over the scalar type and instantiated with
// `double` (values) and `HDual` (first and second derivatives in one pass: seeds e_a, e_b give
// d f/dv_a, d f/dv_b and d2 f/(dv_a dv_b)).
#pragma once
#include <math.h>

#include "dto_internal.h"

struct HDual {
    double v, d1, d2, d12;
    __host__ __device__ HDual() : v(0), d1(0), d2(0), d12(0) {}
    __host__ __device__ HDual(double a) : v(a), d1(0), d2(0), d12(0) {}
    __host__ __device__ HDual(double a, double b, double c, double d) : v(a), d1(b), d2(c), d12(d) {}
};
__host__ __device__ inline HDual operator+(const HDual& a, const HDual& b) { return HDual(a.v + b.v, a.d1 + b.d1, a.d2 + b.d2, a.d12 + b.d12); }
__host__ __device__ inline HDual operator-(const HDual& a, const HDual& b) { return HDual(a.v - b.v, a.d1 - b.d1, a.d2 - b.d2, a.d12 - b.d12); }
__host__ __device__ inline HDual operator-(const HDual& a) { return HDual(-a.v, -a.d1, -a.d2, -a.d12); }
__host__ __device__ inline HDual operator*(const HDual& a, const HDual& b) {
    return HDual(a.v * b.v, a.d1 * b.v + a.v * b.d1, a.d2 * b.v + a.v * b.d2, a.d12 * b.v + a.d1 * b.d2 + a.d2 * b.d1 + a.v * b.d12);
}
__host__ __device__ inline HDual operator+(const HDual& a, double b) { return HDual(a.v + b, a.d1, a.d2, a.d12); }
__host__ __device__ inline HDual operator-(const HDual& a, double b) { return HDual(a.v - b, a.d1, a.d2, a.d12); }
__host__ __device__ inline HDual operator-(double b, const HDual& a) { return HDual(b - a.v, -a.d1, -a.d2, -a.d12); }
__host__ __device__ inline HDual operator*(const HDual& a, double b) { return HDual(a.v * b, a.d1 * b, a.d2 * b, a.d12 * b); }
__host__ __device__ inline HDual operator*(double b, const HDual& a) { return a * b; }
__host__ __device__ inline HDual hd_sqrt(const HDual& a) {
    double s = sqrt(a.v);
    double f1 = 0.5 / s;            // d sqrt
    double f2 = -0.25 / (s * a.v);  // d2 sqrt
    return HDual(s, f1 * a.d1, f1 * a.d2, f1 * a.d12 + f2 * a.d1 * a.d2);
}
__host__ __device__ inline double hd_sqrt(double a) { return sqrt(a); }

// Variable accessors: the variables are never copied into a per-thread array -- `V(i)` builds the i-th
// (hyper-dual) variable on the fly, seeded in directions a and c.  Variables 0..nvk-1 are components of the
// knot (`zk[offs[i]]`), variables nvk.. are global variables (`gp[offs[i]]`, global_objectives.jl:230-240,
// global_knot_point_constraint.jl:151-155: [knot vars; global vars]).
struct ValueVars {
    const double* zk;
    const double* gp;
    const int* offs;
    int nvk;
    __host__ __device__ double operator()(int i) const { return i < nvk ? zk[offs[i]] : gp[offs[i]]; }
};
struct SeededVars {
    const double* zk;
    const double* gp;
    const int* offs;
    int nvk;
    int a, c;  // seed directions of d1 and d2 (-1: none)
    __host__ __device__ HDual operator()(int i) const {
        return HDual(i < nvk ? zk[offs[i]] : gp[offs[i]], i == a ? 1.0 : 0.0, i == c ? 1.0 : 0.0, 0.0);
    }
};

#ifdef __CUDACC__
#include "knot_program.cuh"
#endif

// `Prog`: whether the caller handles knot programs (DTO_G_PROGRAM / DTO_L_PROGRAM, compiled into `pg`).  Kernels are
// instantiated both ways and the host launches the program-capable form only for problems that have programs: the
// interpreter call costs the caller registers, and the catalogue-only forms keep the allocation they were tuned with.
// ---- constraint functions g(v; p) -> out[gd] ---------------------------------------------------
template <bool Prog, class T, class Vars>
__host__ __device__ inline void knot_cfun(int fn, const DProgram& pg, const Vars& v, int nv, const double* p, T* out, int gd) {
#ifdef __CUDA_ARCH__
    if constexpr (Prog) {
        if (fn == DTO_G_PROGRAM) {
            run_knot_program<T, Vars>(pg.code, pg.n_code, v, p, out);
            return;
        }
    }
#endif
    switch (fn) {
        case DTO_G_NORM_MINUS_C: {  // [norm(v) - c]
            T s = T(0.0);
            for (int i = 0; i < nv; ++i) s = s + v(i) * v(i);
            out[0] = hd_sqrt(s) - p[0];
        } break;
        case DTO_G_NORMSQ_MINUS_C: {  // [norm(v)^2 - c]
            T s = T(0.0);
            for (int i = 0; i < nv; ++i) s = s + v(i) * v(i);
            out[0] = s - p[0];
        } break;
        case DTO_G_SQDIST_MINUS_C: {  // [norm(v - p[1:])^2 - p[0]]
            T s = T(0.0);
            for (int i = 0; i < nv; ++i) {
                T d = v(i) - p[1 + i];
                s = s + d * d;
            }
            out[0] = s - p[0];
        } break;
        case DTO_G_LINEAR: {  // A v - b, p = [gd, A (gd x nv column-major), b]
            for (int a = 0; a < gd; ++a) {
                T s = T(0.0);
                for (int i = 0; i < nv; ++i) s = s + v(i) * p[1 + a + (long long)i * gd];
                out[a] = s - p[1 + (long long)gd * nv + a];
            }
        } break;
        case DTO_G_NORM_PRODUCT: {  // [norm(v1) - c1; norm(v1) norm(v2) - c2], p = [c1, c2, n1]
            const int n1 = (int)p[2];
            T s1 = T(0.0), s2 = T(0.0);
            for (int i = 0; i < n1; ++i) s1 = s1 + v(i) * v(i);
            for (int i = n1; i < nv; ++i) s2 = s2 + v(i) * v(i);
            const T r1 = hd_sqrt(s1), r2 = hd_sqrt(s2);
            out[0] = r1 - p[0];
            out[1] = r1 * r2 - p[1];
        } break;
        default:
            for (int a = 0; a < gd; ++a) out[a] = T(0.0);
    }
}

// ---- objective functions l(v; p) -> scalar ------------------------------------------------------
template <bool Prog, class T, class Vars>
__host__ __device__ inline T knot_lfun(int fn, const DProgram& pg, const Vars& v, int nv, const double* p) {
#ifdef __CUDA_ARCH__
    if constexpr (Prog) {
        if (fn == DTO_L_PROGRAM) {
            T r[1];
            run_knot_program<T, Vars>(pg.code, pg.n_code, v, p, r);
            return r[0];
        }
    }
#endif
    switch (fn) {
        case DTO_L_NORMSQ_PLUS_P: {
            T s = T(0.0);
            for (int i = 0; i < nv; ++i) s = s + v(i) * v(i);
            return s + p[0];
        }
        case DTO_L_SQDIST: {
            T s = T(0.0);
            for (int i = 0; i < nv; ++i) {
                T d = v(i) - p[i];
                s = s + d * d;
            }
            return s;
        }
        case DTO_L_LINEAR: {
            T s = T(0.0);
            for (int i = 0; i < nv; ++i) s = s + v(i) * p[i];
            return s;
        }
        case DTO_L_ISO_INFIDELITY: {  // 1 - |<goal|psi>|^2, v = [re; im], p = [gre; gim]
            int h = nv / 2;
            T a = T(0.0), b = T(0.0);
            for (int i = 0; i < h; ++i) {
                a = a + v(i) * p[i] + v(h + i) * p[h + i];
                b = b + v(h + i) * p[i] - v(i) * p[h + i];
            }
            return 1.0 - (a * a + b * b);
        }
        case DTO_L_SPLIT_SQDIST: {  // norm(v[0:h] - v[h:2h])^2
            const int h = nv / 2;
            T s = T(0.0);
            for (int i = 0; i < h; ++i) {
                T d = v(i) - v(h + i);
                s = s + d * d;
            }
            return s;
        }
        default:
            return T(0.0);
    }
}

inline bool knot_cfun_known(int fn) { return fn >= DTO_G_NORM_MINUS_C && fn <= DTO_G_NORM_PRODUCT; }
inline bool knot_lfun_known(int fn) { return fn >= DTO_L_NORMSQ_PLUS_P && fn <= DTO_L_SPLIT_SQDIST; }

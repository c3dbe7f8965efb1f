// Device interpreter of knot programs: a user-written knot function g(v; p) / l(v; p) traced by the front end into an
// SSA tape and compiled at construction (dto_host.cu: compile_knot_program) into register-machine words
// {opcode, dst, a, b} over DTO_MAX_PROGRAM_SLOTS slots.  Instantiated with `double` (values) and the hyper-dual `HDual`
// (first and second derivatives in one pass), exactly like the catalogue of knotfun.cuh, so every call site of the
// catalogue -- values, Jacobians, Hessian pairs, the stored-pattern probe -- runs programs through the same code.
//
// Every thread of a launch runs the same term, so the word stream is warp-uniform: the loads are broadcasts and the
// dispatch does not diverge.  The interpreter is __noinline__: the kernels that call the catalogue keep the register
// allocation they were tuned with, and the slots live in the interpreter's own stack frame.
// Included by knotfun.cuh after HDual and the variable accessors.
#pragma once

__device__ inline double kp_val(double a) { return a; }
__device__ inline double kp_val(const HDual& a) { return a.v; }
// f(a) given f, f' and f'' at the value of a: the one chain rule every unary operation of the hyper-dual path goes through
__device__ inline double kp_chain(double, double f, double, double) { return f; }
__device__ inline HDual kp_chain(const HDual& a, double f, double f1, double f2) {
    return HDual(f, f1 * a.d1, f1 * a.d2, f1 * a.d12 + f2 * a.d1 * a.d2);
}
// a / b: a plain division for values, a times the hyper-dual reciprocal of b for derivatives
__device__ inline double kp_div(double a, double b) { return a / b; }
__device__ inline HDual kp_div(const HDual& a, const HDual& b) {
    const double r = 1.0 / b.v;
    return a * kp_chain(b, r, -r * r, 2.0 * r * r * r);
}

// x^c for a constant c: pow() is valid for negative bases when c is integer-valued; c = 2 is a product (exact)
__device__ inline double kp_pow(double x, double c) { return c == 2.0 ? x * x : pow(x, c); }

template <class T, class Vars>
__device__ __noinline__ void run_knot_program(const int4* __restrict__ code, int n_code, const Vars v, const double* p, T* out) {
    T s[DTO_MAX_PROGRAM_SLOTS];
    const double* consts = reinterpret_cast<const double*>(code + n_code);
    for (int i = 0; i < n_code; ++i) {
        const int4 w = __ldg(code + i);
        const int d = w.y;
        switch (w.x) {
            case DTO_OP_VAR: s[d] = v(w.z); break;
            case DTO_OP_PARAM: s[d] = T(p[w.z]); break;
            case DTO_OP_CONST: s[d] = T(__ldg(consts + w.z)); break;
            case DTO_OP_ADD: s[d] = s[w.z] + s[w.w]; break;
            case DTO_OP_SUB: s[d] = s[w.z] - s[w.w]; break;
            case DTO_OP_MUL: s[d] = s[w.z] * s[w.w]; break;
            case DTO_OP_DIV: s[d] = kp_div(s[w.z], s[w.w]); break;
            case DTO_OP_NEG: s[d] = -s[w.z]; break;
            case DTO_OP_SQRT: {
                const double x = kp_val(s[w.z]), r = sqrt(x);
                s[d] = kp_chain(s[w.z], r, 0.5 / r, -0.25 / (r * x));
            } break;
            case DTO_OP_EXP: {
                const double e = exp(kp_val(s[w.z]));
                s[d] = kp_chain(s[w.z], e, e, e);
            } break;
            case DTO_OP_LOG: {
                const double x = kp_val(s[w.z]), r = 1.0 / x;
                s[d] = kp_chain(s[w.z], log(x), r, -r * r);
            } break;
            case DTO_OP_SIN: {
                double sn, cs;
                sincos(kp_val(s[w.z]), &sn, &cs);
                s[d] = kp_chain(s[w.z], sn, cs, -sn);
            } break;
            case DTO_OP_COS: {
                double sn, cs;
                sincos(kp_val(s[w.z]), &sn, &cs);
                s[d] = kp_chain(s[w.z], cs, -sn, -cs);
            } break;
            case DTO_OP_TANH: {
                const double t = tanh(kp_val(s[w.z])), d1 = 1.0 - t * t;
                s[d] = kp_chain(s[w.z], t, d1, -2.0 * t * d1);
            } break;
            case DTO_OP_POWC: {
                const double x = kp_val(s[w.z]), c = __ldg(consts + w.w);
                const double d1 = c == 0.0 ? 0.0 : (c == 2.0 ? 2.0 * x : c * pow(x, c - 1.0));
                const double d2 = (c == 0.0 || c == 1.0) ? 0.0 : (c == 2.0 ? 2.0 : c * (c - 1.0) * pow(x, c - 2.0));
                s[d] = kp_chain(s[w.z], kp_pow(x, c), d1, d2);
            } break;
            case DTO_OP_OUT: out[d] = s[w.z]; break;
        }
    }
}

"""ctypes binding of libdto_b200.so (include/dto_b200.h).  Fails loudly when the CUDA library is
missing: there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# DTO_B200_LIB: another build of the same library (e.g. the instrumented one of tools/build_profile_lib.sh)
LIB_PATH = os.environ.get("DTO_B200_LIB") or os.path.join(HERE, "lib", "libdto_b200.so")

DTO_OK, DTO_ERR_INVALID, DTO_ERR_UNSUPPORTED, DTO_ERR_CUDA, DTO_ERR_ALLOC = 0, -1, -2, -3, -4
ABI_VERSION = 4

INT_BILINEAR, INT_DERIVATIVE, INT_TDBILINEAR = 1, 2, 3
OBJ_QUADREG, OBJ_MINTIME, OBJ_KNOT, OBJ_NULL, OBJ_LINREG, OBJ_GLOBAL_KNOT = 1, 2, 3, 4, 5, 6
G_FUNCS = {"norm_minus_c": 1, "normsq_minus_c": 2, "sqdist_minus_c": 3, "linear": 4, "norm_product": 5}
L_FUNCS = {"normsq_plus_p": 1, "sqdist": 2, "linear": 3, "iso_infidelity": 4, "split_sqdist": 5}
G_PROGRAM, L_PROGRAM = 100, 100  # knot programs (knot_program.py): the term's `program` indexes ProblemDesc.programs

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_int64_p = C.POINTER(C.c_int64)


class IntegratorDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("x_off", C.c_int32), ("x_dim", C.c_int32), ("u_off", C.c_int32), ("u_dim", C.c_int32),
        ("t_off", C.c_int32), ("spline_order", C.c_int32), ("n_carrier", C.c_int32),
        ("G", c_double_p), ("G_batch_stride", C.c_int64),
        ("A", c_double_p), ("B", c_double_p), ("omega", c_double_p), ("phi", c_double_p),
        ("D", c_double_p), ("omega_d", c_double_p), ("phi_d", c_double_p),
        ("tdb_steps", C.c_int32), ("_pad", C.c_int32),
    ]


class ObjectiveDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("fn", C.c_int32), ("weight", C.c_double), ("n_vars", C.c_int32), ("n_times", C.c_int32),
        ("var_offs", c_int32_p), ("times", c_int32_p), ("R", c_double_p), ("baseline", c_double_p), ("D", C.c_double),
        ("n_params", C.c_int32), ("program", C.c_int32), ("params", c_double_p), ("Qs", c_double_p),
        ("n_gvars", C.c_int32), ("_pad2", C.c_int32), ("gvar_offs", c_int32_p),
    ]


class ConstraintDesc(C.Structure):
    _fields_ = [
        ("fn", C.c_int32), ("equality", C.c_int32), ("n_vars", C.c_int32), ("n_times", C.c_int32),
        ("var_offs", c_int32_p), ("times", c_int32_p), ("g_dim", C.c_int32), ("n_params", C.c_int32), ("params", c_double_p),
        ("n_gvars", C.c_int32), ("program", C.c_int32), ("gvar_offs", c_int32_p),
    ]


class KnotProgramDesc(C.Structure):
    _fields_ = [
        ("n_ops", C.c_int32), ("n_out", C.c_int32), ("ops", c_int32_p), ("out", c_int32_p),
        ("n_consts", C.c_int32), ("_pad", C.c_int32), ("consts", c_double_p),
    ]


class ProblemDesc(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("N", C.c_int32), ("z", C.c_int32), ("dt_off", C.c_int32), ("batch", C.c_int32),
        ("eval_hessian", C.c_int32), ("shard_k0", C.c_int32), ("shard_k1", C.c_int32), ("device", C.c_int32),
        ("n_integrators", C.c_int32), ("n_objectives", C.c_int32), ("n_constraints", C.c_int32),
        ("integrators", C.POINTER(IntegratorDesc)), ("objectives", C.POINTER(ObjectiveDesc)),
        ("constraints", C.POINTER(ConstraintDesc)), ("Z0", c_double_p),
        ("global_dim", C.c_int32), ("n_programs", C.c_int32), ("programs", C.POINTER(KnotProgramDesc)),
    ]


class SizeInfo(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("n_vars", "n_dynamics_cons", "n_nonlinear_cons", "n_cons", "nnz_jac", "nnz_hess")]


class ShardLayout(C.Structure):
    _fields_ = [(n, C.c_int64) for n in ("z_begin", "z_end", "z_halo_end", "n_local_cons", "n_local_jac", "n_local_hess")]


# every symbol include/dto_b200.h declares: (name, restype, argtypes)
_H = C.c_void_p
SYMBOLS = [
    ("dto_abi_version", C.c_int, []),
    ("dto_create", C.c_int, [C.POINTER(ProblemDesc), C.POINTER(_H)]),
    ("dto_destroy", None, [_H]),
    ("dto_last_error", C.c_char_p, [_H]),
    ("dto_sizes", C.c_int, [_H, C.POINTER(SizeInfo)]),
    ("dto_stream", C.c_void_p, [_H]),
    ("dto_jac_structure", C.c_int, [_H, c_int64_p, c_int64_p]),
    ("dto_hess_structure", C.c_int, [_H, c_int64_p, c_int64_p]),
    ("dto_shard_info", C.c_int, [_H, C.POINTER(ShardLayout)]),
    ("dto_shard_maps", C.c_int, [_H, c_int64_p, c_int64_p, c_int64_p]),
    ("dto_constraint_bounds", C.c_int, [_H, c_double_p, c_double_p]),
    ("dto_eval_objective", C.c_int, [_H, C.c_void_p, C.c_void_p]),
    ("dto_eval_gradient", C.c_int, [_H, C.c_void_p, C.c_void_p]),
    ("dto_eval_constraint", C.c_int, [_H, C.c_void_p, C.c_void_p]),
    ("dto_eval_jacobian", C.c_int, [_H, C.c_void_p, C.c_void_p]),
    ("dto_eval_hessian", C.c_int, [_H, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]),
    ("dto_eval_jacobian_product", C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("dto_eval_jacobian_transpose_product", C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("dto_eval_all", C.c_int, [_H, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("dto_upload", C.c_int, [_H, C.c_void_p]),
    ("dto_cache_stats", C.c_int, [_H, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    ("dto_register_outputs", C.c_int, [_H, C.c_void_p, C.c_void_p]),
    ("dto_unregister_outputs", C.c_int, [_H]),
    ("dto_eval_all_dev", C.c_int, [_H, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("dto_violation_dev", C.c_int, [_H, C.c_void_p, C.c_void_p]),
    ("dto_synchronize", C.c_int, [_H]),
    ("dto_shard_export", C.c_int, [_H, C.c_void_p]),
    ("dto_shard_link", C.c_int, [_H, C.c_int, C.c_int, C.c_void_p]),
    ("dto_shard_link_local", C.c_int, [C.POINTER(_H), C.c_int]),
    ("dto_upload_dev", C.c_int, [_H, C.c_void_p]),
    ("dto_allreduce_scalars_dev", C.c_int, [_H, C.c_void_p, C.c_void_p]),
    ("dto_shard_scalars_dev", C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("dto_local_Z", C.c_void_p, [_H]),
    ("dto_launch_count", C.c_int64, [_H]),
    ("dto_last_download_bytes", C.c_int64, [_H]),
    ("dto_kernel_variant", C.c_char_p, [_H, C.c_int]),
    ("dto_kernel_timing", C.c_int, [_H, C.c_int]),
    ("dto_kernel_time_ms", C.c_int, [_H, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
]

_lib = None


class DtoError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libdto_b200 error {code}: {msg}")
        self.code = code


def load():
    """Load libdto_b200.so and bind every declared symbol.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
            "directtrajopt.jl_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    if lib.dto_abi_version() != ABI_VERSION:
        raise ImportError("libdto_b200.so ABI version mismatch; rebuild")
    _lib = lib
    return lib


def check(rc, handle=None):
    if rc != DTO_OK:
        msg = load().dto_last_error(handle)
        raise DtoError(rc, msg.decode() if msg else "")

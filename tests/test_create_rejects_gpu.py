"""Every rejection a problem descriptor can reach in dto_create: each cell starts from a small valid problem, introduces
one defect into the raw descriptor on its way to the library, and checks the return code and the whole message of
dto_last_error(NULL).  Knot-program tapes are checked in test_knot_program_gpu.py; device and allocation failures are
not provoked."""
import ctypes as C

import numpy as np
import pytest

import dto_b200 as dto
from dto_b200 import problem_templates as pt

pytestmark = pytest.mark.gpu

INV, UNS = dto._lib.DTO_ERR_INVALID, dto._lib.DTO_ERR_UNSUPPORTED


def _smem_optin():
    import torch

    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def _smem_msg(what, need):
    return f"{what} needs {need} bytes of shared memory per block, above the device's limit of {_smem_optin()} bytes"


def _generic_smem(n, m):
    """bilinear_generic.cu: generic_smem_bytes(n, m, want_jac = true, want_hess = true)"""
    ncol = 1 + m + m * (m + 1) // 2 + n + 1 + m
    return 8 * ((n | 1) * n + 3 * ncol * n + 3 * n)


def _std():
    return pt.standard_problem(N=6)


def _glob():
    return pt.global_problem(N=6)


def _carrier(n_drives=2, spline_order=0):
    return pt.carrier_problem(N=4, state_dim=8, n_drives=n_drives, spline_order=spline_order)


def _program_con():
    """the standard problem with a knot-program constraint that takes a parameter"""
    prob = _std()
    traj = prob.trajectory
    con = dto.NonlinearKnotPointConstraint(dto.KnotProgram(lambda v, p: [v[0] * p[0] - np.sin(v[1])], params=[2.0]), "u", traj,
                                           times=range(2, traj.N), equality=False)
    return dto.DirectTrajOptProblem(traj, prob.objective, prob.integrators, constraints=[con])


def _wide_knot():
    """a linear-spline time-dependent problem whose knot carries 110 more variables: 126 per knot, coupled to the
    neighbour, is beyond the Hessian assembler's shared memory"""
    base = _carrier(spline_order=1)
    t = base.trajectory
    comps = {name: t.data[t.components[name], :] for name in t.names}
    comps["w"] = np.random.default_rng(3).standard_normal((110, t.N))
    traj = dto.NamedTrajectory(comps, controls=("dt",), timestep="dt")
    ints = [dto.TimeDependentBilinearIntegrator(base.integrators[0].G, "x", "u", "t", traj, spline_order=1),
            dto.DerivativeIntegrator("u", "du", traj), dto.DerivativeIntegrator("du", "ddu", traj)]
    J = dto.QuadraticRegularizer("u", traj, 1.0) + dto.QuadraticRegularizer("w", traj, 0.5)
    return dto.DirectTrajOptProblem(traj, J, ints)


def _obj(d, kind, min_gvars=0):
    for i in range(d.n_objectives):
        o = d.objectives[i]
        if o.kind == kind and o.n_vars > 0 and (min_gvars == 0 or o.n_gvars >= min_gvars):
            return o
    raise AssertionError(f"no objective of kind {kind}")


def _con(d, min_gvars=0):
    for i in range(d.n_constraints):
        c = d.constraints[i]
        if c.n_vars > 0 and c.n_gvars >= min_gvars:
            return c
    raise AssertionError("no such constraint")


def _set(**fields):
    def edit(d):
        for k, v in fields.items():
            setattr(d, k, v)

    return edit


def _repeat(arr):  # second entry := first
    arr[1] = arr[0]


QUAD, KNOT, GKNOT = dto._lib.OBJ_QUADREG, dto._lib.OBJ_KNOT, dto._lib.OBJ_GLOBAL_KNOT

# id: (base problem, edit of the descriptor, return code, message or a function of nothing that gives it)
CELLS = {
    # header, shard range, shard batch, global_dim
    "abi_version": (_std, _set(abi_version=2), INV, "ABI version mismatch"),
    "program_table": (_std, _set(n_programs=-1), INV, "bad knot program table"),
    "N": (_std, _set(N=1), INV, "need N >= 2, z >= 1, batch >= 1"),
    "z": (_std, _set(z=0), INV, "need N >= 2, z >= 1, batch >= 1"),
    "batch": (_std, _set(batch=0), INV, "need N >= 2, z >= 1, batch >= 1"),
    "dt_off": (_std, lambda d: setattr(d, "dt_off", d.z), INV, "timestep component outside the knot"),
    "no_integrator": (_std, _set(n_integrators=0), UNS, "at least one integrator is required (dense block Hessian structure)"),
    "too_many_terms": (_std, _set(n_objectives=17), UNS, "too many integrators / objective terms / constraints"),
    "shard_range": (_std, _set(shard_k0=3, shard_k1=2), INV, "bad shard range"),
    "shard_past_N": (_std, _set(shard_k0=2, shard_k1=7), INV, "bad shard range"),
    "shard_batch": (_std, _set(shard_k0=1, shard_k1=3, batch=2), UNS, "knot-range shards require batch == 1"),
    "global_dim": (_std, _set(global_dim=1025), INV, "global_dim outside 0..1024"),
    "global_dim_negative": (_std, _set(global_dim=-1), INV, "global_dim outside 0..1024"),
    "shard_globals": (_glob, _set(shard_k0=1, shard_k1=3), UNS, "knot-range shards do not support global variables"),
    # integrators
    "int_state": (_std, lambda d: setattr(d.integrators[0], "x_off", d.z - 1), INV, "integrator state component outside the knot"),
    "int_kind": (_std, lambda d: setattr(d.integrators[0], "kind", 9), UNS, "unknown integrator kind"),
    "bilinear_generators": (_std, lambda d: setattr(d.integrators[0], "G", None), INV,
                            "bilinear integrator: bad drive component or missing generators"),
    "bilinear_drive": (_std, lambda d: setattr(d.integrators[0], "u_off", d.z - 1), INV,
                       "bilinear integrator: bad drive component or missing generators"),
    "bilinear_n97": (lambda: pt.scaled_problem(N=3, state_dim=100, n_controls=1, generator_scale=0.01), lambda d: None, UNS,
                     "bilinear integrator: state dimension > 96 not supported"),
    "bilinear_generic_smem": (lambda: pt.scaled_problem(N=3, state_dim=88, n_controls=4, generator_scale=1.0 / 88), lambda d: None, UNS,
                              lambda: _smem_msg("bilinear integrator: the generic kernel at state dimension 88 with 4 drives and the Hessian",
                                                _generic_smem(88, 4))),
    "derivative_dim": (_std, lambda d: setattr(d.integrators[1], "u_dim", d.integrators[1].x_dim + 1), INV,
                       "derivative integrator: derivative component must match the variable's dimension"),
    "tdb_components": (_carrier, lambda d: setattr(d.integrators[0], "t_off", -1), INV, "tdbilinear integrator: bad components"),
    "tdb_spline_order": (_carrier, lambda d: setattr(d.integrators[0], "spline_order", 2), UNS, "Unsupported spline order"),
    "tdb_fits": (lambda: _carrier(n_drives=5), lambda d: None, UNS,
                 lambda: "tdbilinear integrator: more than 4 drives or 4 carriers, or a state too large for the device's "
                         f"{_smem_optin()} bytes of shared memory per block"),
    # objectives
    "obj_kind": (_std, lambda d: setattr(_obj(d, QUAD), "kind", 99), UNS, "unknown objective kind"),
    "obj_catalogue": (_std, lambda d: setattr(_obj(d, KNOT), "fn", 999), UNS, "knot objective function is not in the device catalogue"),
    "obj_var_list": (_std, lambda d: setattr(_obj(d, KNOT), "n_vars", 0), INV, "objective: bad variable list"),
    "obj_var_list_null": (_std, lambda d: setattr(_obj(d, QUAD), "var_offs", None), INV, "objective: bad variable list"),
    "obj_global_list": (_glob, lambda d: setattr(_obj(d, GKNOT, 2), "n_gvars", 0), INV, "global objective: missing global variable list"),
    "obj_global_range": (_glob, lambda d: _obj(d, GKNOT, 2).gvar_offs.__setitem__(0, d.global_dim), INV,
                         "global objective: variable outside global_data"),
    "obj_global_repeat": (_glob, lambda d: _repeat(_obj(d, GKNOT, 2).gvar_offs), UNS, "global objective: repeated global variable"),
    "obj_var_range": (_std, lambda d: _obj(d, KNOT).var_offs.__setitem__(0, d.z), INV, "objective: variable outside the knot"),
    "obj_var_repeat": (_std, lambda d: _repeat(_obj(d, QUAD).var_offs), UNS, "objective: repeated variable"),
    "obj_time_range": (_std, lambda d: _obj(d, QUAD).times.__setitem__(0, d.N + 1), INV, "objective: time index outside 1..N"),
    "obj_time_repeat": (_std, lambda d: _repeat(_obj(d, QUAD).times), UNS, "objective: repeated time index"),
    "reg_R": (_std, lambda d: setattr(_obj(d, QUAD), "R", None), INV, "regularizer: missing R"),
    "reg_dt": (_std, lambda d: _obj(d, QUAD).var_offs.__setitem__(0, d.dt_off), UNS,
               "regularizer on the timestep component itself is not supported"),
    "obj_Qs": (_std, lambda d: setattr(_obj(d, KNOT), "Qs", None), INV, "knot objective: missing Qs/params"),
    # Hessian assembler
    "wide_knot": (_wide_knot, lambda d: None, UNS,
                  lambda: _smem_msg("Hessian assembly of a knot of 126 variables coupled to its neighbour", 8 * 126 * 126 * 2)),
    # constraints
    "con_catalogue": (_std, lambda d: setattr(_con(d), "fn", 999), UNS, "knot constraint function is not in the device catalogue"),
    "con_var_list": (_std, lambda d: setattr(_con(d), "n_vars", 0), INV, "constraint: bad variable list or g_dim"),
    "con_g_dim_zero": (_std, lambda d: setattr(_con(d), "g_dim", 0), INV, "constraint: bad variable list or g_dim"),
    "con_g_dim": (_std, lambda d: setattr(_con(d), "g_dim", 2), INV, "constraint: g_dim must be 1 for this function"),
    "con_norm_product": (_glob, lambda d: setattr(_con(d, 1), "n_params", 2), INV, "constraint: norm_product has g_dim 2 and 3 parameters"),
    "con_global_range": (_glob, lambda d: _con(d, 1).gvar_offs.__setitem__(0, d.global_dim), INV, "constraint: variable outside global_data"),
    "con_global_repeat": (_glob, lambda d: _repeat(_con(d, 2).gvar_offs), UNS, "constraint: repeated global variable"),
    "con_Z0": (_std, _set(Z0=None), INV, "knot constraints need the initial trajectory Z0 (stored Jacobian pattern)"),
    "con_var_range": (_std, lambda d: _con(d).var_offs.__setitem__(0, d.z), INV, "constraint: variable outside the knot"),
    "con_var_repeat": (_std, lambda d: _repeat(_con(d).var_offs), UNS, "constraint: repeated variable"),
    "con_time_range": (_std, lambda d: _con(d).times.__setitem__(0, 0), INV, "constraint: time index outside 1..N"),
    "con_time_repeat": (_std, lambda d: _repeat(_con(d).times), UNS, "constraint: repeated time index"),
    "con_params": (_program_con, lambda d: setattr(_con(d), "params", None), INV, "constraint: missing params"),
}


@pytest.mark.parametrize("cell", list(CELLS))
def test_one_defect_is_rejected(cell, monkeypatch):
    base, edit, code, msg = CELLS[cell]
    prob = base()
    real = dto._lib.load()
    seen = {}

    class Lib:
        def __getattr__(self, name):
            return getattr(real, name)

        def dto_create(self, desc, out):
            edit(desc._obj)  # the ProblemDesc behind byref()
            rc = real.dto_create(desc, out)
            seen["rc"], seen["msg"] = rc, real.dto_last_error(None).decode()
            return rc

    monkeypatch.setattr(dto._lib, "load", lambda: Lib())
    with pytest.raises((dto.DtoError, dto.UnsupportedComponent)):
        dto.Evaluator(prob)
    assert seen["rc"] == code
    assert seen["msg"] == (msg() if callable(msg) else msg)


def test_valid_bases_are_accepted():
    """the cells' starting points are valid problems: every rejection above comes from its one defect"""
    for base in (_std, _glob, _carrier, _program_con):
        dto.Evaluator(base()).close()


def test_null_descriptor():
    lib = dto._lib.load()
    h = C.c_void_p()
    assert lib.dto_create(None, C.byref(h)) == INV
    assert lib.dto_last_error(None).decode() == "null descriptor"

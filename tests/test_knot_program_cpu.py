"""KnotProgram on the CPU: the tracer records what f computes, refuses what a device program cannot express, the
second-order jets that give the oracle's reference for a user function are right, and the ctypes mirror of the new descriptors matches the C header."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import dto_b200 as dto
import dto_oracle as orc
from dto_b200 import knot_program as kp
from dto_b200 import problem_templates as pt
from helpers.jets import jets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def every_op(v, p):
    """uses every opcode, parameters and constants; three outputs"""
    a = v[0] * v[1] + np.sin(v[2]) / p[0] - np.exp(0.3 * v[3])
    b = np.sqrt(v @ v + 1.0) * np.cos(v[4]) - np.log(2.0 + v[1] ** 2) + np.tanh(v[0] - v[5])
    c = -(v[2] ** 3) + (v[3] + 3.0 - p[1]) ** -1.5 + 1.0 / (3.0 + v[4] ** 2) + (v[5] + 4.0) ** 0.5 + p[1] * v[0] ** 4
    return [a, b, c]


def test_tape_replays_f():
    rng = np.random.default_rng(0)
    per_time = rng.uniform(1.0, 2.0, (3, 2))
    prog = dto.KnotProgram(every_op, per_time=per_time)
    tape = prog.trace(6)
    assert tape.out.size == 3 and prog.g_dim(6) == 3
    ops = set(tape.ops[:, 0].tolist())
    assert ops == set(range(kp.OP_VAR, kp.OP_POWC + 1))
    for t in range(3):
        p = prog.param_table(3)[t]
        for _ in range(5):
            v = rng.uniform(-1.0, 1.0, 6)
            np.testing.assert_allclose(tape.replay(v, p), np.array(every_op(v, p), float), rtol=1e-15, atol=1e-15)


def test_operands_precede_their_uses():
    tape = dto.KnotProgram(every_op, params=[1.5, 0.5]).trace(6)
    for i, (op, a, b) in enumerate(tape.ops):
        if op >= kp.OP_ADD:
            assert 0 <= a < i
        if kp.OP_ADD <= op <= kp.OP_DIV:
            assert 0 <= b < i


def test_common_subexpressions_are_shared():
    tape = dto.KnotProgram(lambda v: [v[0] * v[1] + v[0] * v[1], np.sin(v[0] * v[1])]).trace(2)
    muls = [o for o in tape.ops if o[0] == kp.OP_MUL]
    assert len(muls) == 1
    assert sum(1 for o in tape.ops if o[0] == kp.OP_VAR) == 2


def test_sum_and_matmul_trace():
    tape = dto.KnotProgram(lambda v: [sum(v * v), v @ v, np.sum(v)]).trace(4)
    v = np.array([0.5, -1.0, 2.0, 3.0])
    np.testing.assert_allclose(tape.replay(v), [v @ v, v @ v, v.sum()], rtol=1e-15)


@pytest.mark.parametrize("f", [
    lambda v: [v[0] if v[1] > 0 else v[2]],     # comparison
    lambda v: [v[0] if v[1] else v[2]],         # truth value
    lambda v: [v[0] ** v[1]],                   # traced exponent
    lambda v: [2.0 ** v[0]],                    # traced exponent, reflected
    lambda v: [np.arctan(v[0])],                # other ufunc on a scalar tracer
    lambda v: list(np.arctan(v)),               # other ufunc on an object array
    lambda v: [abs(v[0])],                      # not smooth
    lambda v: [np.abs(v[0])],
    lambda v: [max(v[0], v[1])],
    lambda v: [float(v[0])],
], ids=["compare", "bool", "pow", "rpow", "arctan", "arctan_array", "abs", "np_abs", "max", "float"])
def test_rejections(f):
    with pytest.raises(dto.UnsupportedComponent):
        dto.KnotProgram(f).trace(3)


def test_constructors_accept_programs_and_refuse_bare_callables():
    G, traj = pt.bilinear_dynamics_and_trajectory(N=5)
    nx = traj.dims["x"]
    prog = dto.KnotProgram(lambda v: [v[0] - v[nx] ** 2])
    c = dto.NonlinearKnotPointConstraint(prog, ["x", "u"], traj)
    assert c.g_dim == 1 and c.dim == traj.N and c.to_spec(traj)["fn"] is prog
    with pytest.raises(dto.UnsupportedComponent):
        dto.NonlinearKnotPointConstraint(lambda v: [v[0]], "u", traj)
    with pytest.raises(dto.UnsupportedComponent):
        dto.KnotPointObjective(dto.KnotProgram(lambda v: [v[0], v[1]]), "u", traj)
    with pytest.raises(dto.UnsupportedComponent):
        dto.TerminalObjective(dto.KnotProgram(lambda v: v[:2]), "x", traj)
    o = dto.TerminalObjective(dto.KnotProgram(lambda v: v @ v), "x", traj)
    assert o.to_spec(traj)["fn"].g_dim(nx) == 1


# ---- reference derivatives: jets of a user function ---------------------------------------------------------------------------------
def test_jets_match_central_differences():
    rng = np.random.default_rng(1)
    p = np.array([1.3, 0.7])
    f = lambda v: np.array(every_op(v, p), float)
    for _ in range(3):
        v = rng.uniform(-0.8, 0.8, 6)
        val, J, H = jets(every_op, v, p)
        np.testing.assert_allclose(val, f(v), rtol=1e-15)
        h = 1e-6
        Jfd = np.stack([(f(v + h * e) - f(v - h * e)) / (2 * h) for e in np.eye(6)], axis=1)
        assert np.abs(J - Jfd).max() <= 1e-8 * max(1.0, np.abs(J).max())
        jac = lambda x: jets(every_op, x, p)[1]
        Hfd = np.stack([(jac(v + h * e) - jac(v - h * e)) / (2 * h) for e in np.eye(6)], axis=2)
        assert np.abs(H - Hfd).max() <= 1e-7 * max(1.0, np.abs(H).max())
        assert np.array_equal(H, H.transpose(0, 2, 1))


def _catalogue_pairs(rng, nv):
    h = nv // 2
    A, b = rng.standard_normal((2, nv)), rng.standard_normal(2)
    c = [  # (catalogue name, parameters, the same function written as a user would)
        ("norm_minus_c", [0.8], lambda v, p: [np.sqrt(v @ v) - p[0]]),
        ("normsq_minus_c", [0.5], lambda v, p: [v @ v - p[0]]),
        ("sqdist_minus_c", np.r_[0.1, rng.standard_normal(nv)], lambda v, p: [(v - p[1:]) @ (v - p[1:]) - p[0]]),
        ("linear", np.r_[2, A.reshape(-1, order="F"), b], lambda v, p: A @ v - b),
        ("norm_product", [1.0, 0.5, 3], lambda v, p: [np.sqrt(v[:3] @ v[:3]) - p[0],
                                                      np.sqrt(v[:3] @ v[:3]) * np.sqrt(v[3:] @ v[3:]) - p[1]]),
    ]
    l = [
        ("normsq_plus_p", [0.3], lambda v, p: v @ v + p[0]),
        ("sqdist", rng.standard_normal(nv), lambda v, p: (v - p) @ (v - p)),
        ("linear", rng.standard_normal(nv), lambda v, p: p @ v),
        ("iso_infidelity", rng.standard_normal(nv), lambda v, p: 1.0 - ((v[:h] @ p[:h] + v[h:] @ p[h:]) ** 2
                                                                     + (v[h:] @ p[:h] - v[:h] @ p[h:]) ** 2)),
        ("split_sqdist", [0.0], lambda v, p: (v[:h] - v[h:]) @ (v[:h] - v[h:])),
    ]
    return c, l


def test_jets_reproduce_catalogue_closed_forms():
    rng = np.random.default_rng(2)
    nv = 8
    cons, objs = _catalogue_pairs(rng, nv)
    for _ in range(3):
        v = rng.standard_normal(nv)
        for name, p, f in cons:
            p = np.asarray(p, float)
            for x, y in zip(jets(f, v, p), orc._cfun(name, v, p)):
                assert np.abs(x - y).max() <= 1e-13 * max(1.0, np.abs(y).max()), name
        for name, p, f in objs:
            p = np.asarray(p, float)
            for x, y in zip((a[0] for a in jets(f, v, p)), orc._lfun(name, v, p)):
                assert np.abs(np.asarray(x) - y).max() <= 1e-13 * max(1.0, np.abs(y).max()), name


# ---- ctypes layout of the ABI-4 descriptors --------------------------------------------------------------------------
def test_program_struct_layout_matches_header(tmp_path):
    L = dto._lib
    fields = [("dto_knot_program", "n_ops"), ("dto_knot_program", "n_out"), ("dto_knot_program", "ops"), ("dto_knot_program", "out"),
              ("dto_knot_program", "n_consts"), ("dto_knot_program", "consts"), ("dto_problem_desc", "global_dim"),
              ("dto_problem_desc", "n_programs"), ("dto_problem_desc", "programs"), ("dto_objective_desc", "program"),
              ("dto_constraint_desc", "program")]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dto_b200.h"\nint main(void) {\n'
                   + "".join(f'    printf("%zu\\n", offsetof({s}, {f}));\n' for s, f in fields)
                   + '    printf("%zu\\n%zu\\n%d\\n", sizeof(dto_knot_program), sizeof(dto_problem_desc), DTO_B200_ABI_VERSION);\n'
                   + "    return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    cls = {"dto_knot_program": L.KnotProgramDesc, "dto_problem_desc": L.ProblemDesc, "dto_objective_desc": L.ObjectiveDesc,
           "dto_constraint_desc": L.ConstraintDesc}
    want = [getattr(cls[s], f).offset for s, f in fields] + [ctypes.sizeof(L.KnotProgramDesc), ctypes.sizeof(L.ProblemDesc), L.ABI_VERSION]
    assert got == want


def test_opcodes_match_header():
    header = open(os.path.join(ROOT, "include", "dto_b200.h")).read()
    for name in ("VAR", "PARAM", "CONST", "ADD", "SUB", "MUL", "DIV", "NEG", "SQRT", "EXP", "LOG", "SIN", "COS", "TANH", "POWC"):
        assert f"DTO_OP_{name} = {getattr(kp, 'OP_' + name)}" in header
    assert f"DTO_G_PROGRAM = {dto._lib.G_PROGRAM}" in header and f"DTO_L_PROGRAM = {dto._lib.L_PROGRAM}" in header

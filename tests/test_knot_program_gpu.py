"""KnotProgram terms on the device: parity with the CPU oracle (which takes a KnotProgram term's reference from
second-order jets of the user's own function, helpers/jets.py), equivalence with the catalogue, batches, knot-range
shards, the host-pointer callbacks, and the construction-time refusal of malformed or oversized programs."""
import ctypes as C

import numpy as np
import pytest

import dto_b200 as dto
import dto_oracle as orc
from dto_b200 import problem_templates as pt
from helpers import blocks
from helpers.jets import with_user_functions

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def oracle_user_functions(monkeypatch):
    """the oracle evaluates KnotProgram terms by second-order jets of the user's own function (helpers/jets.py)"""
    with_user_functions(monkeypatch, orc)

TOL = 1e-10


def relerr(got, ref):
    scale = max(np.abs(ref).max() if ref.size else 0.0, 1e-300)
    return np.abs(got - ref).max() / scale if ref.size else 0.0


def mixed(v, p):
    """g_dim = 3, every operation, per-time parameters"""
    a = v[0] * v[1] + np.sin(v[2]) / p[0] - np.exp(0.3 * v[3])
    b = np.sqrt(v @ v + 1.0) * np.cos(v[4]) - np.log(2.0 + v[1] ** 2) + np.tanh(v[0] - v[5])
    c = -(v[2] ** 3) + (v[3] + 3.0 - p[1]) ** -1.5 + 1.0 / (3.0 + v[4] ** 2) + p[1] * v[0] ** 4 - v[5] / (2.0 + v[1] ** 2)
    return [a, b, c]


def docstring_problem(N=8):
    """x[1] - u[1]^2 (knot_point_constraint.jl:71) on [x; u]; u[1] = 0 at knots 2 and 5 of Z0, so that the u entry is
    dropped from the stored pattern there; plus a g_dim = 3 equality and inequality mixing every operation."""
    G, traj = pt.bilinear_dynamics_and_trajectory(N=N, seed=1)
    traj.data[traj.components["u"][0], [1, 4]] = 0.0
    nx = traj.dims["x"]
    ints = [dto.BilinearIntegrator(G, "x", "u", traj), dto.DerivativeIntegrator("u", "du", traj),
            dto.DerivativeIntegrator("du", "ddu", traj)]
    J = dto.QuadraticRegularizer("u", traj, 1.0) + dto.MinimumTimeObjective(traj)
    rng = np.random.default_rng(5)
    cons = [
        dto.NonlinearKnotPointConstraint(dto.KnotProgram(lambda v: [v[0] - v[nx] ** 2]), ["x", "u"], traj),
        dto.NonlinearKnotPointConstraint(dto.KnotProgram(mixed, per_time=rng.uniform(1, 2, (3, 2))), ["x", "u"], traj,
                                         times=[1, 3, N], equality=True),
        dto.NonlinearKnotPointConstraint(dto.KnotProgram(mixed, params=[1.5, 0.4]), ["u", "x"], traj, times=range(2, N), equality=False),
    ]
    return dto.DirectTrajOptProblem(traj, J, ints, constraints=cons)


def gate_problem(N=6):
    """n = 32 gate problem: a per-time-parameter KnotPointObjective and a TerminalObjective infidelity as programs
    (528 Hessian pairs per knot)."""
    prob = pt.quantum_gate_problem(N=N, levels=16, n_drives=4)
    traj = prob.trajectory
    n = traj.dims["x"]
    h = n // 2
    goal = np.zeros(n)
    goal[1] = 1.0
    infid = dto.KnotProgram(lambda v, p: 1.0 - ((v[:h] @ p[:h] + v[h:] @ p[h:]) ** 2 + (v[h:] @ p[:h] - v[:h] @ p[h:]) ** 2), params=goal)
    rng = np.random.default_rng(3)
    smooth = dto.KnotProgram(lambda v, p: p[0] * (v @ v) + np.cos(p[1] * v[0]) * v[3] ** 2, per_time=rng.uniform(0.5, 1.5, (3, 2)))
    J = prob.objective + dto.TerminalObjective(infid, "x", traj, Q=2.0) + dto.KnotPointObjective(smooth, ["u", "x"], traj, times=[1, 3, N])
    return dto.DirectTrajOptProblem(traj, J, prob.integrators)


def global_program_problem(N=9):
    """pt.global_problem with its four global terms written as programs"""
    base = pt.global_problem(N=N)
    traj = base.trajectory
    J = dto.QuadraticRegularizer("u", traj, 1.0) + dto.MinimumTimeObjective(traj)
    J = J + dto.GlobalObjective(dto.KnotProgram(lambda v: v @ v + np.sin(v[0])), "g", traj, Q=2.0)
    J = J + 0.5 * dto.GlobalKnotPointObjective(dto.KnotProgram(lambda v: v @ v * np.exp(0.1 * v[-1])), ["u"], ["g"], traj,
                                               times=[1, N], Qs=[1.0, 2.0])
    J = J + dto.TerminalObjective(dto.KnotProgram(lambda v: (v[:4] - v[4:]) @ (v[:4] - v[4:])), "x", traj, global_names="x_goal", Q=100.0)
    cons = [
        dto.NonlinearKnotPointConstraint(dto.KnotProgram(lambda v: [np.sqrt(v @ v) - 1.0]), "u", traj, times=range(2, N), equality=False),
        dto.NonlinearGlobalKnotPointConstraint(dto.KnotProgram(lambda v: [np.sqrt(v[:2] @ v[:2]) - 1.0,
                                                                        np.sqrt(v[:2] @ v[:2]) * np.sqrt(v[2:] @ v[2:]) - 1.0]),
                                               ["u"], ["g"], traj, equality=False),
        dto.NonlinearGlobalConstraint(dto.KnotProgram(lambda v: [v @ v - 1.0, np.tanh(v[0]) * v[-1]]), "g", traj, equality=False),
    ]
    return dto.DirectTrajOptProblem(traj, J, base.integrators, constraints=cons)


PROBLEMS = {"docstring": docstring_problem, "gate_n32": gate_problem, "global": global_program_problem}


@pytest.fixture(scope="module", params=list(PROBLEMS))
def case(request):
    prob = PROBLEMS[request.param]()
    ev = dto.Evaluator(prob)
    yield request.param, prob, ev
    ev.close()


def test_structures_match_oracle(case):
    name, prob, ev = case
    spec, Z = prob.to_spec(), prob.trajectory.vec()
    jr, jc = ev.jacobian_structure()
    orow, ocol = orc.jacobian_structure(spec, Z)
    assert np.array_equal(jr, orow) and np.array_equal(jc, ocol)
    hr, hc = ev.hessian_lagrangian_structure()
    orow, ocol = orc.hessian_structure(spec, Z)
    assert np.array_equal(hr, orow) and np.array_equal(hc, ocol)


def test_values_match_oracle(case):
    name, prob, ev = case
    spec = prob.to_spec()
    rng = np.random.default_rng(7)
    Z0 = prob.trajectory.vec()
    Z = Z0 + 0.05 * rng.standard_normal(Z0.size)
    dts = slice(spec["components"][spec["timestep"]][0], spec["N"] * spec["z"], spec["z"])
    Z[dts] = np.abs(Z[dts])
    jst, hst = orc.jacobian_structure(spec, Z0), orc.hessian_structure(spec, Z0)
    mu = rng.random(ev.n_constraints)
    assert abs(ev.eval_objective(Z) - orc.eval_objective(spec, Z)) <= TOL * max(1.0, abs(orc.eval_objective(spec, Z)))
    grad = np.full(ev.n_vars, np.nan)
    ev.eval_objective_gradient(grad, Z)
    assert relerr(grad, orc.eval_objective_gradient(spec, Z)) <= TOL
    g = np.full(ev.n_constraints, np.nan)
    ev.eval_constraint(g, Z)
    gref = orc.eval_constraint(spec, Z)
    assert relerr(g, gref) <= TOL and blocks.vec_block_relerr(spec, g, gref) <= TOL
    J = np.full(ev.nnz_jacobian, np.nan)
    ev.eval_constraint_jacobian(J, Z)
    Jref = orc.eval_constraint_jacobian(spec, Z, jst)
    assert relerr(J, Jref) <= TOL and blocks.jac_block_relerr(spec, jst, J, Jref) <= TOL
    for sigma in (2.0, 0.0):
        H = np.full(ev.nnz_hessian, np.nan)
        ev.eval_hessian_lagrangian(H, Z, sigma, mu)
        Href = orc.eval_hessian_lagrangian(spec, Z, sigma, mu, hst)
        assert relerr(H, Href) <= TOL and blocks.hess_block_relerr(spec, hst, H, Href) <= TOL


def test_docstring_entry_dropped_from_pattern():
    prob = docstring_problem()
    ev = dto.Evaluator(prob)
    traj = prob.trajectory
    rows, cols = ev.jacobian_structure()
    row0 = ev.n_dynamics_constraints  # first row of the docstring constraint: one row per knot
    u0 = traj.components["u"][0]
    for k in range(1, traj.N + 1):
        stored = set(cols[rows == row0 + k].tolist())
        assert ((k - 1) * traj.dim + u0 + 1 in stored) == (k not in (2, 5))
        assert (k - 1) * traj.dim + traj.components["x"][0] + 1 in stored
    ev.close()


# ---- the catalogue, written as programs ---------------------------------------------------------------------------------
def _as_program(fn, params):
    """the KnotProgram equal to catalogue entry `fn` with parameter table `params`"""
    name = fn.name
    forms = {
        "norm_minus_c": lambda v, p: [np.sqrt(v @ v) - p[0]],
        "normsq_minus_c": lambda v, p: [v @ v - p[0]],
        "sqdist_minus_c": lambda v, p: [(v - p[1:]) @ (v - p[1:]) - p[0]],
        "normsq_plus_p": lambda v, p: v @ v + p[0],
        "sqdist": lambda v, p: (v - p) @ (v - p),
        "iso_infidelity": lambda v, p: 1.0 - ((v[: v.size // 2] @ p[: v.size // 2] + v[v.size // 2:] @ p[v.size // 2:]) ** 2
                                              + (v[v.size // 2:] @ p[: v.size // 2] - v[: v.size // 2] @ p[v.size // 2:]) ** 2),
        "split_sqdist": lambda v, p: (v[: v.size // 2] - v[v.size // 2:]) @ (v[: v.size // 2] - v[v.size // 2:]),
    }
    return dto.KnotProgram(forms[name], per_time=params)


def _linear_program(params, gd, nv):
    A = params[0][1:1 + gd * nv].reshape(nv, gd).T
    b = params[0][1 + gd * nv:1 + gd * nv + gd]
    return dto.KnotProgram(lambda v: A @ v - b)


def program_twin(prob):
    """`prob` with every catalogue knot function replaced by the equal KnotProgram"""
    traj = prob.trajectory
    terms = []
    for ob, w in prob.objective_terms():
        if isinstance(ob, dto.KnotPointObjective):
            f = dto.KnotProgram(lambda v, p: p @ v, per_time=ob.params) if ob.l.name == "linear" else _as_program(ob.l, ob.params)
            ob = dto.KnotPointObjective(f, ob.var_names, traj, times=ob.times, Qs=ob.Qs)
        terms.append((ob, w))
    J = dto.CompositeObjective([o for o, _ in terms], [w for _, w in terms])
    cons = []
    for c in prob.nonlinear_constraints():
        if c.g.name == "linear":
            f = _linear_program(c.params, c.g_dim, c.var_dim)
        else:
            f = _as_program(c.g, c.params)
        cons.append(dto.NonlinearKnotPointConstraint(f, c.var_names, traj, times=c.times, equality=c.equality))
    return dto.DirectTrajOptProblem(traj, J, prob.integrators, constraints=cons)


def all_outputs(ev, Z, sigma, mu):
    n_grad = ev.shard_layout.z_end - ev.shard_layout.z_begin + ev.global_dim
    J, grad = np.empty(ev.batch), np.empty(ev.batch * n_grad)
    g, jac, hess = np.empty(ev.batch * ev.n_constraints), np.empty(ev.batch * ev.nnz_jacobian), np.empty(ev.batch * ev.nnz_hessian)
    ev.eval_all(Z, sigma, mu, J, grad, g, jac, hess)
    return J, grad, g, jac, hess


def test_catalogue_as_programs_matches_catalogue():
    from test_parity_gpu import catalogue_problem

    cat = catalogue_problem()
    twin = program_twin(cat)
    evc, evp = dto.Evaluator(cat), dto.Evaluator(twin)
    assert all(isinstance(c.g, dto.KnotProgram) for c in twin.nonlinear_constraints())
    for a, b in zip(evc.jacobian_structure() + evc.hessian_lagrangian_structure(), evp.jacobian_structure() + evp.hessian_lagrangian_structure()):
        assert np.array_equal(a, b)
    rng = np.random.default_rng(9)
    Z = cat.trajectory.vec() + 0.05 * rng.standard_normal(evc.n_vars)
    mu = rng.random(evc.n_constraints)
    for x, y in zip(all_outputs(evc, Z, 1.3, mu), all_outputs(evp, Z, 1.3, mu)):
        assert np.abs(x - y).max() <= 1e-13 * max(1.0, np.abs(x).max())
    evc.close()
    evp.close()


# ---- batches and knot-range shards --------------------------------------------------------------------------------------
def test_batch_is_bit_identical_to_single_problems():
    prob = docstring_problem()
    B = 3
    rng = np.random.default_rng(2)
    single, batched = dto.Evaluator(prob), dto.Evaluator(prob, batch=B)
    Z0 = prob.trajectory.vec()
    Zs = [Z0 + 0.03 * rng.standard_normal(Z0.size) for _ in range(B)]
    mus = [rng.random(single.n_constraints) for _ in range(B)]
    outb = all_outputs(batched, np.concatenate(Zs), 0.9, np.concatenate(mus))
    for b in range(B):
        for x, y in zip(all_outputs(single, Zs[b], 0.9, mus[b]), outb):
            n = x.size
            assert np.array_equal(x, y[b * n:(b + 1) * n])
    single.close()
    batched.close()


def _shard_problem(N=11):
    """docstring constraint + a program objective at several knots + a terminal program, no globals (shardable)"""
    prob = docstring_problem(N=N)
    traj = prob.trajectory
    J = prob.objective + dto.KnotPointObjective(dto.KnotProgram(lambda v: np.exp(0.2 * v[0]) * (v @ v)), ["u", "du"], traj, times=[2, 6, 7, N])
    J = J + dto.TerminalObjective(dto.KnotProgram(lambda v: (v @ v - 1.0) ** 2), "x", traj)
    return dto.DirectTrajOptProblem(traj, J, prob.integrators, constraints=prob.constraints)


@pytest.mark.parametrize("peer_halo", [False, True])
def test_knot_range_shards_reassemble_the_whole_problem(peer_halo):
    prob = _shard_problem()
    cuts = [(1, 4), (5, 7), (8, 11)]
    rng = np.random.default_rng(4)
    whole = dto.Evaluator(prob)
    Z0 = prob.trajectory.datavec
    Z = Z0 + 0.02 * rng.standard_normal(Z0.size)
    mu = rng.random(whole.n_constraints)
    Jw, gradw, gw, jacw, hessw = all_outputs(whole, Z, 0.7, mu)
    shards = [dto.Evaluator(prob, shard=c) for c in cuts]
    if peer_halo:
        dto.Evaluator.shard_link_local(shards)

    def local_Z(sh):
        L = sh.shard_layout
        Zl = Z[L.z_begin:L.z_halo_end].copy()
        if peer_halo and L.z_halo_end > L.z_end:
            Zl[L.z_end - L.z_begin:] = np.nan  # must come from the neighbour's window
        return Zl

    for sh in shards:
        sh.upload(local_Z(sh))
    J = 0.0
    grad, g, jac, hess = (np.full_like(a, np.nan) for a in (gradw, gw, jacw, hessw))
    for sh in shards:
        L = sh.shard_layout
        rows, jpos, hpos = sh.shard_maps()
        out = all_outputs(sh, local_Z(sh), 0.7, mu[rows])
        J += out[0][0]
        grad[L.z_begin:L.z_end] = out[1]
        g[rows], jac[jpos], hess[hpos] = out[2], out[3], out[4]
    assert np.array_equal(grad, gradw) and np.array_equal(g, gw) and np.array_equal(jac, jacw) and np.array_equal(hess, hessw)
    assert abs(J - Jw[0]) <= 1e-13 * max(1.0, abs(Jw[0]))
    for e in shards + [whole]:
        e.close()


# ---- host-pointer callbacks ---------------------------------------------------------------------------------------------
def test_callbacks_equal_eval_all():
    """the five callbacks in the order Ipopt calls them (objective first: early start on a new iterate) against one fused
    pass on another handle, bit for bit; Jacobian products against the materialised Jacobian"""
    prob = _shard_problem()
    ev, ref = dto.Evaluator(prob), dto.Evaluator(prob)
    rng = np.random.default_rng(6)
    for _ in range(3):
        Z = prob.trajectory.vec() + 0.02 * rng.standard_normal(ev.n_vars)
        mu = rng.random(ev.n_constraints)
        Jf, gradf, gf, jacf, hessf = all_outputs(ref, Z, 1.1, mu)
        assert ev.eval_objective(Z) == Jf[0]
        grad, g, jac, hess = np.empty_like(gradf), np.empty_like(gf), np.empty_like(jacf), np.empty_like(hessf)
        ev.eval_objective_gradient(grad, Z)
        ev.eval_constraint(g, Z)
        ev.eval_constraint_jacobian(jac, Z)
        ev.eval_hessian_lagrangian(hess, Z, 1.1, mu)
        assert np.array_equal(grad, gradf) and np.array_equal(g, gf) and np.array_equal(jac, jacf) and np.array_equal(hess, hessf)
    rows, cols = ev.jacobian_structure()
    Jd = np.zeros((ev.n_constraints, ev.n_vars))
    np.add.at(Jd, (rows - 1, cols - 1), jacf)
    w = rng.standard_normal(ev.n_vars)
    y = np.empty(ev.n_constraints)
    ev.eval_constraint_jacobian_product(y, Z, w)
    assert np.allclose(y, Jd @ w, rtol=0, atol=1e-12 * max(1.0, np.abs(Jd @ w).max()))
    w = rng.standard_normal(ev.n_constraints)
    y = np.empty(ev.n_vars)
    ev.eval_constraint_jacobian_transpose_product(y, Z, w)
    assert np.allclose(y, Jd.T @ w, rtol=0, atol=1e-12 * max(1.0, np.abs(Jd.T @ w).max()))
    ev.close()
    ref.close()


# ---- construction-time refusal --------------------------------------------------------------------------------------------
def _problem_with(prog, names=("x", "u")):
    G, traj = pt.bilinear_dynamics_and_trajectory(N=5, seed=2)
    c = dto.NonlinearKnotPointConstraint(prog, list(names), traj)
    return dto.DirectTrajOptProblem(traj, dto.QuadraticRegularizer("u", traj, 1.0), [dto.BilinearIntegrator(G, "x", "u", traj)], constraints=[c])


def _expect(code, prob, match):
    if code == dto._lib.DTO_ERR_UNSUPPORTED:
        with pytest.raises(dto.UnsupportedComponent, match=match):
            dto.Evaluator(prob)
    else:
        with pytest.raises(dto.DtoError, match=match) as e:
            dto.Evaluator(prob)
        assert e.value.code == code


def _tampered(edit, params=None):
    """a valid program whose traced tape is edited before it reaches the library (the raw descriptor path)"""
    prog = dto.KnotProgram((lambda v, p: [v[0] * p[0] - np.sin(v[1])]) if params is not None else (lambda v: [v[0] * v[1] - np.sin(v[1])]),
                           params=params)
    prob = _problem_with(prog)
    tape = prog.trace(prob.nonlinear_constraints()[0].var_dim)
    edit(tape)
    return prob


def test_malformed_programs_are_rejected():
    inv = dto._lib.DTO_ERR_INVALID
    nv = 6  # x (4) + u (2)
    _expect(inv, _tampered(lambda t: t._ops.__setitem__(-1, (5, len(t._ops) - 1, 0))), "operand out of range")  # forward operand
    _expect(inv, _tampered(lambda t: t._ops.__setitem__(0, (1, nv, 0))), "operand out of range")                 # variable >= nv
    _expect(inv, _tampered(lambda t: t._ops.__setitem__(1, (2, 1, 0)), params=[2.0]), "operand out of range")    # parameter >= n_params
    _expect(inv, _tampered(lambda t: t._ops.__setitem__(0, (42, 0, 0))), "unknown opcode")
    _expect(inv, _tampered(lambda t: setattr(t, "out", np.r_[t.out, t.out])), "outputs where the term has 1")     # n_out != g_dim


def test_bad_program_index_is_rejected(monkeypatch):
    prob = _problem_with(dto.KnotProgram(lambda v: [v[0] - v[4] ** 2]))
    real = dto._lib.load()

    class Lib:
        def __getattr__(self, name):
            return getattr(real, name)

        def dto_create(self, desc, out):
            d = desc._obj  # the ProblemDesc behind byref()
            d.constraints[0].program = 3
            return real.dto_create(desc, out)

    monkeypatch.setattr(dto._lib, "load", lambda: Lib())
    with pytest.raises(dto.DtoError, match="knot program index 3") as e:
        dto.Evaluator(prob)
    assert e.value.code == dto._lib.DTO_ERR_INVALID


def test_program_limits():
    header = open(__file__.replace("tests/test_knot_program_gpu.py", "include/dto_b200.h")).read()
    assert "#define DTO_MAX_PROGRAM_OPS 4096" in header and "#define DTO_MAX_PROGRAM_SLOTS 32" in header
    # more operations than DTO_MAX_PROGRAM_OPS
    long = dto.KnotProgram(lambda v: [sum(np.sin(v[i % 5] * (1.0 + i)) for i in range(1400))])
    _expect(dto._lib.DTO_ERR_UNSUPPORTED, _problem_with(long), "above the limit of 4096")
    # 40 values that must all be live at once: the sum consumes them, the product reuses every one afterwards
    G, traj = pt.bilinear_dynamics_and_trajectory(N=4, seed=2)
    traj2 = dto.NamedTrajectory({**{n: traj.data[traj.components[n], :] for n in traj.names}, "w": np.ones((40, 4))},
                                controls=("dt",), timestep="dt")

    def wide(v):
        s = [np.sin(v[i]) for i in range(40)]
        prod = s[39]
        for i in range(38, -1, -1):
            prod = prod * s[i]
        return [sum(s) * prod]

    def with_w(prog):
        c = dto.NonlinearKnotPointConstraint(prog, "w", traj2)
        return dto.DirectTrajOptProblem(traj2, dto.QuadraticRegularizer("u", traj2, 1.0), [dto.BilinearIntegrator(G, "x", "u", traj2)],
                                        constraints=[c])

    _expect(dto._lib.DTO_ERR_UNSUPPORTED, with_w(dto.KnotProgram(wide)), "live values")
    # v @ v over 128 variables: 128 leaves would be live in trace order, the compiled order needs a handful of slots
    traj3 = dto.NamedTrajectory({**{n: traj.data[traj.components[n], :] for n in traj.names},
                                 "w": np.random.default_rng(0).standard_normal((128, 4))}, controls=("dt",), timestep="dt")
    J = dto.QuadraticRegularizer("u", traj3, 1.0) + dto.KnotPointObjective(dto.KnotProgram(lambda v: v @ v), "w", traj3, times=[2, 4])
    prob = dto.DirectTrajOptProblem(traj3, J, [dto.BilinearIntegrator(G, "x", "u", traj3)])
    ev = dto.Evaluator(prob)
    Z = traj3.vec()
    spec = prob.to_spec()
    assert abs(ev.eval_objective(Z) - orc.eval_objective(spec, Z)) <= 1e-12 * abs(orc.eval_objective(spec, Z))
    grad = np.empty(ev.n_vars)
    ev.eval_objective_gradient(grad, Z)
    assert relerr(grad, orc.eval_objective_gradient(spec, Z)) <= 1e-12
    ev.close()

"""Parity of the CUDA evaluator (through the C ABI) against the CPU oracle on identical seeded
trajectories: structures bit-exact, values within 1e-10 relative to the array's max-norm
(BASELINE.json north_star tolerance; SURVEY.md section 7 explains why the norm is per block)."""
import numpy as np
import pytest

import dto_b200 as dto
import dto_oracle as orc
from dto_b200 import problem_templates as pt
from helpers import blocks
from helpers.kernels import interval_kernels, norm as kernel_name

pytestmark = pytest.mark.gpu

TOL = 1e-10


def relerr(got, ref):
    scale = max(np.abs(ref).max() if ref.size else 0.0, 1e-300)
    return np.abs(got - ref).max() / scale if ref.size else 0.0


def catalogue_problem(N=7, seed=3):
    """Every entry of the device knot-function catalogue, multi-variable constraints, per-time
    parameters, a structurally-zero derivative (dropped from the stored pattern) and a baseline."""
    rng = np.random.default_rng(seed)
    G, traj = pt.bilinear_dynamics_and_trajectory(N=N, seed=seed)
    integrators = [dto.BilinearIntegrator(G, "x", "u", traj), dto.DerivativeIntegrator("u", "du", traj),
                   dto.DerivativeIntegrator("du", "ddu", traj)]
    J = dto.TerminalObjective(dto.IsoInfidelity(traj.goal["x"]), "x", traj, Q=3.0)
    J = J + 0.5 * dto.KnotPointObjective(dto.NormSqPlus(per_time=[1.0, 2.0]), "u", traj, times=[1, N], Qs=[1.0, 2.0])
    J = J + dto.KnotPointObjective(dto.LinearCost(rng.standard_normal(6)), ["x", "du"], traj, times=[2, 3])
    J = J + dto.KnotPointObjective(dto.SqDist(rng.standard_normal(2)), "ddu", traj)
    J = J + dto.QuadraticRegularizer("du", traj, [0.3, 0.7], baseline=rng.standard_normal((2, N)), times=[1, 3, N])
    J = J + 2.0 * dto.MinimumTimeObjective(traj, D=0.7)
    A = rng.standard_normal((2, 6))
    A[1, 2] = 0.0  # never stored: SparseArrays drops the zero derivative
    cons = [
        dto.NonlinearKnotPointConstraint(dto.NormSqMinus(0.5), "x", traj, times=[1, 4], equality=True),
        dto.NonlinearKnotPointConstraint(dto.SqDistMinus(rng.standard_normal(4), 0.1), ["u", "du"], traj, times=[2, 3, N], equality=False),
        dto.NonlinearKnotPointConstraint(dto.LinearMap(A, rng.standard_normal(2)), ["x", "u"], traj, equality=True),
        dto.NonlinearKnotPointConstraint(dto.NormMinus(1.0), "u", traj, times=range(2, N), equality=False),
    ]
    return dto.DirectTrajOptProblem(traj, J, integrators, constraints=cons)


def zero_drive_problem(n=16, N=4):
    """A drive whose matrix is identically zero (all u-derivatives vanish but the columns stay in the structure)."""
    rng = np.random.default_rng(3)
    G0 = rng.standard_normal((n, n)) / n
    traj = dto.NamedTrajectory({"x": rng.standard_normal((n, N)), "u": rng.standard_normal((1, N)), "dt": np.full(N, 0.1)},
                               timestep="dt", controls=("u",))
    return dto.DirectTrajOptProblem(traj, dto.QuadraticRegularizer("u", traj, 1.0),
                                    dto.BilinearIntegrator(lambda u: G0 + u[0] * np.zeros((n, n)), "x", "u", traj))


def nonnormal_problem(n=32, N=6, scale=30.0, m=2):
    """Strongly non-normal generators (strictly upper-triangular drift, ||dt G||_1 ~ 3 but ||(dt G)^2||^(1/2) far smaller):
    the series plan (series_plan.cu) shortens the Taylor series the most here."""
    rng = np.random.default_rng(11)
    G0 = scale * np.triu(rng.standard_normal((n, n)), 1) / n
    Gd = [0.2 * rng.standard_normal((n, n)) / np.sqrt(n) for _ in range(m)]
    traj = dto.NamedTrajectory({"x": rng.standard_normal((n, N)), "u": 0.3 * rng.standard_normal((m, N)), "dt": np.full(N, 0.1)},
                               timestep="dt", controls=("u", "dt"), bounds={"dt": (0.01, 0.5)})
    return dto.DirectTrajOptProblem(traj, dto.QuadraticRegularizer("u", traj, 1.0) + dto.MinimumTimeObjective(traj, D=1.0),
                                    dto.BilinearIntegrator((G0, Gd), "x", "u", traj))


PROBLEMS = {
    "readme_c1": lambda: pt.readme_problem(N=50),
    "catalogue": catalogue_problem,
    "scaled_n8_stages": lambda: pt.scaled_problem(N=6, state_dim=8, n_controls=2, generator_scale=8.0),
    "scaled_n6_stages": lambda: pt.scaled_problem(N=5, state_dim=6, n_controls=3, generator_scale=9.0),
    "scaled_n24_m3": lambda: pt.scaled_problem(N=6, state_dim=24, n_controls=3, generator_scale=0.5),
    "scaled_n48_m1": lambda: pt.scaled_problem(N=4, state_dim=48, n_controls=1, generator_scale=0.3),
    "standard": lambda: pt.standard_problem(N=10),
    "evaluator_test": lambda: pt.evaluator_test_problem(N=10),
    "benchmark_N51": lambda: pt.bilinear_benchmark(N=51),
    "scaled_n5": lambda: pt.scaled_problem(N=6, state_dim=5, n_controls=2, generator_scale=0.7),
    "scaled_n8": lambda: pt.scaled_problem(N=12, state_dim=8, n_controls=2),
    "scaled_n16_bignorm": lambda: pt.scaled_problem(N=8, state_dim=16, n_controls=2),
    "gate_n32": lambda: pt.quantum_gate_problem(N=12, levels=16, n_drives=4),
    "gate_n6": lambda: pt.quantum_gate_problem(N=7, levels=3, n_drives=2),
    "gate_n64": lambda: pt.quantum_gate_problem(N=5, levels=32, n_drives=2),
    "linreg": lambda: pt.linear_regularizer_problem(N=8),
    # edge cases: the shortest trajectory, all drives and Hessian rows at n = 48/64 (series-mode propagator),
    # scaling-and-squaring (theta = 3) and multi-stage series (theta = 12), a zero drive matrix
    "N2_n8": lambda: pt.scaled_problem(N=2, state_dim=8, n_controls=2),
    "N2_readme": lambda: pt.readme_problem(N=2),
    "n64_m4": lambda: pt.scaled_problem(N=3, state_dim=64, n_controls=4, generator_scale=0.4),
    "n48_m4": lambda: pt.scaled_problem(N=3, state_dim=48, n_controls=4, generator_scale=0.4),
    "n32_theta3": lambda: pt.scaled_problem(N=4, state_dim=32, n_controls=3, generator_scale=3.0),
    "n16_theta12": lambda: pt.scaled_problem(N=4, state_dim=16, n_controls=2, generator_scale=12.0),
    "zero_drive_n16": zero_drive_problem,
    "nonnormal_n32": nonnormal_problem,
    "nonnormal_n24_big": lambda: nonnormal_problem(n=24, N=4, scale=90.0, m=3),
    # global (non-time-varying) variables: all four global term kinds, the reference's test functions
    "global": lambda: pt.global_problem(N=9),
    "global_ref_fixture": lambda: pt.global_problem(N=6, with_goal=False),
    "global_dim3": lambda: pt.global_problem(N=12, global_dim=3, seed=5),
    "global_goal": lambda: pt.global_goal_problem(N=11),
}


@pytest.fixture(scope="module", params=list(PROBLEMS))
def case(request):
    prob = PROBLEMS[request.param]()
    ev = dto.Evaluator(prob)
    yield request.param, prob, ev
    ev.close()


def test_structures_bit_exact(case):
    name, prob, ev = case
    spec, Z = prob.to_spec(), prob.trajectory.vec()
    jr, jc = ev.jacobian_structure()
    orow, ocol = orc.jacobian_structure(spec, Z)
    assert jr.size == orow.size and np.array_equal(jr, orow) and np.array_equal(jc, ocol)
    hr, hc = ev.hessian_lagrangian_structure()
    orow, ocol = orc.hessian_structure(spec, Z)
    assert hr.size == orow.size and np.array_equal(hr, orow) and np.array_equal(hc, ocol)
    nd, nn = orc.n_constraints(spec)
    assert (ev.n_dynamics_constraints, ev.n_nonlinear_constraints, ev.n_constraints) == (nd, nn, nd + nn)


def test_values_match_oracle(case):
    name, prob, ev = case
    spec = prob.to_spec()
    rng = np.random.default_rng(7)
    Z0 = prob.trajectory.vec()
    Z = Z0 + 0.05 * rng.standard_normal(Z0.size)  # an iterate away from the initial point
    dts = slice(spec["components"][spec["timestep"]][0], spec["N"] * spec["z"], spec["z"])
    Z[dts] = np.abs(Z[dts])
    jst, hst = orc.jacobian_structure(spec, Z0), orc.hessian_structure(spec, Z0)
    mu = rng.random(ev.n_constraints)
    sigma = 2.0

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
    # relative to the block norm (BASELINE.md section 2): per (row block, component) Jacobian block, per Hessian knot region
    assert relerr(J, Jref) <= TOL and blocks.jac_block_relerr(spec, jst, J, Jref) <= TOL
    H = np.full(ev.nnz_hessian, np.nan)
    ev.eval_hessian_lagrangian(H, Z, sigma, mu)
    Href = orc.eval_hessian_lagrangian(spec, Z, sigma, mu, hst)
    assert relerr(H, Href) <= TOL and blocks.hess_block_relerr(spec, hst, H, Href) <= TOL
    # sigma == 0 skips the objective (evaluator.jl:626)
    ev.eval_hessian_lagrangian(H, Z, 0.0, mu)
    H0 = orc.eval_hessian_lagrangian(spec, Z, 0.0, mu, hst)
    assert relerr(H, H0) <= TOL and blocks.hess_block_relerr(spec, hst, H, H0) <= TOL


def test_fused_eval_all_equals_separate_callbacks(case):
    name, prob, ev = case
    rng = np.random.default_rng(11)
    Z = prob.trajectory.vec()
    mu = rng.random(ev.n_constraints)
    Jv, grad = np.empty(1), np.empty(ev.n_vars)
    g, jac, hess = np.empty(ev.n_constraints), np.empty(ev.nnz_jacobian), np.empty(ev.nnz_hessian)
    ev.eval_all(Z, 1.5, mu, Jv, grad, g, jac, hess)
    g2, jac2, hess2, grad2 = np.empty_like(g), np.empty_like(jac), np.empty_like(hess), np.empty_like(grad)
    ev.eval_constraint(g2, Z)
    ev.eval_constraint_jacobian(jac2, Z)
    ev.eval_hessian_lagrangian(hess2, Z, 1.5, mu)
    ev.eval_objective_gradient(grad2, Z)
    assert np.array_equal(g, g2) and np.array_equal(jac, jac2) and np.array_equal(hess, hess2) and np.array_equal(grad, grad2)
    assert Jv[0] == ev.eval_objective(Z)


def test_jacobian_products(case):
    """evaluator.jl:808-853: products vs the oracle's dense Jacobian, atol 1e-10."""
    name, prob, ev = case
    rng = np.random.default_rng(5)
    Z = prob.trajectory.vec()
    spec = prob.to_spec()
    jst = orc.jacobian_structure(spec, Z)
    Jd = np.zeros((ev.n_constraints, ev.n_vars))
    np.add.at(Jd, (jst[0] - 1, jst[1] - 1), orc.eval_constraint_jacobian(spec, Z, jst))
    w = rng.standard_normal(ev.n_vars)
    y = np.empty(ev.n_constraints)
    ev.eval_constraint_jacobian_product(y, Z, w)
    assert np.allclose(y, Jd @ w, atol=1e-10 * max(1, np.abs(Jd @ w).max()))
    w = rng.standard_normal(ev.n_constraints)
    y = np.empty(ev.n_vars)
    ev.eval_constraint_jacobian_transpose_product(y, Z, w)
    assert np.allclose(y, Jd.T @ w, atol=1e-10 * max(1, np.abs(Jd.T @ w).max()))


def test_matrix_free_products_match_materialised(monkeypatch):
    """Jacobian-vector products straight from the series (no Jacobian values formed) against the reference's
    materialise-then-multiply path (evaluator.jl:406-456), on a problem with two integrator kinds and knot
    constraints with never-stored entries."""
    big = pt.scaled_problem(N=40, state_dim=16, n_controls=2, generator_scale=0.6)
    for pr in (big, pt.quantum_gate_problem(N=9, levels=16, n_drives=4)):
        Z = pr.trajectory.datavec.copy()
        res = {}
        for mode in ("", "materialize"):
            if mode:
                monkeypatch.setenv("DTO_B200_JVP", mode)
            else:
                monkeypatch.delenv("DTO_B200_JVP", raising=False)
            ev = dto.Evaluator(pr)
            rng = np.random.default_rng(11)
            w1, w2 = rng.standard_normal(ev.n_vars), rng.standard_normal(ev.n_constraints)
            y1, y2 = np.empty(ev.n_constraints), np.empty(ev.n_vars)
            l0 = ev.launch_count
            ev.eval_constraint_jacobian_product(y1, Z, w1)
            ev.eval_constraint_jacobian_transpose_product(y2, Z, w2)
            res[mode] = (y1, y2, ev.launch_count - l0)
            ev.close()
        for a, b in zip(res[""][:2], res["materialize"][:2]):
            assert relerr(a, b) <= 1e-12
    monkeypatch.delenv("DTO_B200_JVP", raising=False)


def test_global_variables_in_a_batch_and_on_shards():
    """Batches carry their own global variables ([batch][z*N + global_dim]); knot-range shards reject them."""
    prob = pt.global_problem(N=7, seed=2)
    rng = np.random.default_rng(9)
    B = 3
    Z = np.stack([prob.trajectory.vec() + 0.03 * rng.standard_normal(prob.trajectory.vec().size) for _ in range(B)])
    ev1, evb = dto.Evaluator(prob), dto.Evaluator(prob, batch=B)
    mu = rng.random((B, ev1.n_constraints))
    Jb, gradb = np.empty(B), np.empty((B, ev1.n_vars))
    gb, jacb, hessb = np.empty((B, ev1.n_constraints)), np.empty((B, ev1.nnz_jacobian)), np.empty((B, ev1.nnz_hessian))
    evb.eval_all(Z, 1.3, mu, Jb, gradb, gb, jacb, hessb)
    for b in range(B):
        J, grad = np.empty(1), np.empty(ev1.n_vars)
        g, jac, hess = np.empty(ev1.n_constraints), np.empty(ev1.nnz_jacobian), np.empty(ev1.nnz_hessian)
        ev1.eval_all(Z[b], 1.3, mu[b], J, grad, g, jac, hess)
        assert J[0] == Jb[b] and np.array_equal(grad, gradb[b]) and np.array_equal(g, gb[b])
        assert np.array_equal(jac, jacb[b]) and np.array_equal(hess, hessb[b])
    with pytest.raises(dto.UnsupportedComponent):
        dto.Evaluator(prob, shard=(1, 4))
    ev1.close()
    evb.close()


def test_features_and_bounds():
    prob = pt.standard_problem(N=6)
    ev = dto.Evaluator(prob, eval_hessian=False)
    assert ev.features_available() == ["Grad", "Jac"]
    H = np.empty(ev.nnz_hessian)
    with pytest.raises(dto.DtoError):
        ev.eval_hessian_lagrangian(H, prob.trajectory.datavec, 1.0, np.ones(ev.n_constraints))
    lo, hi = ev.constraint_bounds()
    assert np.all(hi == 0) and np.all(lo[: ev.n_dynamics_constraints] == 0) and np.all(np.isneginf(lo[ev.n_dynamics_constraints :]))
    ev.close()
    assert dto.Evaluator(prob).features_available() == ["Grad", "Jac", "Hess"]


def test_unsupported_components_raise_at_construction():
    G, traj = pt.bilinear_dynamics_and_trajectory(N=5)
    with pytest.raises(dto.UnsupportedComponent):
        dto.BilinearIntegrator(lambda u: pt.GZ + u[0] ** 2 * pt.GX, "x", "u", traj)
    with pytest.raises(dto.UnsupportedComponent):
        dto.NonlinearKnotPointConstraint(lambda u: [u[0]], "u", traj)


def _wide_knot_problem(kind, extra, N=3):
    """A bilinear (n = 64) or linear-spline time-dependent (n = 64) problem whose knot carries `extra` more variables that
    only a QuadraticRegularizer reads: the knot width z, not the state, sets the Hessian assembler's shared memory."""
    rng = np.random.default_rng(21)
    base = (pt.scaled_problem(N=N, state_dim=64, n_controls=2, generator_scale=0.1) if kind == "bilinear"
            else pt.carrier_problem(N=N, state_dim=64, n_drives=2, spline_order=1))
    t = base.trajectory
    comps = {name: t.data[t.components[name], :] for name in t.names}
    comps["w"] = rng.standard_normal((extra, N))
    traj = dto.NamedTrajectory(comps, controls=("dt",), timestep="dt")
    if kind == "bilinear":
        G = base.integrators[0].G
        ints = [dto.BilinearIntegrator((G[0], list(G[1:])), "x", "u", traj), dto.DerivativeIntegrator("u", "du", traj)]
    else:
        ints = [dto.TimeDependentBilinearIntegrator(base.integrators[0].G, "x", "u", "t", traj, spline_order=1),
                dto.DerivativeIntegrator("u", "du", traj), dto.DerivativeIntegrator("du", "ddu", traj)]
    J = dto.QuadraticRegularizer("u", traj, 1.0) + dto.QuadraticRegularizer("w", traj, 0.5)
    return dto.DirectTrajOptProblem(traj, J, ints)


@pytest.mark.parametrize("shape", [("bilinear", n, m) for n in (72, 80, 84, 88, 96) for m in (1, 4)]
                         + [("wide_knot", "bilinear", 115), ("wide_knot", "tdb", 60)], ids=lambda s: "-".join(map(str, s)))
def test_accepted_shapes_evaluate(shape):
    """Every shape dto_create accepts evaluates correctly; a shape no kernel can launch (the generic interval kernel
    stages the generator and every jet column of an interval, the Hessian assembler a z x z tile per knot, two with
    cross-knot coupling) is rejected at construction, naming the device's shared-memory limit."""
    if shape[0] == "bilinear":
        prob = pt.scaled_problem(N=3, state_dim=shape[1], n_controls=shape[2], generator_scale=1.0 / shape[1])
    else:
        prob = _wide_knot_problem(shape[1], shape[2])
    try:
        ev = dto.Evaluator(prob)
    except dto.UnsupportedComponent as e:
        assert "shared memory" in str(e) and "limit" in str(e), str(e)
        assert shape[0] != "bilinear" or shape[1] > 72  # every n <= 72 fits
        return
    spec = prob.to_spec()
    rng = np.random.default_rng(4)
    Z0 = prob.trajectory.vec()
    Z = Z0 + 0.02 * rng.standard_normal(Z0.size)
    jst, hst = orc.jacobian_structure(spec, Z0), orc.hessian_structure(spec, Z0)
    mu = rng.random(ev.n_constraints)
    Jv, grad = np.full(1, np.nan), np.full(ev.n_vars, np.nan)
    g, J, H = np.full(ev.n_constraints, np.nan), np.full(ev.nnz_jacobian, np.nan), np.full(ev.nnz_hessian, np.nan)
    ev.eval_all(Z, 1.2, mu, Jv, grad, g, J, H)
    tol = TOL if shape[0] == "bilinear" or shape[1] == "bilinear" else TDB_TOL
    assert relerr(g, orc.eval_constraint(spec, Z)) <= tol
    assert blocks.jac_block_relerr(spec, jst, J, orc.eval_constraint_jacobian(spec, Z, jst)) <= tol
    assert blocks.hess_block_relerr(spec, hst, H, orc.eval_hessian_lagrangian(spec, Z, 1.2, mu, hst)) <= tol
    assert relerr(grad, orc.eval_objective_gradient(spec, Z)) <= TOL
    ev.close()


# ---- TimeDependentBilinearIntegrator (K7) --------------------------------------------------------------
TDB_TOL = 1e-10  # fixed-order extrapolation integrator vs the oracle's rtol=1e-13 variational solve (DESIGN.md "TDBI parity")

_GBS = ("tdb_kernel",)


def _tdb(nt, warps, split=False):
    return (f"tdb_dmma_kernel<{nt}, {warps}>",) + ((f"tdb_exp_kernel<{nt}>",) if split else ())


# kernels: the interval kernels of one fused evaluation with the Hessian (tdb_dmma.cu make_plan: the interval is split into
# an exp kernel when its tiles need more than 8 warps, unless DTO_B200_TDB_SPLIT=0 asks for one 16-warp CTA; the CUDA-core
# kernel takes n % 8 != 0, n = 40 / 56, and 1 + np > 8 parameters)
TDB_CELLS = [
    (1, 4, 2, 0, None, _GBS), (0, 4, 2, 0, None, _GBS), (1, 6, 1, 2, None, _GBS), (1, 16, 2, 0, None, _tdb(2, 8)),
    (1, 8, 2, 1, None, _tdb(1, 8)), (0, 24, 3, 0, None, _tdb(3, 8)), (1, 32, 1, 2, None, _tdb(4, 8)), (0, 8, 4, 1, None, _tdb(1, 8)),
    (1, 32, 2, 0, None, _tdb(4, 8, True)), (0, 32, 4, 0, None, _tdb(4, 8, True)),              # NT = 4 split
    (0, 48, 1, 0, None, _tdb(6, 8, True)), (1, 48, 2, 1, None, _tdb(6, 8, True)),              # NT = 6
    (1, 32, 2, 0, "0", _tdb(4, 16)), (0, 48, 1, 0, "0", _tdb(6, 16)), (1, 64, 2, 0, "0", _tdb(8, 16)),  # one 16-warp CTA
    (1, 16, 3, 0, None, _GBS), (1, 32, 4, 0, None, _GBS),                                      # 1 + np > 8
    (1, 40, 2, 0, None, _GBS), (0, 56, 2, 0, None, _GBS), (0, 16, 2, 4, None, _tdb(2, 8)),     # n = 40 / 56; four carriers
]


@pytest.mark.parametrize("order,n,m,carriers,split,kernels", TDB_CELLS,
                         ids=[f"{c[0]}-{c[1]}-{c[2]}-{c[3]}" + ("" if c[4] is None else f"-split{c[4]}") for c in TDB_CELLS])
def test_tdbilinear_matches_exact_variational_solution(monkeypatch, order, n, m, carriers, split, kernels):
    if split is not None:
        monkeypatch.setenv("DTO_B200_TDB_SPLIT", split)
    rng = np.random.default_rng(9)
    prob = pt.carrier_problem(N=5, state_dim=n, n_drives=m, spline_order=order, dt=0.2)
    if carriers:
        g = prob.integrators[0].G

        def skew():
            M = rng.standard_normal((n, n))
            return 0.3 * (M - M.T) / n

        prob.integrators[0].G = dto.CarrierGenerator(g.G0, g.A, g.B, g.omega, g.phi + 0.3, D=np.stack([skew() for _ in range(carriers)]),
                                                     omega_d=1.0 + rng.random(carriers), phi_d=rng.random(carriers))
    spec = prob.to_spec()
    ev = dto.Evaluator(prob)
    Z0 = prob.trajectory.vec()
    Z = Z0 + 0.02 * rng.standard_normal(Z0.size)
    jst, hst = orc.jacobian_structure(spec, Z0), orc.hessian_structure(spec, Z0)
    jr, jc = ev.jacobian_structure()
    hr, hc = ev.hessian_lagrangian_structure()
    assert np.array_equal(jr, jst[0]) and np.array_equal(jc, jst[1]) and np.array_equal(hr, hst[0]) and np.array_equal(hc, hst[1])
    mu = rng.random(ev.n_constraints)
    g = np.empty(ev.n_constraints)
    ev.eval_constraint(g, Z)
    assert relerr(g, orc.eval_constraint(spec, Z)) <= TDB_TOL
    J = np.empty(ev.nnz_jacobian)
    ev.eval_constraint_jacobian(J, Z)
    Jref = orc.eval_constraint_jacobian(spec, Z, jst)
    assert relerr(J, Jref) <= TDB_TOL and blocks.jac_block_relerr(spec, jst, J, Jref) <= TDB_TOL
    H = np.empty(ev.nnz_hessian)
    ev.eval_hessian_lagrangian(H, Z, 1.5, mu)
    Href = orc.eval_hessian_lagrangian(spec, Z, 1.5, mu, hst)
    assert relerr(H, Href) <= TDB_TOL and blocks.hess_block_relerr(spec, hst, H, Href) <= TDB_TOL
    if order == 1:  # cross-knot Hessian entries are genuinely nonzero for the linear spline
        z = spec["z"]
        cross = (hr - 1) // z != (hc - 1) // z
        assert np.abs(Href[cross]).max() > 1e-6
    # the fused evaluation runs exactly the intended instantiations
    bufs = [np.empty(ev.n_constraints), np.empty(ev.nnz_jacobian), np.empty(ev.nnz_hessian)]
    ks = interval_kernels(lambda: ev.eval_all(Z + 1e-3, 1.5, mu, None, None, *bufs))
    assert ks == {kernel_name(k) for k in kernels}, sorted(ks)
    Zb = Z + 1e-3
    assert relerr(bufs[0], orc.eval_constraint(spec, Zb)) <= TDB_TOL
    assert blocks.jac_block_relerr(spec, jst, bufs[1], orc.eval_constraint_jacobian(spec, Zb, jst)) <= TDB_TOL
    assert blocks.hess_block_relerr(spec, hst, bufs[2], orc.eval_hessian_lagrangian(spec, Zb, 1.5, mu, hst)) <= TDB_TOL
    ev.close()


def test_c3_shape_matches_oracle():
    """BASELINE config c3 at its real shape (n = 64, 2 drives, linear spline, derivative chain u -> du -> ddu, knot
    constraint norm(u) - 1 <= 0 at knots 2..N-1) on a short trajectory: the `tdb_dmma_kernel<8,8>` + `tdb_exp_kernel<8>`
    instantiations, whole problem against the oracle, values relative to the block norm."""
    rng = np.random.default_rng(13)
    prob = pt.carrier_problem(N=8, state_dim=64, n_drives=2, spline_order=1)
    spec = prob.to_spec()
    ev = dto.Evaluator(prob)
    assert ev.kernel_variant(0) == "gbs-dmma"
    Z0 = prob.trajectory.vec()
    Z = Z0 + 0.02 * rng.standard_normal(Z0.size)
    jst, hst = orc.jacobian_structure(spec, Z0), orc.hessian_structure(spec, Z0)
    jr, jc = ev.jacobian_structure()
    hr, hc = ev.hessian_lagrangian_structure()
    assert np.array_equal(jr, jst[0]) and np.array_equal(jc, jst[1]) and np.array_equal(hr, hst[0]) and np.array_equal(hc, hst[1])
    mu = rng.random(ev.n_constraints)
    Jv, grad = np.empty(1), np.empty(ev.n_vars)
    g, J, H = np.empty(ev.n_constraints), np.empty(ev.nnz_jacobian), np.empty(ev.nnz_hessian)
    ev.eval_all(Z, 1.5, mu, Jv, grad, g, J, H)
    gref, Jref = orc.eval_constraint(spec, Z), orc.eval_constraint_jacobian(spec, Z, jst)
    Href = orc.eval_hessian_lagrangian(spec, Z, 1.5, mu, hst)
    assert relerr(g, gref) <= TDB_TOL and blocks.vec_block_relerr(spec, g, gref) <= TDB_TOL
    assert relerr(J, Jref) <= TDB_TOL and blocks.jac_block_relerr(spec, jst, J, Jref) <= TDB_TOL
    assert relerr(H, Href) <= TDB_TOL and blocks.hess_block_relerr(spec, hst, H, Href) <= TDB_TOL
    assert relerr(grad, orc.eval_objective_gradient(spec, Z)) <= TOL
    assert abs(Jv[0] - orc.eval_objective(spec, Z)) <= TOL * max(1.0, abs(Jv[0]))
    ev.close()


def test_c3_full_size_sampled_intervals():
    """config c3 at N = 1000: sampled intervals (first, last, random) against the oracle's variational solve."""
    rng = np.random.default_rng(14)
    prob = pt.carrier_problem(N=1000, state_dim=64, n_drives=2, spline_order=1)
    spec = prob.to_spec()
    ev = dto.Evaluator(prob)
    Z = prob.trajectory.vec() + 0.02 * rng.standard_normal(ev.n_vars)
    mu = rng.random(ev.n_constraints)
    Jv, grad = np.empty(1), np.empty(ev.n_vars)
    g, J, H = np.empty(ev.n_constraints), np.empty(ev.nnz_jacobian), np.empty(ev.nnz_hessian)
    ev.eval_all(Z, 0.8, mu, Jv, grad, g, J, H)
    ks = sorted({1, 2, 999, 1000} | {int(k) for k in rng.integers(1, 1001, size=12)})
    er, ej, eh = blocks.sampled_interval_check(spec, Z, 0.8, mu, g, J, H, ks, jac_structure=ev.jacobian_structure())
    assert er <= TDB_TOL and ej <= TDB_TOL and eh <= TDB_TOL, (er, ej, eh)
    ev.close()


@pytest.mark.parametrize("n,dt", [(8, 1.5), (6, 2.0), (16, 0.8)])
def test_tdbilinear_large_steps(n, dt):
    """Large |dt| (||G|| + carrier frequency): the kernels choose the number of macro steps per interval from the iterate
    (tdb_item_steps: theta ~ 3..8 here, i.e. several macro steps) instead of silently losing accuracy with one
    (the reference's Tsit5 adapts its steps the same way, time_dependent_bilinear_integrator.jl:117-127)."""
    rng = np.random.default_rng(17)
    prob = pt.carrier_problem(N=4, state_dim=n, n_drives=2, spline_order=1, dt=dt)
    spec = prob.to_spec()
    ev = dto.Evaluator(prob)
    Z0 = prob.trajectory.vec()
    Z = Z0 + 0.02 * rng.standard_normal(Z0.size)
    jst, hst = orc.jacobian_structure(spec, Z0), orc.hessian_structure(spec, Z0)
    mu = rng.random(ev.n_constraints)
    g, J, H = np.empty(ev.n_constraints), np.empty(ev.nnz_jacobian), np.empty(ev.nnz_hessian)
    ev.eval_all(Z, 1.0, mu, None, None, g, J, H)
    assert relerr(g, orc.eval_constraint(spec, Z)) <= TDB_TOL
    Jref = orc.eval_constraint_jacobian(spec, Z, jst)
    assert relerr(J, Jref) <= TDB_TOL and blocks.jac_block_relerr(spec, jst, J, Jref) <= TDB_TOL
    Href = orc.eval_hessian_lagrangian(spec, Z, 1.0, mu, hst)
    assert relerr(H, Href) <= TDB_TOL
    ev.close()


def test_tdbilinear_variants_agree(monkeypatch):
    """The tensor-core variant of K7 and the CUDA-core variant integrate the same equations with the same
    extrapolation scheme: they must agree far below the parity tolerance (and the dispatch must pick them)."""
    prob = pt.carrier_problem(N=6, state_dim=16, n_drives=2, spline_order=1, dt=0.2)
    Z = prob.trajectory.vec()
    outs = {}
    for pin in ("", "generic"):
        if pin:
            monkeypatch.setenv("DTO_B200_KERNEL", pin)
        ev = dto.Evaluator(prob)
        assert ev.kernel_variant(0) == ("gbs" if pin else "gbs-dmma")
        mu = np.random.default_rng(2).random(ev.n_constraints)
        bufs = [np.empty(1), np.empty(ev.n_vars), np.empty(ev.n_constraints), np.empty(ev.nnz_jacobian), np.empty(ev.nnz_hessian)]
        ev.eval_all(Z, 1.0, mu, *bufs)
        outs[pin] = bufs
        ev.close()
    for a, b in zip(outs[""], outs["generic"]):
        assert relerr(a, b) <= 1e-12


def test_series_plan_matches_norm_based_series(monkeypatch):
    """The series plan (Taylor length from ||A^2||^(1/2), series_plan.cu) only drops terms below the 2^-53 tail: results
    agree with the ||A||_1-sized series to round-off, also for non-normal generators where the plan saves the most."""
    for mk in (nonnormal_problem, lambda: pt.quantum_gate_problem(N=9, levels=16, n_drives=4),
               lambda: pt.scaled_problem(N=5, state_dim=32, n_controls=3, generator_scale=3.0)):
        prob = mk()
        rng = np.random.default_rng(2)
        Z = prob.trajectory.vec() * (1 + 0.05 * rng.standard_normal(prob.trajectory.vec().size))
        outs = {}
        for plan in ("1", "0"):
            monkeypatch.setenv("DTO_B200_SERIES_PLAN", plan)
            ev = dto.Evaluator(prob)
            assert ev.kernel_variant(0) == "persistent"
            mu = np.random.default_rng(5).random(ev.n_constraints)
            bufs = [np.full(ev.n_constraints, np.nan), np.full(ev.nnz_jacobian, np.nan), np.full(ev.nnz_hessian, np.nan)]
            ev.eval_all(Z, 1.0, mu, None, None, *bufs)
            outs[plan] = bufs
            ev.close()
        for a, b in zip(outs["1"], outs["0"]):
            assert relerr(a, b) <= 1e-13


def _eval_dev(ev, Z, sigma, mu):
    """dto_eval_all_dev into device buffers, read back with torch: one pass over the whole trajectory, never cut into
    knot ranges"""
    import torch

    dev = torch.device("cuda", torch.cuda.current_device())
    dZ, dmu = torch.from_numpy(np.ascontiguousarray(Z)).to(dev), torch.from_numpy(np.ascontiguousarray(mu)).to(dev)
    outs = [torch.full((n,), float("nan"), dtype=torch.float64, device=dev)
            for n in (1, ev.n_vars, ev.n_constraints, ev.nnz_jacobian, ev.nnz_hessian)]
    torch.cuda.synchronize()
    ev.eval_all_dev(dZ.data_ptr(), sigma, dmu.data_ptr(), *[o.data_ptr() for o in outs])
    ev.synchronize()
    return [o.cpu().numpy() for o in outs]


def test_host_pipeline_matches_single_pass():
    """dto_eval_all with host buffers cuts large problems into knot ranges whose Jacobian columns and Hessian
    blocks leave over PCIe while later ranges are computed; the result must be bit-identical to the
    single-pass device-pointer evaluation (also with knot constraints and derivative integrators), for every
    interval kernel with its own cut plan."""
    cases = [  # (kernel variant, problem, knot ranges of the host-pointer call)
        ("persistent", pt.scaled_problem(N=700, state_dim=32, n_controls=2, generator_scale=0.3), 2),
        ("octet", pt.scaled_problem(N=1000, state_dim=16, n_controls=2, generator_scale=0.25), 4),
        # 599 intervals: one cut at two rounds of one CTA per SM (296 on a 148-SM B200)
        ("gbs-dmma", pt.carrier_problem(N=600, state_dim=64, n_drives=2), 2),
    ]
    for variant, prob, ranges in cases:
        Z = prob.trajectory.vec()
        ev = dto.Evaluator(prob)
        assert ev.kernel_variant(0) == variant
        mu = np.random.default_rng(5).random(ev.n_constraints)
        ref = _eval_dev(ev, Z, 1.7, mu)
        bufs = [np.full(1, np.nan), np.full(ev.n_vars, np.nan), np.full(ev.n_constraints, np.nan),
                np.full(ev.nnz_jacobian, np.nan), np.full(ev.nnz_hessian, np.nan)]
        assert 8 * (ev.nnz_jacobian + ev.nnz_hessian) >= 8 << 20, variant
        ev.kernel_timing(True)
        ev.eval_all(Z, 1.7, mu, *bufs)
        _, launches = ev.kernel_time_ms()  # one per knot range (one interval kernel per range)
        ev.kernel_timing(False)
        assert launches == ranges, variant
        assert all(np.isfinite(b).all() for b in bufs), variant
        for a, b in zip(ref, bufs):
            assert np.array_equal(a, b), variant
        ev.close()


def test_structural_zero_hessian_delivery():
    """Host-pointer path of bilinear/derivative problems: only the Hessian columns a term can touch cross PCIe (one 2-D
    copy per run of equal knots), host threads write the structural zeros of the caller's buffer meanwhile.  Must be
    bit-identical to the whole array of the device-pointer evaluation, including knots where an objective reaches into
    the x block."""
    prob = pt.quantum_gate_problem(N=640, levels=16, n_drives=4)
    t = prob.trajectory
    J = prob.objective + dto.KnotPointObjective(dto.SqDist(np.linspace(-1, 1, 32)), "x", t, times=[5, 6, 300], Qs=[1.0, 2.0, 3.0])
    prob2 = dto.DirectTrajOptProblem(t, J, prob.integrators)
    for pr in (prob, prob2, pt.scaled_problem(N=700, state_dim=32, n_controls=2, generator_scale=0.3)):
        Z = pr.trajectory.vec()
        ev = dto.Evaluator(pr)
        mu = np.random.default_rng(5).random(ev.n_constraints)
        ref = _eval_dev(ev, Z, 1.7, mu)
        for rep in range(2):  # the second call reuses the handle's worker threads
            bufs = [np.full(1, np.nan), np.full(ev.n_vars, np.nan), np.full(ev.n_constraints, np.nan),
                    np.full(ev.nnz_jacobian, np.nan), np.full(ev.nnz_hessian, np.nan)]
            ev.eval_all(Z, 1.7, mu, *bufs)
            assert all(np.isfinite(b).all() for b in bufs), rep
            for a, b in zip(ref, bufs):
                assert np.array_equal(a, b), rep
        H = np.full(ev.nnz_hessian, np.nan)
        ev.eval_hessian_lagrangian(H, Z, 1.7, mu)
        assert np.array_equal(H, bufs[4])
        ev.close()


@pytest.mark.parametrize("kind", ["persistent", "octet", "generic", "dmma", "tdb"])
def test_absurd_steps_poison_their_interval(monkeypatch, kind):
    """An iterate whose |dt| ||G|| is not finite or absurdly large (>= 1e8 for the Taylor kernels, > 256 for the
    extrapolation kernels, whose step count is capped there) must not come back as plausible numbers: the interval's
    residual rows are NaN (an evaluation error for the solver), every other interval is untouched."""
    if kind == "tdb":
        prob = pt.carrier_problem(N=6, state_dim=8, n_drives=2)
        big = 1e4
    else:
        if kind in ("generic", "dmma"):
            monkeypatch.setenv("DTO_B200_KERNEL", kind)
        n = 16 if kind == "octet" else 32
        prob = pt.scaled_problem(N=6, state_dim=n, n_controls=2, generator_scale=0.3)
        big = 1e12
    ev = dto.Evaluator(prob)
    spec = prob.to_spec()
    Z = prob.trajectory.vec().copy()
    g0 = np.empty(ev.n_constraints)
    ev.eval_constraint(g0, Z)
    assert np.isfinite(g0).all()
    z, dt_off = spec["z"], spec["components"][spec["timestep"]][0]
    k = 2  # third interval
    Z[k * z + dt_off] = big
    g = np.empty(ev.n_constraints)
    ev.eval_constraint(g, Z)
    n = prob.integrators[0].x_dim
    rows = slice(k * n, (k + 1) * n)  # the first integrator's rows of interval k
    assert np.isnan(g[rows]).all()
    others = np.ones(ev.n_constraints, bool)
    others[rows] = False
    # the derivative integrators of the same interval read the same dt: exclude rows that changed for that reason
    same = others & (g == g0)
    assert same.sum() >= (prob.trajectory.N - 2) * n and np.isfinite(g[others]).all()
    ev.close()


def test_tdb_extrapolation_columns_sized_per_interval(monkeypatch):
    """K7 sizes its extrapolation columns per interval from theta = |dt| (||G|| + omega) (error model theta^(2K+1) / (2^K K!)^2
    <= 1e-14): small steps take 5 of the 8 columns (35 instead of 80 right-hand sides).  The result must agree with the
    eight-column evaluation to round-off, for small and large steps, and intervals of one trajectory may differ in K."""
    prob = pt.carrier_problem(N=7, state_dim=16, n_drives=2, spline_order=1)
    spec = prob.to_spec()
    rng = np.random.default_rng(4)
    Z = prob.trajectory.vec() + 0.02 * rng.standard_normal(prob.trajectory.vec().size)
    dts = slice(spec["components"][spec["timestep"]][0], spec["N"] * spec["z"], spec["z"])
    Z[dts] = np.abs(Z[dts]) * np.array([1.0, 0.2, 6.0, 1.0, 12.0, 0.05, 1.0])  # a different theta (and K, and step count) per interval
    outs = {}
    for tol in ("0", "1e-14"):
        monkeypatch.setenv("DTO_B200_TDB_TOL", tol)
        ev = dto.Evaluator(prob)
        mu = np.random.default_rng(5).random(ev.n_constraints)
        bufs = [np.full(ev.n_constraints, np.nan), np.full(ev.nnz_jacobian, np.nan), np.full(ev.nnz_hessian, np.nan)]
        ev.eval_all(Z, 1.0, mu, None, None, *bufs)
        outs[tol] = bufs
        ev.close()
    for a, b in zip(outs["0"], outs["1e-14"]):
        assert np.isfinite(a).all() and relerr(a, b) <= 1e-11


def test_absurd_drive_poisons_a_planned_interval():
    """The series plan sums in FP32: a drive amplitude that overflows it (or is NaN) must still end as NaN outputs of that
    interval, not as a short series over a huge generator."""
    prob = pt.quantum_gate_problem(N=6, levels=16, n_drives=4)
    ev = dto.Evaluator(prob)
    spec = prob.to_spec()
    z, u_off = spec["z"], spec["components"]["u"][0]
    for bad in (1e200, np.nan):
        Z = prob.trajectory.vec().copy()
        Z[3 * z + u_off] = bad
        g = np.empty(ev.n_constraints)
        ev.eval_constraint(g, Z)
        n = prob.integrators[0].x_dim
        assert np.isnan(g[3 * n:4 * n]).all() and np.isfinite(g[:3 * n]).all() and np.isfinite(g[4 * n:5 * n]).all()
    ev.close()

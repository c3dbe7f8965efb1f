"""Iterate cache and registered outputs (SURVEY.md section 8 row a2 / 8b "Z de-duplication inside the handle").

The reference copies Z in every callback (src/solvers/evaluator.jl:474-482) and Ipopt / MadNLP call the five callbacks
separately on one iterate (src/solvers/ipopt_solver/solver.jl:85; benchmark/benchmarks.jl:23-38 times them separately).
Here the five calls on one iterate cost one upload, one mu-independent interval pass and one adjoint pass, and their
outputs are bit-identical to the fused dto_eval_all."""
import numpy as np
import pytest

import dto_b200 as dto
from dto_b200 import problem_templates as pt

pytestmark = pytest.mark.gpu


def _five_calls(ev, Z, sigma, mu):
    g, jac, hess, grad = np.full(ev.n_constraints, np.nan), np.full(ev.nnz_jacobian, np.nan), np.full(ev.nnz_hessian, np.nan), np.full(ev.n_vars, np.nan)
    J = ev.eval_objective(Z)
    ev.eval_objective_gradient(grad, Z)
    ev.eval_constraint(g, Z)
    ev.eval_constraint_jacobian(jac, Z)
    ev.eval_hessian_lagrangian(hess, Z, sigma, mu)
    return J, grad, g, jac, hess


def _fused(ev, Z, sigma, mu):
    J, grad = np.empty(1), np.empty(ev.n_vars)
    g, jac, hess = np.empty(ev.n_constraints), np.empty(ev.nnz_jacobian), np.empty(ev.nnz_hessian)
    ev.eval_all(Z, sigma, mu, J, grad, g, jac, hess)
    return J[0], grad, g, jac, hess


PROBLEMS = {
    "gate_n32_persistent": lambda: pt.quantum_gate_problem(N=40, levels=16, n_drives=4),
    "gate_n32_pipelined": lambda: pt.quantum_gate_problem(N=700, levels=16, n_drives=4),
    "scaled_n8_octet": lambda: pt.scaled_problem(N=60, state_dim=8, n_controls=2, generator_scale=0.35),
    "scaled_n16_octet_long": lambda: pt.scaled_problem(N=3000, state_dim=16, n_controls=2, generator_scale=0.25),
    "scaled_n24_m3": lambda: pt.scaled_problem(N=9, state_dim=24, n_controls=3, generator_scale=0.5),
    "n16_theta12_stages": lambda: pt.scaled_problem(N=5, state_dim=16, n_controls=2, generator_scale=12.0),
    "standard_constraints": lambda: pt.standard_problem(N=10),       # generic kernel + knot constraints: no jets, two full passes
    "carrier_tdb": lambda: pt.carrier_problem(N=5, state_dim=8, n_drives=2),
    "global": lambda: pt.global_problem(N=7),
}


@pytest.mark.parametrize("name", list(PROBLEMS))
def test_five_callbacks_bit_identical_to_fused(name):
    prob = PROBLEMS[name]()
    ev = dto.Evaluator(prob)
    rng = np.random.default_rng(3)
    Z0 = prob.trajectory.vec()
    for it in range(3):  # three iterates: cache must follow the iterate
        Z = Z0 + 0.01 * it * rng.standard_normal(Z0.size)
        mu = rng.random(ev.n_constraints)
        h0, m0 = ev.cache_stats()
        l0 = ev.launch_count
        seq = _five_calls(ev, Z, 1.3, mu)
        h1, m1 = ev.cache_stats()
        assert (h1 - h0, m1 - m0) == (4, 1), name
        seq_launches = ev.launch_count - l0
        # a second multiplier estimate on the same iterate (what a solver's restoration / second-order correction does)
        mu2 = rng.random(ev.n_constraints)
        H2 = np.empty(ev.nnz_hessian)
        ev.eval_hessian_lagrangian(H2, Z, 0.4, mu2)
        fused = _fused(ev, Z, 1.3, mu)
        for a, b in zip(seq, fused):
            assert np.array_equal(np.asarray(a), np.asarray(b)), name
        assert np.array_equal(H2, _fused(ev, Z, 0.4, mu2)[4]), name
        # after the fused call the callbacks still answer correctly (its Hessian pass used another mu)
        H3 = np.empty(ev.nnz_hessian)
        ev.eval_hessian_lagrangian(H3, Z, 1.3, mu)
        assert np.array_equal(H3, seq[4]), name
    ev.close()


def test_interval_kernel_runs_once_per_iterate():
    """c2 shape: the sequence launches the interval kernel twice (mu-independent pass + adjoint pass), not five times."""
    prob = pt.quantum_gate_problem(N=300, levels=16, n_drives=4)
    ev = dto.Evaluator(prob)
    Z = prob.trajectory.vec()
    mu = np.random.default_rng(0).random(ev.n_constraints)
    _five_calls(ev, Z, 1.0, mu)  # warm
    Z2 = Z + 1e-3
    ev.kernel_timing(True)
    _five_calls(ev, Z2, 1.0, mu)
    _, n_interval_launches = ev.kernel_time_ms()
    ev.kernel_timing(False)
    assert n_interval_launches == 2
    ev.close()


@pytest.mark.parametrize("name", ["gate_n32_pipelined", "scaled_n16_octet_long", "gate_n32_persistent"])
def test_registered_outputs(name):
    """dto_register_outputs: structural constants written once, value-dependent entries per call; speculative delivery of
    the Jacobian during the constraint callback.  Bit-identical to unregistered buffers, over several iterates, and
    fewer bytes cross PCIe."""
    prob = PROBLEMS[name]()
    ev_ref, ev = dto.Evaluator(prob), dto.Evaluator(prob)
    jac, hess = np.full(ev.nnz_jacobian, np.nan), np.full(ev.nnz_hessian, np.nan)
    ev.register_outputs(jac, hess)
    rng = np.random.default_rng(5)
    Z0 = prob.trajectory.vec()
    for it in range(3):
        Z = Z0 + 0.01 * it * rng.standard_normal(Z0.size)
        mu = rng.random(ev.n_constraints)
        ref = _five_calls(ev_ref, Z, 1.1, mu)
        g, grad = np.empty(ev.n_constraints), np.empty(ev.n_vars)
        J = ev.eval_objective(Z)
        ev.eval_objective_gradient(grad, Z)
        ev.eval_constraint(g, Z)            # starts the Jacobian's delivery to `jac`
        ev.eval_constraint_jacobian(jac, Z)  # joins it
        b_jac = ev.last_d2h_bytes
        ev.eval_hessian_lagrangian(hess, Z, 1.1, mu)
        b_hess = ev.last_d2h_bytes
        for a, b in zip(ref, (J, grad, g, jac, hess)):
            assert np.array_equal(np.asarray(a), np.asarray(b)), (name, it)
        if name != "gate_n32_persistent":  # large problems: only the value-dependent part of the Hessian moves
            assert b_jac == 0 and b_hess < 0.5 * 8 * ev.nnz_hessian
        # fused call into the registered arrays
        ev.eval_all(Z + 1e-3, 1.1, mu, None, None, None, jac, hess)
        f = _fused(ev_ref, Z + 1e-3, 1.1, mu)
        assert np.array_equal(jac, f[3]) and np.array_equal(hess, f[4])
        # an unregistered buffer on the same handle is delivered whole
        other = np.full(ev.nnz_jacobian, np.nan)
        ev.eval_constraint_jacobian(other, Z + 1e-3)
        assert np.array_equal(other, f[3])
    ev.unregister_outputs()
    ev.eval_constraint_jacobian(jac, Z0)
    jr = np.empty(ev.nnz_jacobian)
    ev_ref.eval_constraint_jacobian(jr, Z0)
    assert np.array_equal(jac, jr)
    ev.close()
    ev_ref.close()


def test_eval_all_rejects_bad_buffers():
    prob = pt.standard_problem(N=6)
    ev = dto.Evaluator(prob)
    Z = prob.trajectory.vec()
    with pytest.raises(ValueError):
        ev.eval_all(Z, 1.0, np.ones(ev.n_constraints), None, None, None, np.empty(ev.nnz_jacobian - 1), None)
    with pytest.raises(ValueError):
        ev.eval_all(Z, 1.0, np.ones(ev.n_constraints), None, None, None, np.empty(ev.nnz_jacobian, np.float32), None)
    with pytest.raises(ValueError):
        ev.eval_all(Z, 1.0, np.ones(ev.n_constraints - 1), None, None, None, None, np.empty(ev.nnz_hessian))
    with pytest.raises(ValueError):
        ev.eval_constraint_jacobian_product(np.empty(ev.n_constraints), Z, np.ones(ev.n_vars - 1))
    ev.close()


def _objective(ev, Z):
    """Objective and gradient alone from the fused call."""
    J, grad = np.empty(1), np.empty(ev.n_vars)
    ev.eval_all(Z, 1.0, None, J, grad)
    return J[0], grad


def test_early_start_of_the_mu_independent_pass():
    """The first callback on a new iterate (objective or gradient) also starts the residual / Jacobian / jets pass and
    returns without waiting for it.  Whatever order the callbacks then come in -- including iterates that are dropped
    after the objective alone -- the outputs are those of the fused call on a second handle (which never starts early),
    bit for bit."""
    prob = pt.quantum_gate_problem(N=300, levels=16, n_drives=4)
    ev_ref = dto.Evaluator(prob)
    ev = dto.Evaluator(prob)
    jac_reg, hess_reg = np.full(ev.nnz_jacobian, np.nan), np.full(ev.nnz_hessian, np.nan)
    rng = np.random.default_rng(11)
    Z0 = prob.trajectory.vec()
    new = lambda: Z0 + 0.01 * rng.standard_normal(Z0.size)
    buf = lambda n: np.full(n, np.nan)
    for registered in (False, True):
        if registered:
            ev.register_outputs(jac_reg, hess_reg)
        # A: the solver's order
        Z, mu = new(), rng.random(ev.n_constraints)
        ref = _fused(ev_ref, Z, 1.2, mu)
        got = _five_calls(ev, Z, 1.2, mu)
        for a, b in zip(ref, got):
            assert np.array_equal(np.asarray(a), np.asarray(b))
        # B: line-search style -- objective / gradient alone on iterates that are then dropped, then a full sequence
        for _ in range(3):
            Zt = new()
            J_r, grad_r = _objective(ev_ref, Zt)
            grad_g = buf(ev.n_vars)
            assert ev.eval_objective(Zt) == J_r
            ev.eval_objective_gradient(grad_g, Zt)
            assert np.array_equal(grad_g, grad_r)
        for _ in range(6):  # the early start pauses after unused ones and comes back once the pass is asked for again
            Z, mu = new(), rng.random(ev.n_constraints)
            for a, b in zip(_fused(ev_ref, Z, 0.7, mu), _five_calls(ev, Z, 0.7, mu)):
                assert np.array_equal(np.asarray(a), np.asarray(b))
        # C: objective twice, then the Hessian straight away (its jets come from the early-started pass)
        Z, mu = new(), rng.random(ev.n_constraints)
        ref = _fused(ev_ref, Z, 1.0, mu)
        assert ev.eval_objective(Z) == ev.eval_objective(Z) == ref[0]
        Hg = buf(ev.nnz_hessian)
        ev.eval_hessian_lagrangian(Hg, Z, 1.0, mu)
        assert np.array_equal(Hg, ref[4])
        # D: objective, then the fused call on the same iterate
        Z, mu = new(), rng.random(ev.n_constraints)
        ev.eval_objective(Z)
        for a, b in zip(_fused(ev_ref, Z, 1.1, mu), _fused(ev, Z, 1.1, mu)):
            assert np.array_equal(np.asarray(a), np.asarray(b))
        # E: gradient first, then the Jacobian into an unregistered buffer, then the residual
        Z = new()
        ref = _fused(ev_ref, Z, 1.0, rng.random(ev.n_constraints))
        gg = buf(ev.n_vars)
        ev.eval_objective_gradient(gg, Z)
        jg = buf(ev.nnz_jacobian)
        ev.eval_constraint_jacobian(jg, Z)
        cg = buf(ev.n_constraints)
        ev.eval_constraint(cg, Z)
        assert np.array_equal(gg, ref[1]) and np.array_equal(jg, ref[3]) and np.array_equal(cg, ref[2])
    ev.unregister_outputs()
    ev.close()
    ev_ref.close()

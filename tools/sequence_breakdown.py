"""Wall time of each of the five callbacks on a new iterate (c2 by default), registered and plain output buffers, and of the
fused call.  Usage: python tools/sequence_breakdown.py [c2|c4]"""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
import dto_b200 as dto  # noqa: E402

wl = sys.argv[1] if len(sys.argv) > 1 else "c2"
prob = bench.build_problem(wl, 42)
rng = np.random.default_rng(0)


def run(register, reps=30):
    ev = dto.Evaluator(prob)
    Z = prob.trajectory.vec()
    pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
    Zs = [pin(Z + 1e-3 * i * rng.standard_normal(Z.size)) for i in range(3)]
    mus = [pin(rng.random(ev.n_constraints)) for _ in range(3)]
    grad, g = pin(np.empty(ev.n_vars)), pin(np.empty(ev.n_constraints))
    jac, hess = pin(np.empty(ev.nnz_jacobian)), pin(np.empty(ev.nnz_hessian))
    J = pin(np.empty(1))
    if register:
        ev.register_outputs(jac, hess)
    names = ["objective", "gradient", "constraint", "jacobian", "hessian"]
    acc = np.zeros(5)
    for i in range(reps + 5):
        z, m = Zs[i % 3], mus[i % 3]
        t = [time.perf_counter()]
        ev.eval_objective(z); t.append(time.perf_counter())
        ev.eval_objective_gradient(grad, z); t.append(time.perf_counter())
        ev.eval_constraint(g, z); t.append(time.perf_counter())
        ev.eval_constraint_jacobian(jac, z); t.append(time.perf_counter())
        ev.eval_hessian_lagrangian(hess, z, 1.0, m); t.append(time.perf_counter())
        if i >= 5:
            acc += np.diff(t)
    acc *= 1e3 / reps
    t0 = time.perf_counter()
    for i in range(reps):
        ev.eval_all(Zs[i % 3], 1.0, mus[i % 3], J, grad, g, jac, hess)
    fused = (time.perf_counter() - t0) * 1e3 / reps
    print(f"{wl} register={int(register)} sequence {acc.sum():.3f} ms = " +
          " + ".join(f"{n} {v:.3f}" for n, v in zip(names, acc)) + f" | fused {fused:.3f} ms, d2h {ev.last_d2h_bytes / 1e6:.1f} MB", flush=True)
    ev.close()


for reg in (True, False):
    run(reg)

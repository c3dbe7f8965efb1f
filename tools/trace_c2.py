"""Device timeline (DTO_B200_TRACE=1) of the fused host-pointer call and of the callback sequence at c2, registered outputs."""
import os, sys, time
os.environ["DTO_B200_TRACE"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import bench, dto_b200 as dto
prob = bench.build_problem("c2", 42)
ev = dto.Evaluator(prob)
rng = np.random.default_rng(0)
pin = lambda a: torch.from_numpy(a).pin_memory().numpy()
Z = prob.trajectory.vec()
Zs = [pin(Z + 1e-3 * i * rng.standard_normal(Z.size)) for i in range(3)]
mu = pin(rng.random(ev.n_constraints))
J, grad, g = pin(np.empty(1)), pin(np.empty(ev.n_vars)), pin(np.empty(ev.n_constraints))
jac, hess = pin(np.empty(ev.nnz_jacobian)), pin(np.empty(ev.nnz_hessian))
ev.register_outputs(jac, hess)
for i in range(6):
    t0 = time.perf_counter()
    ev.eval_all(Zs[i % 3], 1.0, mu, J, grad, g, jac, hess)
    print(f"fused wall {1e3 * (time.perf_counter() - t0):.3f} ms", file=sys.stderr)
for i in range(4):
    z = Zs[i % 3]
    t = [time.perf_counter()]
    ev.eval_objective(z); t.append(time.perf_counter())
    ev.eval_objective_gradient(grad, z); t.append(time.perf_counter())
    ev.eval_constraint(g, z); t.append(time.perf_counter())
    ev.eval_constraint_jacobian(jac, z); t.append(time.perf_counter())
    ev.eval_hessian_lagrangian(hess, z, 1.0, mu); t.append(time.perf_counter())
    print("sequence wall ms " + " ".join(f"{1e3 * d:.3f}" for d in np.diff(t)), file=sys.stderr)

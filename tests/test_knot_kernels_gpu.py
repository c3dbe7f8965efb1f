"""Every instantiation of the knot-side kernels against the oracle.

The kernels around the interval kernels are template families too, and the host picks one from the problem's shape:
the group width GS of the Hessian assembler (K3) and the objective kernel (K6) is 8, 16 or 32 lanes per knot (knot width
z <= 16, <= 24, wider), the assembler runs 8, 4, 2 or 1 groups per CTA (z x z tiles up to 64 KB, opt-in shared memory
above 48 KB), `Prog` is true when a knot program is among the terms, the objective is summed in two levels above 2048
owned knots, and from 256 intervals on the objective and knot-pair kernels run on a second stream beside the interval
kernels.  Each cell records the knot-side kernels the CUDA profiler sees over all its calls and asserts that they are
exactly the ones it is meant to reach; the coverage guard asserts that the cells together reached KNOT_KERNELS.

Wide knots are a small bilinear core (n = 4: generic interval kernel; n = 8: octet, which also writes the derivative
integrators' rows) plus extra components that only the knot terms read.  Every cell puts knot functions of
nv = 1, GS - 1, GS, GS + 1 and, where the knot is wide enough, more than 32 variables on the knot, so that the lane loops
wrap and the packed-pair cursor of the assembler jumps several rows per step."""
from dataclasses import dataclass, field

import numpy as np
import pytest

import dto_b200 as dto
import dto_oracle as orc
from dto_b200 import problem_templates as pt
from helpers import blocks
from helpers.jets import with_user_functions
from helpers.kernels import knot_kernels, norm as _norm

# These kernels evaluate the same closed forms as the oracle in FP64: anything above round-off is a bug.  Measured on a
# B200 (1000 W): every cell within 2.1e-14 of the oracle (octet z = 20 residual; sigma = 0 Hessian of the glob batch)
TOL = 1e-12
# the time-dependent integrator's own entries (left-knot cells) against the oracle's variational solve (test_parity_gpu.py);
# measured 1.7e-13
TDB_TOL = 1e-10

_GS = (8, 16, 32)
_B = ("false", "true")
KNOT_KERNELS = sorted(
    [f"hessian_assemble_kernel<{g}, {p}>" for g in _GS for p in _B]
    + [f"hessian_assemble_left_kernel<{g}, {p}>" for g in _GS for p in _B]
    + [f"objective_kernel<{g}, {p}>" for g in _GS for p in _B]
    + [f"knot_objective_pairs_kernel<{p}>" for p in _B]
    + [f"constraint_product_kernel<{p}>" for p in _B] + ["analytic_product_kernel"]
    + ["analytic_kernel<8>", "analytic_kernel<32>", "constraint_kernel", "knot_program_kernel"]
    + [f"global_grad_kernel<{p}>" for p in _B] + [f"global_hess_kernel<{p}>" for p in _B] + ["column_sum_kernel", "kg_sum_kernel"]
    + ["objective_chunk_kernel", "objective_reduce_kernel", "violation_kernel", "jac_product_kernel", "hpp_contract_kernel"])


@pytest.fixture(autouse=True)
def oracle_user_functions(monkeypatch):
    """the oracle evaluates KnotProgram terms by second-order jets of the user's own function (helpers/jets.py)"""
    with_user_functions(monkeypatch, orc)


def _gs(z):
    return 8 if z <= 16 else (16 if z <= 24 else 32)


@dataclass
class Cell:
    id: str
    core: str              # "generic" (n = 4) or "octet" (n = 8)
    z: int
    terms: str = "cat"     # "cat": catalogue knot terms; "prog": plus a program constraint and objective; "glob": plus
                           # global terms (catalogue); "globprog": global terms as programs
    N: int = 6
    batch: int = 1
    env: dict = field(default_factory=dict)
    big: bool = False      # Hessian and Jacobian compared on sampled knots
    kernels: tuple = ()


def _kernels(core, z, terms, N=6, batch=1, env=None):
    """the knot-side kernels of one cell's calls: fused eval_all, the five callbacks, sigma = 0, eval_all_dev, the violation,
    the Jacobian products (single problems of fewer than 2048 knots)"""
    gs = _gs(z)
    prog = terms in ("prog", "globprog")
    glob = terms in ("glob", "globprog")
    k = {f"hessian_assemble_kernel<{gs}, {'true' if prog else 'false'}>", f"objective_kernel<{gs}, {'true' if prog else 'false'}>",
         "objective_reduce_kernel", "violation_kernel", "knot_objective_pairs_kernel<false>", "constraint_kernel"}
    if prog:
        k |= {"knot_objective_pairs_kernel<true>", "knot_program_kernel"}
    if N > 2048:
        k.add("objective_chunk_kernel")
    if core == "generic":
        k.add("analytic_kernel<8>" if 2 * z * 2 <= 64 else "analytic_kernel<32>")
    else:
        k.add("hpp_contract_kernel")  # the Hessian callback contracts the jets the residual callback kept
    if glob:
        p = "true" if terms == "globprog" else "false"
        k |= {f"global_grad_kernel<{p}>", f"global_hess_kernel<{p}>", "column_sum_kernel", "kg_sum_kernel"}
    if N >= 2048 or batch > 1:
        pass
    elif core == "octet" and not glob and not (env or {}).get("DTO_B200_JVP"):
        k |= {"analytic_product_kernel", "constraint_product_kernel<false>"} | ({"constraint_product_kernel<true>"} if prog else set())
    else:
        k.add("jac_product_kernel")
    return tuple(sorted(k))


def _cell(core, z, terms="cat", N=6, batch=1, env=None, tag=""):
    cid = f"{core}_z{z}_{terms}" + ("" if N == 6 else f"_N{N}") + ("" if batch == 1 else f"_B{batch}") + tag
    return Cell(cid, core, z, terms, N, batch, env or {}, N >= 2048, _kernels(core, z, terms, N, batch, env))


CELLS = (
    # group widths at their boundaries (z = 16 | 17, 24 | 25) and the groups per CTA: W = 4 (z = 37), 2 (z = 50), 1 (z = 70),
    # opt-in shared memory (z = 100); analytic_kernel<8> up to z = 16
    [_cell("generic", z) for z in (16, 17, 24, 25, 37, 50, 70, 100)]
    # octet core: the derivative rows come out of the interval kernel, matrix-free products; materialised under JVP=materialize
    + [_cell("octet", z) for z in (16, 20, 40)] + [_cell("octet", 16, env={"DTO_B200_JVP": "materialize"}, tag="_materialize")]
    # knot programs (the Prog = true twins) at every group width
    + [_cell("generic", 16, "prog"), _cell("octet", 24, "prog"), _cell("generic", 50, "prog"), _cell("octet", 16, "prog")]
    # global variables, catalogue and programs; three terms couple (x, x_goal) at knot 3
    + [_cell("generic", z, "glob") for z in (16, 24, 37)] + [_cell("generic", 16, "globprog"), _cell("generic", 25, "globprog")]
    # batches
    + [_cell("generic", 17, "glob", batch=3), _cell("octet", 20, "prog", batch=3)]
    # 2048 owned knots (one-level sum) and 2049 (two levels), with a batch; objective and knot pairs on the second stream
    + [_cell("generic", 16, N=2048), _cell("generic", 16, N=2049), _cell("generic", 16, N=2049, batch=3)]
)


# ---- problems -------------------------------------------------------------------------------------------------------------
def _pick(dims, nv):
    """component names (trajectory order) whose widths add up to nv"""
    best = {0: []}
    for name, d in dims.items():
        for s, names in list(best.items()):
            if s + d <= nv and s + d not in best:
                best[s + d] = names + [name]
    assert nv in best, (dims, nv)
    return best[nv]


def _prog_con(v, p):
    n = v.size
    return [np.sqrt(v @ v + 1.0) * np.cos(v[0]) - p[0], v[0] * v[n - 1] + np.tanh(v[n // 2]) - np.exp(0.3 * v[1 % n]) / (2.0 + v[0] ** 2)]


def _prog_obj(v, p):
    n = v.size
    return p[0] * (v @ v) + np.sin(v[0]) * v[n - 1] ** 2 + np.log(2.0 + v[n // 2] ** 2)


def _problem(cell, seed=3):
    rng = np.random.default_rng(seed)
    N = cell.N
    if cell.core == "generic":
        G, t0 = pt.bilinear_dynamics_and_trajectory(N=N, seed=seed)

        def integrators(t):
            return [dto.BilinearIntegrator(G, "x", "u", t), dto.DerivativeIntegrator("u", "du", t), dto.DerivativeIntegrator("du", "ddu", t)]
    else:
        base = pt.scaled_problem(N=N, state_dim=8, n_controls=2, seed=seed, generator_scale=0.35)
        t0, G = base.trajectory, base.integrators[0].G

        def integrators(t):
            return [dto.BilinearIntegrator((G[0], list(G[1:])), "x", "u", t), dto.DerivativeIntegrator("u", "du", t)]
    comps = {n: t0.data[t0.components[n], :] for n in t0.names}
    e = cell.z - t0.dim
    assert e >= 2
    # e - 1 extra variables in components of 1, 2, 4, ... entries (every function width is a sum of whole components)
    # and one more, s, away from zero
    rest, width = e - 1, 1
    while rest:
        comps[f"w{width}"] = rng.uniform(-1.0, 1.0, (min(width, rest), N))
        rest -= min(width, rest)
        width *= 2
    comps["s"] = rng.uniform(0.5, 1.5, (1, N))
    wide = max((n for n in comps if n.startswith("w")), key=lambda n: comps[n].shape[0])
    glob = cell.terms in ("glob", "globprog")
    nx = t0.dims["x"]
    gcomps = {"g": rng.uniform(0.5, 1.0, 3), "x_goal": rng.standard_normal(nx)} if glob else None
    traj = dto.NamedTrajectory(comps, controls=("dt",), timestep="dt", global_components=gcomps)
    assert traj.dim == cell.z
    dims = {n: traj.dims[n] for n in traj.names if n != "dt"}
    gs = _gs(cell.z)
    targets = sorted({min(v, cell.z - 1) for v in (1, gs - 1, gs, gs + 1, 35)})
    nvs = [targets[i % len(targets)] for i in range(10)]
    even = lambda v: max(2, v - v % 2)
    some = [1, 3, N] if N > 3 else [1, N]
    mid = list(range(2, N))

    def names(nv):
        return _pick(dims, nv)

    def qs(n):
        return rng.uniform(0.5, 2.0, n)

    # objective: every catalogue knot function, the regularizers and minimum time
    nv = nvs[0]
    J = dto.KnotPointObjective(dto.NormSqPlus(per_time=rng.uniform(0.1, 1.0, N)), names(nv), traj, Qs=qs(N))
    nv = nvs[1]
    J = J + 0.5 * dto.KnotPointObjective(dto.SqDist(rng.standard_normal(nv)), names(nv), traj, times=some, Qs=qs(len(some)))
    nv = nvs[2]
    J = J + dto.KnotPointObjective(dto.LinearCost(rng.standard_normal(nv)), names(nv), traj, times=mid, Qs=qs(len(mid)))
    nv = even(nvs[3])
    goal = rng.standard_normal(nv)
    J = J + dto.KnotPointObjective(dto.IsoInfidelity(goal / np.linalg.norm(goal)), names(nv), traj, times=some, Qs=qs(len(some)))
    nv = even(nvs[4])
    J = J + 1.5 * dto.KnotPointObjective(dto.SplitSqDist(), names(nv), traj, Qs=qs(N))
    nw = traj.dims[wide]
    J = J + dto.QuadraticRegularizer(wide, traj, rng.uniform(0.2, 1.0, nw), baseline=rng.standard_normal((nw, N)), times=some)
    J = J + dto.QuadraticRegularizer("u", traj, rng.uniform(0.2, 1.0, 2))
    J = J + 0.7 * dto.LinearRegularizer("du", traj, rng.standard_normal(2), times=some)
    J = J + 2.0 * dto.MinimumTimeObjective(traj, D=0.7)
    # constraints: every catalogue knot function, equality and inequality
    A = rng.standard_normal((2, nvs[8]))
    A[1, 0] = 0.0  # never stored: the reference drops the zero derivative
    cons = [
        dto.NonlinearKnotPointConstraint(dto.NormMinus(1.0), names(nvs[5]), traj, times=mid, equality=False),
        dto.NonlinearKnotPointConstraint(dto.NormSqMinus(0.5), names(nvs[6]), traj, times=some, equality=True),
        dto.NonlinearKnotPointConstraint(dto.SqDistMinus(rng.standard_normal(nvs[7]), 0.1), names(nvs[7]), traj, equality=False),
        dto.NonlinearKnotPointConstraint(dto.LinearMap(A, rng.standard_normal(2)), names(nvs[8]), traj, times=some, equality=True),
        dto.NonlinearKnotPointConstraint(dto.NormProduct(even(nvs[9]) // 2, 1.0, 0.5), names(even(nvs[9])), traj, times=mid, equality=False),
    ]
    if cell.terms == "prog":
        nv = nvs[3]
        J = J + dto.KnotPointObjective(dto.KnotProgram(_prog_obj, per_time=rng.uniform(0.5, 1.5, (len(some), 1))), names(nv), traj,
                                       times=some, Qs=qs(len(some)))
        cons.append(dto.NonlinearKnotPointConstraint(dto.KnotProgram(_prog_con, per_time=rng.uniform(0.5, 1.5, (len(mid), 1))),
                                                     names(nvs[4]), traj, times=mid, equality=False))
    if glob:
        J, cons = _global_terms(cell, traj, J, cons, rng, names(nvs[1]))
    return dto.DirectTrajOptProblem(traj, J, integrators(traj), constraints=cons)


def _global_terms(cell, traj, J, cons, rng, knot_names):
    """the four global term kinds; three terms and the terminal objective couple (x, x_goal) at knot 3 / N"""
    N = traj.N
    if cell.terms == "glob":
        gobj, gknot, split = dto.NormSqPlus(0.3), dto.NormSqPlus(0.0), dto.SplitSqDist()
        gcon, gknotcon = dto.NormMinus(1.0), dto.NormProduct(sum(traj.dims[n] for n in knot_names), 1.0, 1.0)
    else:
        gobj = dto.KnotProgram(lambda v: v @ v + np.sin(v[0]))
        gknot = dto.KnotProgram(lambda v: (v @ v) * np.exp(0.1 * v[-1]))
        split = dto.KnotProgram(lambda v: (v[: v.size // 2] - v[v.size // 2:]) @ (v[: v.size // 2] - v[v.size // 2:]) + 0.1 * v[0] * v[-1])
        gcon = dto.KnotProgram(lambda v: [v @ v - 1.0, np.tanh(v[0]) * v[-1]])
        nk = sum(traj.dims[n] for n in knot_names)
        gknotcon = dto.KnotProgram(lambda v: [np.sqrt(v[:nk] @ v[:nk]) - 1.0, np.sqrt(v[:nk] @ v[:nk]) * np.sqrt(v[nk:] @ v[nk:]) - 1.0])
    J = J + dto.GlobalObjective(gobj, "g", traj, Q=2.0)
    J = J + 0.5 * dto.GlobalKnotPointObjective(gknot, knot_names, ["g"], traj, times=[1, N], Qs=[1.0, 2.0])
    for q in rng.uniform(0.5, 3.0, 3):
        J = J + dto.GlobalKnotPointObjective(split, "x", "x_goal", traj, times=[3, N], Qs=[q, 0.5 * q])
    J = J + dto.TerminalObjective(split, "x", traj, global_names="x_goal", Q=10.0)
    cons = cons + [dto.NonlinearGlobalKnotPointConstraint(gknotcon, knot_names, ["g"], traj, equality=False),
                   dto.NonlinearGlobalConstraint(gcon, "g", traj, equality=False)]
    return J, cons


# ---- comparisons ----------------------------------------------------------------------------------------------------------
def _obj_scale(spec, Z):
    """max(1, sum over terms and listed knots of |w J_k|): what the order of the objective's sum can change"""
    s = 0.0
    for ob in spec["objectives"]:
        w = ob.get("weight", 1.0)
        if ob["kind"] == "mintime":
            s += abs(w * ob["D"]) * np.abs(Z[np.arange(spec["N"] - 1) * spec["z"] + orc.dt_offset(spec)]).sum()
            continue
        for i, k in enumerate(ob["times"]):
            one = dict(ob, times=[k])
            if ob["kind"] in ("knot", "global_knot"):
                one["params"], one["Qs"] = [ob["params"][i]], [ob["Qs"][i]]
            s += abs(w * orc._objective_term(spec, one, Z, False, False)[0])
    return max(1.0, s)


def _grad_block_relerr(spec, got, ref):
    """per trajectory component (all knots) and per global variable: max|got - ref| / max|ref| of the block"""
    z, N = spec["z"], spec["N"]
    comp, nc = blocks._component_of_column(spec)
    n = ref.size
    idx = np.arange(n)
    grp = np.where(idx < N * z, comp[np.minimum(idx % z, z - 1)], nc + idx - N * z)
    gid, gerr = blocks._group_max(grp, np.abs(got - ref))
    _, gmag = blocks._group_max(grp, np.abs(ref))
    whole = max(np.abs(ref).max(), 1e-300)
    return float((gerr / np.where(gmag > 0, gmag, whole)).max())


def relerr(got, ref):
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-300)) if ref.size else 0.0


def _iterate(prob, rng, noise=0.05):
    spec = prob.to_spec()
    Z0 = prob.trajectory.vec()
    Z = Z0 + noise * rng.standard_normal(Z0.size)
    dts = slice(orc.dt_offset(spec), spec["N"] * spec["z"], spec["z"])
    Z[dts] = np.abs(Z[dts])
    return Z


def _dev_eval(ev, Z, sigma, mu):
    """eval_all_dev into device buffers, then the violation of the device residual; (outputs, violation) read back"""
    import torch

    dev = torch.device("cuda", torch.cuda.current_device())
    B = ev.batch
    n_grad = ev.shard_layout.z_end - ev.shard_layout.z_begin + ev.global_dim
    dZ, dmu = torch.from_numpy(np.ascontiguousarray(Z).ravel()).to(dev), torch.from_numpy(np.ascontiguousarray(mu).ravel()).to(dev)
    outs = [torch.full((B * n,), float("nan"), dtype=torch.float64, device=dev)
            for n in (1, n_grad, ev.n_constraints, ev.nnz_jacobian, ev.nnz_hessian)]
    viol = torch.full((B,), float("nan"), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    ev.eval_all_dev(dZ.data_ptr(), sigma, dmu.data_ptr(), *[o.data_ptr() for o in outs])
    ev.violation_dev(outs[2].data_ptr(), viol.data_ptr())
    ev.synchronize()
    return [o.cpu().numpy().reshape(B, -1) for o in outs], viol.cpu().numpy()


_SEEN = {}  # cell id -> knot-side kernels seen in its profiled calls


def _record(cid, seen, declared, worst):
    _SEEN[cid] = seen
    print(f"\n{cid}: worst relative error " + " ".join(f"{k}={v:.1e}" for k, v in worst.items()) + f"  kernels={sorted(seen)}")
    assert seen == {_norm(k) for k in declared}, (cid, sorted(seen - {_norm(k) for k in declared}), sorted({_norm(k) for k in declared} - seen))


@pytest.mark.gpu
@pytest.mark.parametrize("cell", CELLS, ids=lambda c: c.id)
def test_knot_kernels_match_oracle(cell, monkeypatch):
    for k, v in cell.env.items():
        monkeypatch.setenv(k, v)
    B = cell.batch
    prob = _problem(cell)
    spec = prob.to_spec()
    ev = dto.Evaluator(prob, batch=B)
    rng = np.random.default_rng(7)
    Z0 = prob.trajectory.vec()
    jst, hst = orc.jacobian_structure(spec, Z0), orc.hessian_structure(spec, Z0)
    jr, jc = ev.jacobian_structure()
    hr, hc = ev.hessian_lagrangian_structure()
    assert np.array_equal(jr, jst[0]) and np.array_equal(jc, jst[1]) and np.array_equal(hr, hst[0]) and np.array_equal(hc, hst[1])
    nc, nv, nj, nh = ev.n_constraints, ev.n_vars, ev.nnz_jacobian, ev.nnz_hessian
    Z = np.stack([_iterate(prob, rng) for _ in range(B)])
    mu = rng.random((B, nc))
    res = {}

    def nan(*shape):
        return np.full(shape, np.nan)

    def device():
        fused = [nan(B), nan(B, nv), nan(B, nc), nan(B, nj), nan(B, nh)]
        ev.eval_all(Z, 1.3, mu, *fused)
        # the five callbacks in the order a solver calls them, then the sigma = 0 Hessian
        sep = [nan(B), nan(B, nv), nan(B, nc), nan(B, nj), nan(B, nh)]
        sep[0][:] = ev.eval_objective(Z)
        ev.eval_objective_gradient(sep[1], Z)
        ev.eval_constraint(sep[2], Z)
        ev.eval_constraint_jacobian(sep[3], Z)
        ev.eval_hessian_lagrangian(sep[4], Z, 1.3, mu)
        H0 = nan(B, nh)
        ev.eval_hessian_lagrangian(H0, Z, 0.0, mu)
        reps = []
        for _ in range(3):  # repeated Hessians of one iterate: bit-identical (no atomics in any sum)
            H = nan(B, nh)
            ev.eval_all(Z, 1.3, mu, None, None, None, None, H)
            reps.append(H)
        res.update(fused=fused, sep=sep, H0=H0, reps=reps, dev=_dev_eval(ev, Z, 1.3, mu))
        if B == 1 and not cell.big:  # products against the oracle's dense Jacobian: not at 2048 knots
            w1, w2 = rng.standard_normal(nv), rng.standard_normal(nc)
            y1, y2 = nan(nc), nan(nv)
            ev.eval_constraint_jacobian_product(y1, Z[0], w1)
            ev.eval_constraint_jacobian_transpose_product(y2, Z[0], w2)
            res["prod"] = (w1, w2, y1, y2)

    seen = knot_kernels(device)
    fused, sep, H0, reps, (dev, viol) = res["fused"], res["sep"], res["H0"], res["reps"], res["dev"]
    for a, b in zip(fused, sep):  # fused and separate callbacks: bit for bit
        assert np.array_equal(a, b), cell.id
    for a, b in zip(fused, dev):  # host and device pointers
        assert np.array_equal(a.reshape(B, -1), b), cell.id
    for H in reps:
        assert np.array_equal(H, fused[4]), cell.id

    worst = {}

    def check(key, e):
        worst[key] = max(worst.get(key, 0.0), e)
        assert e <= TOL, (cell.id, key, e)

    for b in range(B):
        Zb, mub = Z[b], mu[b]
        Jr = orc.eval_objective(spec, Zb)
        check("obj", abs(fused[0][b] - Jr) / _obj_scale(spec, Zb))
        gr = orc.eval_objective_gradient(spec, Zb)
        check("grad", max(relerr(fused[1][b], gr), _grad_block_relerr(spec, fused[1][b], gr)))
        if cell.big:
            ks = sorted({1, 2, 3, 1024, 2047, cell.N - 1, cell.N} | {int(k) for k in rng.integers(1, cell.N + 1, size=6)})
            for sigma, H in ((1.3, fused[4][b]), (0.0, H0[b])):
                er, ej, eh = blocks.sampled_interval_check(spec, Zb, sigma, mub, fused[2][b], fused[3][b], H, ks, jac_structure=(jr, jc))
                check("g", er)
                check("jac", ej)
                check("hess" if sigma else "hess0", eh)
            nd, _ = orc.n_constraints(spec)
            gcon = np.concatenate([orc._cfun(c["fn"], Zb[orc.term_indices(spec, c, k)], np.atleast_1d(c["params"][i]))[0]
                                   for c in spec["constraints"] for i, k in enumerate(c["times"])])
            check("g", max(relerr(fused[2][b][nd:], gcon), blocks.vec_block_relerr(spec, fused[2][b], np.r_[fused[2][b][:nd], gcon])))
            gref = np.r_[fused[2][b][:nd], gcon]
        else:
            gref = orc.eval_constraint(spec, Zb)
            check("g", max(relerr(fused[2][b], gref), blocks.vec_block_relerr(spec, fused[2][b], gref)))
            jref = orc.eval_constraint_jacobian(spec, Zb, jst)
            check("jac", max(relerr(fused[3][b], jref), blocks.jac_block_relerr(spec, jst, fused[3][b], jref)))
            for key, sigma, H in (("hess", 1.3, fused[4][b]), ("hess0", 0.0, H0[b])):
                href = orc.eval_hessian_lagrangian(spec, Zb, sigma, mub, hst)
                check(key, max(relerr(H, href), blocks.hess_block_relerr(spec, hst, H, href)))
        # the violation reduction against the oracle's residual: |g| on equality rows, max(0, g) on inequality rows
        v, _ = orc.violation(spec, gref)
        check("viol", abs(viol[b] - v.max()) / max(np.abs(gref).max(), 1e-300))

    if "prod" in res:
        w1, w2, y1, y2 = res["prod"]
        jref = orc.eval_constraint_jacobian(spec, Z[0], jst)
        Jd = np.zeros((nc, nv))
        np.add.at(Jd, (jst[0] - 1, jst[1] - 1), jref)
        # error scale: sum |J_ij| |w_j| bounds what the summation order can change
        check("prod", np.abs(y1 - Jd @ w1).max() / (np.abs(Jd) @ np.abs(w1)).max())
        check("prod", np.abs(y2 - Jd.T @ w2).max() / (np.abs(Jd.T) @ np.abs(w2)).max())
    ev.close()
    _record(cell.id, seen, cell.kernels, worst)


# ---- a knot-range shard that owns more than 2048 knots --------------------------------------------------------------------
SHARD_KERNELS = ("hessian_assemble_kernel<8, false>", "objective_kernel<8, false>", "objective_chunk_kernel", "objective_reduce_kernel",
                 "knot_objective_pairs_kernel<false>", "constraint_kernel", "analytic_kernel<8>")


@pytest.mark.gpu
def test_shard_owning_more_than_2048_knots():
    """knots 1..2049 of a 2100-knot problem: the shard's objective takes the two-level sum over its own knots; its rows,
    Jacobian and Hessian entries are those of the whole-problem evaluation"""
    cell = Cell("shard", "generic", 16, N=2100)
    prob = _problem(cell)
    spec = prob.to_spec()
    rng = np.random.default_rng(8)
    Z = _iterate(prob, rng)
    whole = dto.Evaluator(prob)
    mu = rng.random(whole.n_constraints)
    ref = [np.empty(1), np.empty(whole.n_vars), np.empty(whole.n_constraints), np.empty(whole.nnz_jacobian), np.empty(whole.nnz_hessian)]
    whole.eval_all(Z, 1.3, mu, *ref)
    sh = dto.Evaluator(prob, shard=(1, 2049))
    L = sh.shard_layout
    rows, jpos, hpos = sh.shard_maps()
    out = [np.empty(1), np.empty(L.z_end - L.z_begin), np.empty(sh.n_constraints), np.empty(sh.nnz_jacobian), np.empty(sh.nnz_hessian)]
    seen = knot_kernels(lambda: sh.eval_all(Z[L.z_begin:L.z_halo_end], 1.3, mu[rows], *out))
    assert np.array_equal(out[2], ref[2][rows]) and np.array_equal(out[3], ref[3][jpos]) and np.array_equal(out[4], ref[4][hpos])
    assert np.array_equal(out[1], ref[1][L.z_begin:L.z_end])
    Jr = orc.objective_by_knot(spec, Z)[:2049].sum()
    e_obj = abs(out[0][0] - Jr) / _obj_scale(spec, Z)
    gr = orc.eval_objective_gradient(spec, Z)
    e_grad = max(relerr(out[1], gr[L.z_begin:L.z_end]), _grad_block_relerr(spec, ref[1], gr))
    assert e_obj <= TOL and e_grad <= TOL, (e_obj, e_grad)
    sh.close()
    whole.close()
    _record("shard_2049_of_2100", seen, SHARD_KERNELS, {"obj": e_obj, "grad": e_grad})


# ---- the left-knot assembler of linked linear-spline shards ---------------------------------------------------------------
LEFT_CELLS = [(n, m, prog) for n, m in ((8, 1), (12, 2), (24, 2)) for prog in (False, True)]


def _left_kernels(n, m, prog):
    z = n + 3 * m + 2
    gs, p = _gs(z), "true" if prog else "false"
    return tuple(sorted({f"hessian_assemble_kernel<{gs}, {p}>", f"hessian_assemble_left_kernel<{gs}, {p}>", f"objective_kernel<{gs}, false>",
                         "objective_reduce_kernel", "constraint_kernel", "analytic_kernel<8>" if 2 * z * m <= 64 else "analytic_kernel<32>"}
                        | ({"knot_program_kernel"} if prog else set())))


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,prog", LEFT_CELLS, ids=[f"n{c[0]}_m{c[1]}" + ("_prog" if c[2] else "") for c in LEFT_CELLS])
def test_left_knot_assembler(n, m, prog):
    """linked shards of a linear-spline time-dependent bilinear problem: a shard that starts after knot 1 assembles its first
    knot in its own launch (hessian_assemble_left_kernel) after the left neighbour's block arrived; the reassembled arrays
    are the whole problem's bit for bit, and the whole problem matches the oracle"""
    N = 9
    base = pt.carrier_problem(N=N, state_dim=n, n_drives=m, spline_order=1, dt=0.2)
    traj = base.trajectory
    cons = list(base.constraints)
    if prog:
        cons.append(dto.NonlinearKnotPointConstraint(dto.KnotProgram(_prog_con, params=[0.8]), ["u", "du"], traj, times=range(2, N), equality=True))
    prob = dto.DirectTrajOptProblem(traj, base.objective, base.integrators, constraints=cons)
    assert traj.dim == n + 3 * m + 2
    spec = prob.to_spec()
    rng = np.random.default_rng(9)
    Z = _iterate(prob, rng, noise=0.02)
    whole = dto.Evaluator(prob)
    mu = rng.random(whole.n_constraints)
    ref = [np.empty(1), np.empty(whole.n_vars), np.empty(whole.n_constraints), np.empty(whole.nnz_jacobian), np.empty(whole.nnz_hessian)]
    whole.eval_all(Z, 1.3, mu, *ref)
    cuts = [(1, 3), (4, 4), (5, N - 1), (N, N)]
    shards = [dto.Evaluator(prob, shard=c) for c in cuts]
    dto.Evaluator.shard_link_local(shards)
    grad, g = np.full(whole.n_vars, np.nan), np.full(whole.n_constraints, np.nan)
    jac, hess = np.full(whole.nnz_jacobian, np.nan), np.full(whole.nnz_hessian, np.nan)
    J = 0.0

    def run():
        nonlocal J
        locs = []
        for sh in shards:
            L = sh.shard_layout
            Zl = Z[L.z_begin:L.z_halo_end].copy()
            if L.z_halo_end > L.z_end:
                Zl[L.z_end - L.z_begin:] = np.nan  # linked shards read the neighbour's window, never the local halo
            sh.upload(Zl)
            locs.append(Zl)
        for sh, Zl in zip(shards, locs):
            L = sh.shard_layout
            rows, jpos, hpos = sh.shard_maps()
            o = [np.empty(1), np.empty(L.z_end - L.z_begin), np.empty(sh.n_constraints), np.empty(sh.nnz_jacobian), np.empty(sh.nnz_hessian)]
            sh.eval_all(Zl, 1.3, mu[rows], *o)
            J += o[0][0]
            grad[L.z_begin:L.z_end] = o[1]
            g[rows], jac[jpos], hess[hpos] = o[2], o[3], o[4]

    seen = knot_kernels(run)
    assert np.array_equal(grad, ref[1]) and np.array_equal(g, ref[2]) and np.array_equal(jac, ref[3]) and np.array_equal(hess, ref[4])
    hst = orc.hessian_structure(spec, traj.vec())
    href = orc.eval_hessian_lagrangian(spec, Z, 1.3, mu, hst)
    e_h = blocks.hess_block_relerr(spec, hst, ref[4], href)
    e_obj = abs(J - orc.eval_objective(spec, Z)) / _obj_scale(spec, Z)
    gr = orc.eval_objective_gradient(spec, Z)
    e_grad = _grad_block_relerr(spec, grad, gr)
    assert e_h <= TDB_TOL and e_obj <= TOL and e_grad <= TOL, (e_h, e_obj, e_grad)
    for e in shards + [whole]:
        e.close()
    _record(f"left_n{n}_m{m}" + ("_prog" if prog else ""), seen, _left_kernels(n, m, prog), {"obj": e_obj, "grad": e_grad, "hess": e_h})


_ALL_IDS = [c.id for c in CELLS] + ["shard_2049_of_2100"] + [f"left_n{n}_m{m}" + ("_prog" if p else "") for n, m, p in LEFT_CELLS]
_ALL_DECLARED = [c.kernels for c in CELLS] + [SHARD_KERNELS] + [_left_kernels(*c) for c in LEFT_CELLS]


@pytest.mark.gpu
def test_every_declared_knot_kernel_ran():
    """A cell whose shape reaches another instantiation fails its own assertion; this guards the list itself: the union of
    what the profiler saw is exactly KNOT_KERNELS."""
    missing = set(_ALL_IDS) - set(_SEEN)
    if missing:
        pytest.skip(f"{len(missing)} cells did not complete in this session")
    union = set().union(*_SEEN.values())
    print("\nknot-side kernel union: " + ", ".join(sorted(union)))
    assert union == {_norm(k) for k in KNOT_KERNELS}, (sorted(union - {_norm(k) for k in KNOT_KERNELS}), sorted({_norm(k) for k in KNOT_KERNELS} - union))


def test_cells_declare_exactly_the_knot_kernel_list():
    declared = set()
    for ks in _ALL_DECLARED:
        declared |= {_norm(k) for k in ks}
    assert declared == {_norm(k) for k in KNOT_KERNELS}, (sorted(declared ^ {_norm(k) for k in KNOT_KERNELS}))
    assert len(set(_ALL_IDS)) == len(_ALL_IDS)


def test_cell_problems_have_the_declared_shapes():
    """the knot widths, the function widths relative to GS and the term kinds the cells are meant to carry"""
    for c in CELLS:
        if c.big:
            continue
        prob = _problem(c)
        spec = prob.to_spec()
        assert spec["z"] == c.z
        gs = _gs(c.z)
        widths = {sum(spec["components"][n][1] for n in t["names"]) for t in spec["objectives"] + spec["constraints"]
                  if t["kind"] in ("knot", "global_knot") and not callable(t["fn"])}
        want = {min(v, c.z - 1) for v in (1, gs - 1, gs, gs + 1)}
        assert want <= widths and (max(widths) > 32 or c.z <= 34), (c.id, sorted(widths))
        fns = {t["fn"] for t in spec["objectives"] + spec["constraints"] if t["kind"] == "knot" and not callable(t["fn"])}
        assert {"normsq_plus_p", "sqdist", "linear", "iso_infidelity", "split_sqdist", "norm_minus_c", "normsq_minus_c", "sqdist_minus_c",
                "norm_product"} <= fns, c.id

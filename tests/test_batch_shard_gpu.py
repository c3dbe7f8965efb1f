"""Multi-problem batches (BASELINE config c5) and knot-range shards with a one-knot halo (config c4),
exercised on ONE GPU: several handles in one process, linked with dto_shard_link_local (the same exchange-window
protocol as CUDA-IPC mapped peers: halo pushed into the neighbour's window, scalars exchanged through the windows)."""
import numpy as np
import pytest

import dto_b200 as dto
import dto_oracle as orc
from dto_b200 import problem_templates as pt

pytestmark = pytest.mark.gpu


def all_outputs(ev, Z, sigma, mu):
    J = np.empty(ev.batch)
    grad = np.empty(ev.batch * (ev.shard_layout.z_end - ev.shard_layout.z_begin))
    g, jac, hess = np.empty(ev.batch * ev.n_constraints), np.empty(ev.batch * ev.nnz_jacobian), np.empty(ev.batch * ev.nnz_hessian)
    ev.eval_all(Z, sigma, mu, J, grad, g, jac, hess)
    return J, grad, g, jac, hess


@pytest.mark.parametrize("builder", [lambda: pt.scaled_problem(N=9, state_dim=8, n_controls=2),
                                     lambda: pt.standard_problem(N=7),
                                     lambda: pt.scaled_problem(N=5, state_dim=5, n_controls=2, generator_scale=0.6)])
def test_batch_equals_independent_problems(builder):
    prob = builder()
    B = 5
    rng = np.random.default_rng(2)
    single = dto.Evaluator(prob)
    batched = dto.Evaluator(prob, batch=B)
    Z0 = prob.trajectory.datavec
    Zs = Z0[None, :] + 0.03 * rng.standard_normal((B, Z0.size))
    mus = rng.random((B, single.n_constraints))
    out_b = all_outputs(batched, Zs, 1.3, mus)
    for b in range(B):
        out_1 = all_outputs(single, Zs[b], 1.3, mus[b])
        for got, ref in zip(out_b, out_1):
            n = ref.size
            assert np.array_equal(got[b * n:(b + 1) * n], ref)
    single.close()
    batched.close()


@pytest.mark.parametrize("B,n,m,N,variant", [(4, 8, 2, 6, "octet"), (3, 8, 2, 20, "octet"), (3, 16, 2, 12, "octet"), (2, 8, 3, 10, "octet"),
                                             (2, 24, 2, 5, "dmma")])
def test_batch_with_per_problem_generators(B, n, m, N, variant):
    """Every problem of the batch brings its own generators: small states run the octet kernel with one problem per octet
    (partial last octets), the others the warp-per-interval tensor-core kernel."""
    rng = np.random.default_rng(5)
    prob = pt.scaled_problem(N=N, state_dim=n, n_controls=m)
    Gs = rng.standard_normal((B, m + 1, n, n)) * (8.0 / n)
    batched = dto.Evaluator(prob, batch=B, batch_G=Gs)
    assert batched.kernel_variant(0) == variant
    Z0 = prob.trajectory.datavec
    Zs = Z0[None, :] + 0.03 * rng.standard_normal((B, Z0.size))
    mus = rng.random((B, batched.n_constraints))
    out_b = all_outputs(batched, Zs, 1.0, mus)
    for b in range(B):
        pb = pt.scaled_problem(N=N, state_dim=n, n_controls=m)
        pb.integrators[0].G = Gs[b]
        spec = pb.to_spec()
        jst, hst = orc.jacobian_structure(spec, Z0), orc.hessian_structure(spec, Z0)
        ref = orc.eval_constraint_jacobian(spec, Zs[b], jst)
        got = out_b[3][b * ref.size:(b + 1) * ref.size]
        assert np.abs(got - ref).max() <= 1e-10 * np.abs(ref).max()
        ref = orc.eval_hessian_lagrangian(spec, Zs[b], 1.0, mus[b], hst)
        got = out_b[4][b * ref.size:(b + 1) * ref.size]
        assert np.abs(got - ref).max() <= 1e-10 * np.abs(ref).max()
    batched.close()


@pytest.mark.parametrize("builder,cuts", [
    (lambda: pt.scaled_problem(N=13, state_dim=8, n_controls=2), [(1, 4), (5, 9), (10, 13)]),
    (lambda: pt.standard_problem(N=11), [(1, 1), (2, 6), (7, 10), (11, 11)]),
    (lambda: pt.quantum_gate_problem(N=9, levels=8, n_drives=2), [(1, 5), (6, 9)]),
])
@pytest.mark.parametrize("peer_halo", [False, True])
def test_knot_range_shards_reassemble_the_whole_problem(builder, cuts, peer_halo):
    prob = builder()
    rng = np.random.default_rng(4)
    whole = dto.Evaluator(prob)
    Z0 = prob.trajectory.datavec
    Z = Z0 + 0.02 * rng.standard_normal(Z0.size)
    mu = rng.random(whole.n_constraints)
    sigma = 0.7
    Jw, gradw, gw, jacw, hessw = all_outputs(whole, Z, sigma, mu)
    shards = [dto.Evaluator(prob, shard=c) for c in cuts]
    if peer_halo:
        dto.Evaluator.shard_link_local(shards)
    J = 0.0
    grad = np.full_like(gradw, np.nan)
    g, jac, hess = np.full_like(gw, np.nan), np.full_like(jacw, np.nan), np.full_like(hessw, np.nan)
    jr, jc = whole.jacobian_structure()
    hr, hc = whole.hessian_lagrangian_structure()
    outs = []
    # two passes so that, with peer halos, every shard's resident Z is current before anyone reads a halo
    for sh in shards:
        L = sh.shard_layout
        Zloc = Z[L.z_begin:L.z_halo_end].copy()
        if peer_halo and L.z_halo_end > L.z_end:
            Zloc[L.z_end - L.z_begin:] = np.nan  # the local halo slot must not be read
        sh.upload(Zloc)  # uploads the shard's Z (linked shards: pushes the first knot into the left neighbour's window)
    for sh in shards:
        L = sh.shard_layout
        Zloc = Z[L.z_begin:L.z_halo_end].copy()
        if peer_halo and L.z_halo_end > L.z_end:
            Zloc[L.z_end - L.z_begin:] = np.nan
        rows, jpos, hpos = sh.shard_maps()
        out = all_outputs(sh, Zloc, sigma, mu[rows])
        J += out[0][0]
        grad[L.z_begin:L.z_end] = out[1]
        assert np.all(np.isnan(g[rows])) and np.all(np.isnan(jac[jpos])) and np.all(np.isnan(hess[hpos]))  # disjoint ownership
        g[rows], jac[jpos], hess[hpos] = out[2], out[3], out[4]
        sr, sc = sh.jacobian_structure()
        assert np.array_equal(sr, jr[jpos]) and np.array_equal(sc, jc[jpos])
        sr, sc = sh.hessian_lagrangian_structure()
        assert np.array_equal(sr, hr[hpos]) and np.array_equal(sc, hc[hpos])
    assert np.array_equal(grad, gradw) and np.array_equal(g, gw) and np.array_equal(jac, jacw) and np.array_equal(hess, hessw)
    assert abs(J - Jw[0]) <= 1e-13 * max(1.0, abs(Jw[0]))
    for e in shards + [whole]:
        e.close()


def test_violation_reduction():
    import torch

    prob = pt.standard_problem(N=9)
    ev = dto.Evaluator(prob)
    Z = prob.trajectory.datavec.copy()
    g = np.empty(ev.n_constraints)
    ev.eval_constraint(g, Z)
    lo, hi = ev.constraint_bounds()
    ref = max(np.abs(g[lo == 0]).max(), np.maximum(g[lo < 0], 0).max())
    dg = torch.from_numpy(g).cuda()
    dv = torch.zeros(1, dtype=torch.float64, device="cuda")
    ev.violation_dev(dg.data_ptr(), dv.data_ptr())
    ev.synchronize()
    assert dv.item() == ref
    # a residual the kernels poisoned with NaN is no feasible point: NaN in an equality row, then in an inequality row
    for row in (int(np.flatnonzero(lo == 0)[3]), int(np.flatnonzero(lo < 0)[1])):
        gn = g.copy()
        gn[row] = np.nan
        dg = torch.from_numpy(gn).cuda()
        ev.violation_dev(dg.data_ptr(), dv.data_ptr())
        ev.synchronize()
        assert np.isnan(dv.item()), row
    ev.close()


def test_linked_shards_follow_a_changing_iterate():
    """Solver-loop pattern on linked shards: every iterate is uploaded once on every shard, the halo knot of THAT iterate
    reaches the left neighbour through the exchange window (the local halo slot holds NaN), the five callbacks run on
    cache hits, and objective / violation are reduced through the windows.  Several iterates, so the double-buffered
    halo slots and the acknowledgements are exercised."""
    import torch

    prob = pt.scaled_problem(N=26, state_dim=8, n_controls=2, generator_scale=0.4)
    cuts = [(1, 7), (8, 8), (9, 20), (21, 26)]
    rng = np.random.default_rng(8)
    whole = dto.Evaluator(prob)
    shards = [dto.Evaluator(prob, shard=c) for c in cuts]
    dto.Evaluator.shard_link_local(shards)
    Z0 = prob.trajectory.datavec
    lo, _ = whole.constraint_bounds()
    for it in range(5):
        Z = Z0 + 0.02 * rng.standard_normal(Z0.size)
        mu = rng.random(whole.n_constraints)
        Jw, gradw, gw, jacw, hessw = all_outputs(whole, Z, 1.1, mu)
        locs = []
        for sh in shards:  # phase 1: every shard uploads the iterate
            L = sh.shard_layout
            Zloc = Z[L.z_begin:L.z_halo_end].copy()
            if L.z_halo_end > L.z_end:
                Zloc[L.z_end - L.z_begin:] = np.nan
            sh.upload(Zloc)
            locs.append(Zloc)
        g, jac, hess = np.full_like(gw, np.nan), np.full_like(jacw, np.nan), np.full_like(hessw, np.nan)
        dJs, dVs, dGs = [], [], []
        for sh, Zloc in zip(shards, locs):  # phase 2: the five callbacks, separately
            rows, jpos, hpos = sh.shard_maps()
            gl, jl, hl = np.empty(sh.n_constraints), np.empty(sh.nnz_jacobian), np.empty(sh.nnz_hessian)
            J = sh.eval_objective(Zloc)
            sh.eval_constraint(gl, Zloc)
            sh.eval_constraint_jacobian(jl, Zloc)
            sh.eval_hessian_lagrangian(hl, Zloc, 1.1, mu[rows])
            g[rows], jac[jpos], hess[hpos] = gl, jl, hl
            l2, _ = sh.constraint_bounds()
            viol = float(np.where(l2 == 0, np.abs(gl), np.maximum(gl, 0)).max()) if gl.size else 0.0
            dJs.append(torch.tensor([J], dtype=torch.float64, device="cuda"))
            dVs.append(torch.tensor([viol], dtype=torch.float64, device="cuda"))
            dGs.append(torch.from_numpy(gl).cuda())
        assert np.array_equal(g, gw) and np.array_equal(jac, jacw) and np.array_equal(hess, hessw), it
        torch.cuda.synchronize()
        for sh, dJ, dV in zip(shards, dJs, dVs):  # the scalar exchange: all ranks enqueue, then all synchronise
            sh.allreduce_scalars_dev(dJ.data_ptr(), dV.data_ptr())
        for sh in shards:
            sh.synchronize()
        vw = np.where(lo == 0, np.abs(gw), np.maximum(gw, 0)).max()
        tot = [float(t.item()) for t in dJs]
        assert all(t == tot[0] for t in tot) and abs(tot[0] - Jw[0]) <= 1e-13 * max(1.0, abs(Jw[0]))
        assert all(float(v.item()) == vw for v in dVs)
        # the fused form: violation of the shard's residuals + exchange in one kernel (dto_shard_scalars_dev), twice in a row
        for rep in range(2):
            dJ2 = [torch.tensor([float(sh.eval_objective(Zloc))], dtype=torch.float64, device="cuda") for sh, Zloc in zip(shards, locs)]
            dV2 = [torch.full((1,), -1.0, dtype=torch.float64, device="cuda") for _ in shards]
            torch.cuda.synchronize()
            for sh, dG, dJ, dV in zip(shards, dGs, dJ2, dV2):
                sh.shard_scalars_dev(dG.data_ptr(), dJ.data_ptr(), dV.data_ptr())
            for sh in shards:
                sh.synchronize()
            assert all(float(t.item()) == tot[0] for t in dJ2) and all(float(v.item()) == vw for v in dV2)
    # one shard's residuals hold a NaN: every rank reports the violation as NaN, from its own rows and from the exchange
    dGs[2][5] = float("nan")
    dJ3 = [torch.tensor([float(sh.eval_objective(Zloc))], dtype=torch.float64, device="cuda") for sh, Zloc in zip(shards, locs)]
    dV3 = [torch.full((1,), -1.0, dtype=torch.float64, device="cuda") for _ in shards]
    torch.cuda.synchronize()
    for sh, dG, dJ, dV in zip(shards, dGs, dJ3, dV3):
        sh.shard_scalars_dev(dG.data_ptr(), dJ.data_ptr(), dV.data_ptr())
    for sh in shards:
        sh.synchronize()
    assert all(np.isnan(float(v.item())) for v in dV3)
    dV4 = [torch.tensor([np.nan if i == 2 else 0.5], dtype=torch.float64, device="cuda") for i in range(len(shards))]
    dJ4 = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in shards]
    torch.cuda.synchronize()
    for sh, dJ, dV in zip(shards, dJ4, dV4):
        sh.allreduce_scalars_dev(dJ.data_ptr(), dV.data_ptr())
    for sh in shards:
        sh.synchronize()
    assert all(np.isnan(float(v.item())) for v in dV4)
    for e in shards + [whole]:
        e.close()

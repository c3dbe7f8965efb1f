"""Knot-range shards of linear-spline time-dependent bilinear problems (BASELINE config c3 shape).

With spline_order = 1, interval k reads u_{k+1}: interval k0 - 1, which the left neighbour owns, adds to the Hessian
region of a shard's first knot k0.  Linked shards hand that block over through the exchange windows (the left neighbour
pushes its last interval's compact second derivatives, the shard assembles its first knot after they arrive), so the
reassembled Hessian is bit-identical to the whole-problem evaluation.  Everything runs on ONE GPU with several handles in
one process (dto_shard_link_local), except the optional two-GPU case."""
import time

import numpy as np
import pytest

import dto_b200 as dto
import dto_oracle as orc
from dto_b200 import problem_templates as pt
from dto_b200.sharding import knot_ranges
from helpers import blocks
from helpers.kernels import interval_kernels, norm as kernel_name

pytestmark = pytest.mark.gpu

TDB_TOL = 1e-10  # K7 against the oracle's variational solve, block-relative (as in test_parity_gpu.py)


def _cuts(N):
    """a one-knot shard in the middle and a last shard that owns no interval"""
    return [(1, 3), (4, 4), (5, N - 1), (N, N)]


def _tdb(nt, warps, split=False):
    return (f"tdb_dmma_kernel<{nt}, {warps}>",) + ((f"tdb_exp_kernel<{nt}>",) if split else ())


# (state dim, drives, N, DTO_B200_TDB_SPLIT, interval kernels of a Hessian evaluation)
CASES = [
    (16, 2, 9, None, _tdb(2, 8)),
    (64, 2, 8, None, _tdb(8, 8, True)),     # c3: n = 64, 2 drives
    (12, 2, 9, None, ("tdb_kernel",)),      # n % 8 != 0
    (40, 2, 8, None, ("tdb_kernel",)),      # a shape the K7 matrix pins to the CUDA-core kernel
    (16, 3, 9, None, ("tdb_kernel",)),      # 1 + np > 8
    (64, 2, 8, "0", _tdb(8, 16)),           # one 16-warp CTA per interval
]


def _problem(n, m, N):
    kw = {} if n == 64 else {"dt": 0.2}
    return pt.carrier_problem(N=N, state_dim=n, n_drives=m, spline_order=1, **kw)


def _iterate(prob, rng):
    Z0 = prob.trajectory.vec()
    return Z0 + 0.02 * rng.standard_normal(Z0.size)


def _local(sh, Z, nan_halo=True):
    """the shard's slice of Z; linked shards must not read the local halo slot, so it holds NaN"""
    L = sh.shard_layout
    Zloc = Z[L.z_begin:L.z_halo_end].copy()
    if nan_halo and L.z_halo_end > L.z_end:
        Zloc[L.z_end - L.z_begin:] = np.nan
    return Zloc


def _whole(ev, Z, sigma, mu):
    J, grad = np.empty(1), np.empty(ev.n_vars)
    g, jac, hess = np.empty(ev.n_constraints), np.empty(ev.nnz_jacobian), np.empty(ev.nnz_hessian)
    ev.eval_all(Z, sigma, mu, J, grad, g, jac, hess)
    return J[0], grad, g, jac, hess


class Reassembled:
    """the whole problem's outputs, filled shard by shard through shard_maps() (NaN where no shard wrote)"""

    def __init__(self, whole):
        self.J = 0.0
        self.grad = np.full(whole.n_vars, np.nan)
        self.g, self.jac = np.full(whole.n_constraints, np.nan), np.full(whole.nnz_jacobian, np.nan)
        self.hess = np.full(whole.nnz_hessian, np.nan)

    def put(self, sh, J=None, grad=None, g=None, jac=None, hess=None):
        L = sh.shard_layout
        rows, jpos, hpos = sh.shard_maps()
        if J is not None:
            self.J += J
        if grad is not None:
            self.grad[L.z_begin:L.z_end] = grad
        if g is not None:
            assert np.all(np.isnan(self.g[rows]))
            self.g[rows] = g
        if jac is not None:
            assert np.all(np.isnan(self.jac[jpos]))
            self.jac[jpos] = jac
        if hess is not None:
            assert np.all(np.isnan(self.hess[hpos]))  # disjoint ownership
            self.hess[hpos] = hess

    def check(self, ref, what=""):
        Jw, gradw, gw, jacw, hessw = ref
        assert np.array_equal(self.grad, gradw), what
        assert np.array_equal(self.g, gw), what
        assert np.array_equal(self.jac, jacw), what
        assert np.array_equal(self.hess, hessw), what
        assert abs(self.J - Jw) <= 1e-13 * max(1.0, abs(Jw)), what


def _eval_all_shards(shards, Z, sigma, mu, whole):
    """every shard uploads the iterate (rank order), then evaluates everything with eval_all (rank order)"""
    locs = [_local(sh, Z) for sh in shards]
    for sh, Zloc in zip(shards, locs):
        sh.upload(Zloc)
    out = Reassembled(whole)
    for sh, Zloc in zip(shards, locs):
        rows = sh.shard_maps()[0]
        L = sh.shard_layout
        J, grad = np.empty(1), np.empty(L.z_end - L.z_begin)
        g, jac, hess = np.empty(sh.n_constraints), np.empty(sh.nnz_jacobian), np.empty(sh.nnz_hessian)
        sh.eval_all(Zloc, sigma, mu[rows], J, grad, g, jac, hess)
        out.put(sh, J[0], grad, g, jac, hess)
    return out


def _eval_all_dev_shards(shards, Z, sigma, mu, whole, order=None, stagger_s=0.0, devices=None):
    """the device-pointer path: every shard's upload_dev + eval_all_dev enqueued (in `order`, default rank order) before
    any shard synchronises; stagger_s: host delay between two shards' enqueues; devices: of the shards (default cuda:0)"""
    import torch

    order = list(range(len(shards))) if order is None else order
    devices = [0] * len(shards) if devices is None else devices
    bufs = {}
    for i in order:
        sh = shards[i]
        dev = torch.device("cuda", devices[i])
        L = sh.shard_layout
        rows = sh.shard_maps()[0]
        b = dict(Z=torch.from_numpy(_local(sh, Z)).to(dev), mu=torch.from_numpy(np.r_[mu[rows], 0.0]).to(dev),  # never empty: a Hessian evaluation needs a mu pointer
                 J=torch.zeros(1, dtype=torch.float64, device=dev), grad=torch.zeros(L.z_end - L.z_begin, dtype=torch.float64, device=dev),
                 g=torch.zeros(max(sh.n_constraints, 1), dtype=torch.float64, device=dev),
                 jac=torch.zeros(sh.nnz_jacobian, dtype=torch.float64, device=dev), hess=torch.zeros(sh.nnz_hessian, dtype=torch.float64, device=dev))
        bufs[i] = b
    for d in range(torch.cuda.device_count()):
        torch.cuda.synchronize(d)  # the input copies have landed before another stream reads them
    for k, i in enumerate(order):
        sh, b = shards[i], bufs[i]
        if k and stagger_s:
            time.sleep(stagger_s)
        sh.upload_dev(b["Z"].data_ptr())
        sh.eval_all_dev(sh.local_Z_ptr, sigma, b["mu"].data_ptr(), b["J"].data_ptr(), b["grad"].data_ptr(), b["g"].data_ptr(),
                        b["jac"].data_ptr(), b["hess"].data_ptr())
    for sh in shards:
        sh.synchronize()
    out = Reassembled(whole)
    for i, sh in enumerate(shards):
        b = bufs[i]
        out.put(sh, float(b["J"].item()), b["grad"].cpu().numpy(), b["g"].cpu().numpy()[:sh.n_constraints], b["jac"].cpu().numpy(),
                b["hess"].cpu().numpy())
    return out


def _close(*evs):
    for e in evs:
        e.close()


@pytest.mark.parametrize("n,m,N,split,kernels", CASES, ids=[f"n{c[0]}-m{c[1]}" + ("" if c[3] is None else f"-split{c[3]}") for c in CASES])
def test_linked_shards_reassemble_the_whole_problem(monkeypatch, n, m, N, split, kernels):
    if split is not None:
        monkeypatch.setenv("DTO_B200_TDB_SPLIT", split)
    rng = np.random.default_rng(21)
    prob = _problem(n, m, N)
    whole = dto.Evaluator(prob)
    Z = _iterate(prob, rng)
    mu = rng.random(whole.n_constraints)
    ref = _whole(whole, Z, 1.3, mu)
    shards = [dto.Evaluator(prob, shard=c) for c in _cuts(N)]  # k0 > 1 with a linear spline: accepted
    dto.Evaluator.shard_link_local(shards)
    hr, hc = whole.hessian_lagrangian_structure()
    for sh in shards:
        hpos = sh.shard_maps()[2]
        sr, sc = sh.hessian_lagrangian_structure()
        assert np.array_equal(sr, hr[hpos]) and np.array_equal(sc, hc[hpos])
    res = {}
    ks = interval_kernels(lambda: res.setdefault("out", _eval_all_shards(shards, Z, 1.3, mu, whole)))
    assert ks == {kernel_name(k) for k in kernels}, sorted(ks)
    res["out"].check(ref)
    # the cross block of every shard boundary is genuinely nonzero: the received block matters
    z = prob.trajectory.dim
    for k0, _ in _cuts(N)[1:]:
        sel = ((hr - 1) // z == k0 - 1) & ((hc - 1) // z == k0 - 2)
        sel |= ((hc - 1) // z == k0 - 1) & ((hr - 1) // z == k0 - 2)
        assert np.abs(ref[4][sel]).max() > 1e-8, k0
    _close(*shards, whole)


@pytest.mark.parametrize("n,N", [(16, 9), (64, 8)])
@pytest.mark.parametrize("sigma", [1.3, 0.0])
def test_linked_shards_match_the_oracle(n, N, sigma):
    rng = np.random.default_rng(22)
    prob = _problem(n, 2, N)
    spec = prob.to_spec()
    whole = dto.Evaluator(prob)
    Z = _iterate(prob, rng)
    mu = rng.random(whole.n_constraints)
    shards = [dto.Evaluator(prob, shard=c) for c in _cuts(N)]
    dto.Evaluator.shard_link_local(shards)
    out = _eval_all_shards(shards, Z, sigma, mu, whole)
    Z0 = prob.trajectory.vec()
    hst = orc.hessian_structure(spec, Z0)
    Href = orc.eval_hessian_lagrangian(spec, Z, sigma, mu, hst)
    assert not np.any(np.isnan(out.hess))
    assert blocks.hess_block_relerr(spec, hst, out.hess, Href) <= TDB_TOL
    assert np.abs(out.hess - Href).max() <= TDB_TOL * np.abs(Href).max()
    _close(*shards, whole)


def test_linked_shards_follow_a_changing_iterate():
    """Solver-loop pattern: five iterates with new Z and mu, each driven through the five separate callbacks (rank order),
    eval_all (rank order) and eval_all_dev enqueued on every shard before any synchronises -- three Hessian evaluations
    per iterate, so both block slots and their acknowledgements turn over many times."""
    import torch  # noqa: F401

    N = 11
    prob = _problem(16, 2, N)
    rng = np.random.default_rng(23)
    whole = dto.Evaluator(prob)
    cuts = [(1, 3), (4, 4), (5, 8), (9, 10), (11, 11)]
    shards = [dto.Evaluator(prob, shard=c) for c in cuts]
    dto.Evaluator.shard_link_local(shards)
    for it in range(5):
        Z = _iterate(prob, rng)
        mu = rng.random(whole.n_constraints)
        sigma = 0.4 + 0.3 * it
        ref = _whole(whole, Z, sigma, mu)
        # the five callbacks
        locs = [_local(sh, Z) for sh in shards]
        for sh, Zloc in zip(shards, locs):
            sh.upload(Zloc)
        out = Reassembled(whole)
        for sh, Zloc in zip(shards, locs):
            rows = sh.shard_maps()[0]
            L = sh.shard_layout
            grad = np.empty(L.z_end - L.z_begin)
            g, jac, hess = np.empty(sh.n_constraints), np.empty(sh.nnz_jacobian), np.empty(sh.nnz_hessian)
            J = sh.eval_objective(Zloc)
            sh.eval_objective_gradient(grad, Zloc)
            sh.eval_constraint(g, Zloc)
            sh.eval_constraint_jacobian(jac, Zloc)
            sh.eval_hessian_lagrangian(hess, Zloc, sigma, mu[rows])
            out.put(sh, J, grad, g, jac, hess)
        out.check(ref, f"callbacks, iterate {it}")
        # the fused host-pointer pass on the same iterate
        out = Reassembled(whole)
        for sh, Zloc in zip(shards, locs):
            rows = sh.shard_maps()[0]
            L = sh.shard_layout
            J, grad = np.empty(1), np.empty(L.z_end - L.z_begin)
            g, jac, hess = np.empty(sh.n_constraints), np.empty(sh.nnz_jacobian), np.empty(sh.nnz_hessian)
            sh.eval_all(Zloc, sigma, mu[rows], J, grad, g, jac, hess)
            out.put(sh, J[0], grad, g, jac, hess)
        out.check(ref, f"eval_all, iterate {it}")
        # the device-pointer path
        _eval_all_dev_shards(shards, Z, sigma, mu, whole).check(ref, f"eval_all_dev, iterate {it}")
    _close(*shards, whole)


def test_registered_outputs_on_linked_shards():
    N = 9
    prob = _problem(16, 2, N)
    rng = np.random.default_rng(24)
    whole = dto.Evaluator(prob)
    shards = [dto.Evaluator(prob, shard=c) for c in _cuts(N)]
    dto.Evaluator.shard_link_local(shards)
    regs = []
    for sh in shards:
        jac, hess = np.empty(sh.nnz_jacobian), np.empty(sh.nnz_hessian)
        sh.register_outputs(jac, hess)
        regs.append((jac, hess))
    for it in range(2):
        Z = _iterate(prob, rng)
        mu = rng.random(whole.n_constraints)
        ref = _whole(whole, Z, 1.1, mu)
        locs = [_local(sh, Z) for sh in shards]
        for sh, Zloc in zip(shards, locs):
            sh.upload(Zloc)
        out = Reassembled(whole)
        for sh, Zloc, (jac, hess) in zip(shards, locs, regs):
            rows = sh.shard_maps()[0]
            sh.eval_constraint_jacobian(jac, Zloc)
            sh.eval_hessian_lagrangian(hess, Zloc, 1.1, mu[rows])
            out.put(sh, jac=jac.copy(), hess=hess.copy())
        assert np.array_equal(out.jac, ref[3]) and np.array_equal(out.hess, ref[4]), it
    for sh in shards:
        sh.unregister_outputs()
    _close(*shards, whole)


def test_unlinked_shard_has_everything_but_the_hessian():
    N = 9
    prob = _problem(16, 2, N)
    rng = np.random.default_rng(25)
    whole = dto.Evaluator(prob)
    Z = _iterate(prob, rng)
    mu = rng.random(whole.n_constraints)
    ref = _whole(whole, Z, 1.0, mu)
    first, mid = dto.Evaluator(prob, shard=(1, 3)), dto.Evaluator(prob, shard=(4, 6))  # k0 > 1: created without error
    out = Reassembled(whole)
    for sh in (first, mid):
        Zloc = _local(sh, Z, nan_halo=False)  # unlinked: the halo knot comes from the caller's slice
        rows = sh.shard_maps()[0]
        L = sh.shard_layout
        grad = np.empty(L.z_end - L.z_begin)
        g, jac = np.empty(sh.n_constraints), np.empty(sh.nnz_jacobian)
        J = sh.eval_objective(Zloc)
        sh.eval_objective_gradient(grad, Zloc)
        sh.eval_constraint(g, Zloc)
        sh.eval_constraint_jacobian(jac, Zloc)
        hess = None
        if sh is first:  # starts at knot 1: no block to receive
            hess = np.empty(sh.nnz_hessian)
            sh.eval_hessian_lagrangian(hess, Zloc, 1.0, mu[rows])
        out.put(sh, J, grad, g, jac, hess)
        rows, jpos, hpos = sh.shard_maps()
        L = sh.shard_layout
        assert np.array_equal(out.grad[L.z_begin:L.z_end], ref[1][L.z_begin:L.z_end])
        assert np.array_equal(out.g[rows], ref[2][rows]) and np.array_equal(out.jac[jpos], ref[3][jpos])
        if hess is not None:
            assert np.array_equal(hess, ref[4][hpos])
    Zloc = _local(mid, Z, nan_halo=False)
    rows = mid.shard_maps()[0]
    for call in (lambda: mid.eval_hessian_lagrangian(np.empty(mid.nnz_hessian), Zloc, 1.0, mu[rows]),
                 lambda: mid.eval_all(Zloc, 1.0, mu[rows], None, None, None, None, np.empty(mid.nnz_hessian))):
        with pytest.raises(dto.DtoError) as ei:
            call()
        assert "link" in str(ei.value) and "left neighbour" in str(ei.value)
    # still usable afterwards
    g = np.empty(mid.n_constraints)
    mid.eval_all(Zloc, 1.0, None, None, None, g, None, None)
    assert np.array_equal(g, ref[2][rows])
    _close(first, mid, whole)


def test_relink_starts_from_clean_windows():
    """Link, three iterates, link the same shards again, two more.  The right shards are enqueued first, each some time
    ahead of its left neighbour (as ranks in separate processes may be): the waits must see the new link's sequence
    numbers, not the old link's, or a shard reads a stale block."""
    N = 11
    prob = _problem(16, 2, N)
    rng = np.random.default_rng(26)
    whole = dto.Evaluator(prob)
    cuts = [(1, 3), (4, 4), (5, 8), (9, 11)]
    shards = [dto.Evaluator(prob, shard=c) for c in cuts]
    rev = list(range(len(shards)))[::-1]
    dto.Evaluator.shard_link_local(shards)
    for it in range(5):
        if it == 3:
            dto.Evaluator.shard_link_local(shards)
        Z = _iterate(prob, rng)
        mu = rng.random(whole.n_constraints)
        ref = _whole(whole, Z, 0.9, mu)
        _eval_all_dev_shards(shards, Z, 0.9, mu, whole, order=rev, stagger_s=0.05).check(ref, f"iterate {it}")
    _close(*shards, whole)


def test_two_gpus_one_shard_each():
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    N = 9
    prob = _problem(16, 2, N)
    rng = np.random.default_rng(27)
    whole = dto.Evaluator(prob, device=0)
    Z = _iterate(prob, rng)
    mu = rng.random(whole.n_constraints)
    ref = _whole(whole, Z, 1.2, mu)
    shards = [dto.Evaluator(prob, shard=c, device=d) for d, c in enumerate(knot_ranges(N, 2))]
    dto.Evaluator.shard_link_local(shards)
    _eval_all_shards(shards, Z, 1.2, mu, whole).check(ref, "host path")
    _eval_all_dev_shards(shards, Z, 1.2, mu, whole, devices=[0, 1]).check(ref, "device path")
    _close(*shards, whole)

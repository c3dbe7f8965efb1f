"""Every instantiation of the bilinear interval kernel (K1) against the oracle.

K1 is a family of template instantiations: octet (n = 8, 16), persistent and dmma (n = 8..64, NT = n / 8 tiles, MT = 2
forward tiles once 1 + m + m(m+1)/2 > 8), the per-problem-generator forms of octet and dmma, generic (any other shape),
and the matrix-free product kernel.  The host picks one at construction and launchers may decline a shape, so the
variant a handle reports is not proof of which kernel produced the numbers.  Each cell below therefore records the
interval kernels the CUDA profiler sees and asserts that they are exactly the ones the cell is meant to reach; the
coverage guard at the end asserts that the cells together reached every instantiation in KERNELS.

Every cell runs on an iterate whose intervals take different code paths: dt = 0, u = 0, and theta = |dt| ||G(u)||_1
below 1.5 (plain series), in (1.5, 4] (scaling branch) and above 4 (multi-stage series)."""
from dataclasses import dataclass, field

import numpy as np
import pytest

import dto_b200 as dto
import dto_oracle as orc
from dto_b200 import problem_templates as pt
from helpers import blocks
from helpers.kernels import interval_kernels, norm as _norm

# measured on a B200 (1000 W): every cell within 4e-13 of the oracle, block-relative (per-problem generators at n = 8 the
# largest, 3.8e-13 in the Jacobian); all other cells below 1e-13
TOL = 1e-12

# the interval-kernel instantiations the cells below must reach between them (demangled names, template arguments)
KERNELS = sorted(
    [f"bilinear_persistent_kernel<{nt}, {mt}>" for nt in (1, 2, 3, 4, 6, 8) for mt in (1, 2)]
    + [f"bilinear_dmma_kernel<{nt}, {mt}>" for nt in (1, 2, 3, 4, 6, 8) for mt in (1, 2)]
    + [f"bilinear_product_kernel<{nt}>" for nt in (1, 2, 3, 4, 6, 8)]
    + [f"bilinear_octet_kernel<1, {m}, false>" for m in (1, 2, 3, 4)]
    + ["bilinear_octet_kernel<2, 1, false>", "bilinear_octet_kernel<2, 2, false>"]
    + ["bilinear_octet_kernel<1, 1, true>", "bilinear_octet_kernel<1, 4, true>", "bilinear_octet_kernel<2, 1, true>"]
    + ["bilinear_generic_kernel"])


@dataclass
class Cell:
    id: str
    n: int
    m: int
    fused: tuple          # interval kernels of one fused eval_all with the Hessian
    hess: tuple           # ... of the Hessian-only callback after the residual and Jacobian callbacks
    prod: tuple = ()      # ... of J w and J' w (the matrix-free product kernel); () = materialised, not profiled
    env: dict = field(default_factory=dict)
    batch: int = 1        # > 1: a batch with different generators per problem
    N: int = 11


def _mt(m):
    return 2 if 1 + m + m * (m + 1) // 2 > 8 else 1


def _persistent(n, m, env=None, N=11, tag=""):
    nt = n // 8
    # at n = 64, m = 4 the product kernel's generators and per-warp matrices exceed shared memory: J w then comes from the
    # Jacobian the persistent kernel materialises (forward role without second derivatives, MT = 1)
    prod = f"bilinear_persistent_kernel<{nt}, 1>" if (n, m) == (64, 4) else f"bilinear_product_kernel<{nt}>"
    return Cell(f"persistent_n{n}_m{m}{tag}" + ("" if N == 11 else f"_N{N}"), n, m,
                (f"bilinear_persistent_kernel<{nt}, {_mt(m)}>",), (f"bilinear_persistent_kernel<{nt}, 1>",),
                (prod,), env or {}, 1, N)


def _dmma(n, m, batch=1, N=11):
    name = (f"bilinear_dmma_kernel<{n // 8}, {_mt(m)}>",)
    return Cell(f"dmma_n{n}_m{m}" + ("" if batch == 1 else f"_B{batch}") + ("" if N == 11 else f"_N{N}"), n, m, name, name, (),
                {} if batch > 1 else {"DTO_B200_KERNEL": "dmma"}, batch, N)


def _octet(n, m, split=None, batch=1, N=11):
    name = (f"bilinear_octet_kernel<{n // 8}, {m}, {'true' if batch > 1 else 'false'}>",)
    env = {} if split is None else {"DTO_B200_OCTET_SPLIT": split}
    tag = ("" if split is None else f"_split{split}") + ("" if batch == 1 else f"_B{batch}") + ("" if N == 11 else f"_N{N}")
    return Cell(f"octet_n{n}_m{m}{tag}", n, m, name, name, (f"bilinear_product_kernel<{n // 8}>",) if batch == 1 else (), env, batch, N)


def _generic(n, m, env=None, N=11):
    name = ("bilinear_generic_kernel",)
    return Cell(f"generic_n{n}_m{m}" + ("_pinned" if env else "") + ("" if N == 11 else f"_N{N}"), n, m, name, name, (), env or {}, 1, N)


_PIN = {"DTO_B200_KERNEL": "persistent"}
CELLS = (
    # persistent: NT = 1..8 x MT = 1, 2; n = 8 / 16 are pinned where octet would take them; n = 64, m = 4 leaves no
    # shared memory for the Paterson-Stockmeyer warps (nE = 0), n = 32 with DTO_B200_K1_NE=0 forces it
    [_persistent(8, 2, _PIN), _persistent(8, 4, _PIN), _persistent(16, 2, _PIN), _persistent(16, 3)]
    + [_persistent(n, m) for n in (24, 32, 48, 64) for m in (2, 3 if n in (24, 48) else 4)]
    + [_persistent(32, 2, {"DTO_B200_K1_NE": "0"}, tag="_ne0"), _persistent(32, 4, N=2)]
    # dmma: the same shapes pinned, and the per-problem-generator batches it runs by default at n >= 24
    + [_dmma(n, m) for n, m in ((8, 2), (8, 4), (16, 2), (16, 3), (24, 2), (24, 3), (32, 2), (32, 4), (48, 2), (48, 3), (64, 2), (64, 4))]
    + [_dmma(24, 2, batch=3), _dmma(48, 3, batch=3), _dmma(64, 4, batch=3), _dmma(24, 2, N=2)]
    # octet: whole octets (default at these sizes) and every octet cut into phases, per-problem generators (PP = true)
    + [_octet(n, m, split) for n, m in ((8, 1), (8, 2), (8, 3), (8, 4), (16, 1), (16, 2)) for split in (None, "1")]
    + [_octet(8, 1, batch=3), _octet(8, 4, batch=3), _octet(16, 1, batch=3), _octet(8, 2, N=2)]
    # generic: states no tensor-core kernel takes, more than four drives, and pinned at n = 64
    + [_generic(n, m) for n in (3, 40, 56, 72) for m in (1, 4)]
    + [_generic(n, m) for n in (8, 32) for m in (5, 6)]
    + [_generic(64, 4, {"DTO_B200_KERNEL": "generic"}), _generic(40, 1, N=2)]
)

# theta = |dt| ||G(u)||_1 per interval of the N = 11 iterate: 0 marks dt = 0; interval 6 also has u = 0
THETAS = [0.6, 0.0, 1.2, 2.2, 3.6, 5.5, 0.9, 8.0, 1.45, 3.0]
U_ZERO = 6


def _problem(cell, seed=42):
    return pt.scaled_problem(N=cell.N, state_dim=cell.n, n_controls=cell.m, seed=seed, generator_scale=1.0 / np.sqrt(cell.n))


def _shaped_iterate(prob, G, seed):
    """Z0 + 3 % noise, then per interval: dt from THETAS (dt = 0 in one, u = 0 in another)."""
    spec = prob.to_spec()
    z, N = spec["z"], spec["N"]
    dt_off, (u_off, m) = spec["components"][spec["timestep"]][0], spec["components"]["u"]
    rng = np.random.default_rng(seed)
    Z0 = prob.trajectory.vec()
    Z = Z0 + 0.03 * rng.standard_normal(Z0.size)
    thetas = THETAS if N == 11 else [1.0] * (N - 1)
    for k, th in enumerate(thetas):
        u = Z[k * z + u_off:k * z + u_off + m]
        if N == 11 and k == U_ZERO:
            u[:] = 0.0
        Gu = G[0] + np.tensordot(u, G[1:], axes=1)
        Z[k * z + dt_off] = th / np.abs(Gu).sum(axis=0).max()
    return Z


def _oracle(spec, Z, sigma, mu, jst, hst):
    return (orc.eval_objective(spec, Z), orc.eval_objective_gradient(spec, Z), orc.eval_constraint(spec, Z),
            orc.eval_constraint_jacobian(spec, Z, jst), orc.eval_hessian_lagrangian(spec, Z, sigma, mu, hst))


def relerr(got, ref):
    return float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-300)) if ref.size else 0.0


def _errors(spec, jst, hst, got, ref):
    """(max-norm relative, block-relative) errors of (J, grad, g, jac, hess)."""
    J, grad, g, jac, hess = got
    Jr, gradr, gr, jacr, hessr = ref
    ej = abs(J - Jr) / max(1.0, abs(Jr))
    return {"obj": (ej, ej), "grad": (relerr(grad, gradr), relerr(grad, gradr)),
            "g": (relerr(g, gr), blocks.vec_block_relerr(spec, g, gr)),
            "jac": (relerr(jac, jacr), blocks.jac_block_relerr(spec, jst, jac, jacr)),
            "hess": (relerr(hess, hessr), blocks.hess_block_relerr(spec, hst, hess, hessr))}


_SEEN = {}  # cell id -> interval kernels seen in its profiled calls


@pytest.mark.gpu
@pytest.mark.parametrize("cell", CELLS, ids=lambda c: c.id)
def test_instantiation_matches_oracle(cell, monkeypatch):
    for k, v in cell.env.items():
        monkeypatch.setenv(k, v)
    B = cell.batch
    prob = _problem(cell)
    rng = np.random.default_rng(3)
    if B > 1:
        Gs = rng.standard_normal((B, cell.m + 1, cell.n, cell.n)) / np.sqrt(cell.n)
        ev = dto.Evaluator(prob, batch=B, batch_G=Gs)
    else:
        Gs = prob.integrators[0].G[None]
        ev = dto.Evaluator(prob)
    probs = []
    for b in range(B):
        pb = _problem(cell)
        pb.integrators[0].G = Gs[b]
        probs.append(pb)
    spec = [p.to_spec() for p in probs]
    Z0 = prob.trajectory.vec()
    jst, hst = orc.jacobian_structure(spec[0], Z0), orc.hessian_structure(spec[0], Z0)
    jr, jc = ev.jacobian_structure()
    hr, hc = ev.hessian_lagrangian_structure()
    assert np.array_equal(jr, jst[0]) and np.array_equal(jc, jst[1]) and np.array_equal(hr, hst[0]) and np.array_equal(hc, hst[1])
    nc, nv, nj, nh = ev.n_constraints, ev.n_vars, ev.nnz_jacobian, ev.nnz_hessian
    seen = set()
    worst = {}

    def check(tag, got, Z, sigma, mu):
        for b in range(B):
            ref = _oracle(spec[b], Z[b], sigma, mu[b], jst, hst)
            for key, (e_max, e_blk) in _errors(spec[b], jst, hst, [x[b] for x in got], ref).items():
                worst[key] = max(worst.get(key, 0.0), e_max, e_blk)
                assert e_max <= TOL and e_blk <= TOL, (cell.id, tag, b, key, e_max, e_blk)

    # fused: eval_all with sigma = 1.3, then the sigma = 0 Hessian
    Z = np.stack([_shaped_iterate(probs[b], Gs[b], seed=10 + b) for b in range(B)])
    mu = rng.random((B, nc))
    out = [np.full(B, np.nan), np.full((B, nv), np.nan), np.full((B, nc), np.nan), np.full((B, nj), np.nan), np.full((B, nh), np.nan)]
    ks = interval_kernels(lambda: ev.eval_all(Z, 1.3, mu, *out))
    assert ks == {_norm(k) for k in cell.fused}, (cell.id, "fused", sorted(ks))
    seen |= ks
    check("fused", out, Z, 1.3, mu)
    H0 = np.full((B, nh), np.nan)
    ev.eval_hessian_lagrangian(H0, Z, 0.0, mu)
    for b in range(B):
        H0ref = orc.eval_hessian_lagrangian(spec[b], Z[b], 0.0, mu[b], hst)
        e = max(relerr(H0[b], H0ref), blocks.hess_block_relerr(spec[b], hst, H0[b], H0ref))
        worst["hess0"] = max(worst.get("hess0", 0.0), e)
        assert e <= TOL, (cell.id, "sigma = 0", b, e)

    # the five callbacks separately on a new iterate (persistent and octet: jets stored by the residual pass, the
    # Hessian callback runs the adjoint-only pass); they must match the oracle and the fused call bit for bit
    Z2 = np.stack([_shaped_iterate(probs[b], Gs[b], seed=20 + b) for b in range(B)])
    mu2 = rng.random((B, nc))
    sep = [np.full(B, np.nan), np.full((B, nv), np.nan), np.full((B, nc), np.nan), np.full((B, nj), np.nan), np.full((B, nh), np.nan)]
    sep[0][:] = ev.eval_objective(Z2)
    ev.eval_objective_gradient(sep[1], Z2)
    ev.eval_constraint(sep[2], Z2)
    ev.eval_constraint_jacobian(sep[3], Z2)
    ks = interval_kernels(lambda: ev.eval_hessian_lagrangian(sep[4], Z2, 1.3, mu2))
    assert ks == {_norm(k) for k in cell.hess}, (cell.id, "Hessian callback", sorted(ks))
    seen |= ks
    check("callbacks", sep, Z2, 1.3, mu2)
    fused2 = [np.full_like(a, np.nan) for a in sep]
    ev.eval_all(Z2, 1.3, mu2, *fused2)
    for a, b in zip(sep, fused2):
        assert np.array_equal(a, b), cell.id

    # J w and J' w against the oracle's dense Jacobian
    if B == 1:
        jref = orc.eval_constraint_jacobian(spec[0], Z[0], jst)
        Jd = np.zeros((nc, nv))
        np.add.at(Jd, (jst[0] - 1, jst[1] - 1), jref)
        w1, w2 = rng.standard_normal(nv), rng.standard_normal(nc)
        y1, y2 = np.full(nc, np.nan), np.full(nv, np.nan)

        def products():
            ev.eval_constraint_jacobian_product(y1, Z[0], w1)
            ev.eval_constraint_jacobian_transpose_product(y2, Z[0], w2)

        if cell.prod:
            ks = interval_kernels(products)
            assert ks == {_norm(k) for k in cell.prod}, (cell.id, "products", sorted(ks))
            seen |= ks
        else:
            products()
        # error scale: sum |J_ij| |w_j| bounds what the summation order can change
        e1 = np.abs(y1 - Jd @ w1).max() / (np.abs(Jd) @ np.abs(w1)).max()
        e2 = np.abs(y2 - Jd.T @ w2).max() / (np.abs(Jd.T) @ np.abs(w2)).max()
        worst["prod"] = max(e1, e2)
        assert e1 <= TOL and e2 <= TOL, (cell.id, e1, e2)
    ev.close()
    _SEEN[cell.id] = seen
    print(f"\n{cell.id}: worst relative error " + " ".join(f"{k}={v:.1e}" for k, v in worst.items()) + f"  kernels={sorted(seen)}")


@pytest.mark.gpu
def test_every_declared_instantiation_ran():
    """A cell whose shape silently falls back to another kernel fails its own assertion; this guards the list itself:
    the union of what the profiler saw is exactly KERNELS."""
    missing = {c.id for c in CELLS} - set(_SEEN)
    if missing:
        pytest.skip(f"{len(missing)} cells did not complete in this session")
    union = set().union(*_SEEN.values())
    print("\nkernel union: " + ", ".join(sorted(union)))
    assert union == {_norm(k) for k in KERNELS}, (sorted(union - {_norm(k) for k in KERNELS}), sorted({_norm(k) for k in KERNELS} - union))


def test_cells_declare_exactly_the_kernel_list():
    expected = set()
    for c in CELLS:
        expected |= {_norm(k) for k in c.fused + c.hess + c.prod}
    assert expected == {_norm(k) for k in KERNELS}
    assert len({c.id for c in CELLS}) == len(CELLS)


def test_block_comparison_rejects_small_perturbations():
    """The block-relative comparison is not vacuous: a 1e-9 relative change of one entry in the smallest nonzero Jacobian
    block, in an all-zero block (a drive whose matrix is zero) and in the smallest nonzero Hessian region is rejected at
    TOL, also where the array's max-norm would accept it."""
    n, N = 8, 5
    rng = np.random.default_rng(1)
    G0 = rng.standard_normal((n, n)) / n
    Gd = [rng.standard_normal((n, n)) / n, np.zeros((n, n))]
    traj = dto.NamedTrajectory({"x": rng.standard_normal((n, N)), "u": rng.standard_normal((2, N)), "dt": np.full(N, 0.1)},
                               timestep="dt", controls=("u",))
    prob = dto.DirectTrajOptProblem(traj, dto.QuadraticRegularizer("u", traj, 1e-4), dto.BilinearIntegrator((G0, Gd), "x", "u", traj))
    spec, Z = prob.to_spec(), prob.trajectory.vec()
    jst, hst = orc.jacobian_structure(spec, Z), orc.hessian_structure(spec, Z)
    mu = rng.random(orc.n_constraints(spec)[0])
    J = orc.eval_constraint_jacobian(spec, Z, jst)
    H = orc.eval_hessian_lagrangian(spec, Z, 1.0, mu, hst)
    assert blocks.jac_block_relerr(spec, jst, J.copy(), J) == 0.0 and blocks.hess_block_relerr(spec, hst, H.copy(), H) == 0.0

    z = spec["z"]
    u_off = spec["components"]["u"][0]
    cols = jst[1] - 1
    rows = jst[0] - 1
    # d r_1 / d u (second drive) at knot 1: stored, all zero
    zero_blk = np.flatnonzero((cols == u_off + 1) & (rows < n))
    assert zero_blk.size and np.all(J[zero_blk] == 0.0)
    # d r_1 / d dt_1: the smallest nonzero block of interval 1
    dt_blk = np.flatnonzero((cols == spec["components"][spec["timestep"]][0]) & (rows < n))
    assert np.abs(J[dt_blk]).max() > 0
    for pos, scale in ((dt_blk[0], np.abs(J[dt_blk]).max()), (zero_blk[0], np.abs(J[rows < n]).max())):
        bad = J.copy()
        bad[pos] += 1e-9 * scale
        assert blocks.jac_block_relerr(spec, jst, bad, J) > TOL
    # the Hessian region of the last knot holds only the tiny regularizer
    last = np.flatnonzero((hst[1] - 1) // z == N - 1)
    small = last[np.argmax(np.abs(H[last]))]
    assert np.abs(H[last]).max() < 1e-2 * np.abs(H).max()
    bad = H.copy()
    bad[small] *= 1 + 1e-9
    assert relerr(bad, H) <= TOL < blocks.hess_block_relerr(spec, hst, bad, H)

"""``DirectTrajOptProblem`` and the B200-backed ``Evaluator`` -- the drop-in for
``Solvers.Evaluator <: MOI.AbstractNLPEvaluator`` (/root/reference/src/solvers/evaluator.jl:66-456).

Method names, argument order, in-place output semantics and 1-based structures are the reference's;
every value is computed by libdto_b200.so's CUDA kernels through the C ABI (include/dto_b200.h)."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .knot_program import KnotProgram
from .components import (AbstractIntegrator, AbstractNonlinearConstraint, AbstractObjective, BilinearIntegrator,
                         CompositeObjective, DerivativeIntegrator, GlobalKnotPointObjective, KnotPointObjective,
                         MinimumTimeObjective, NullObjective, NonlinearGlobalKnotPointConstraint,
                         LinearRegularizer, QuadraticRegularizer, TimeDependentBilinearIntegrator, UnsupportedComponent)


class DirectTrajOptProblem:
    """``DirectTrajOptProblem(traj, obj, integrators; constraints)`` (problems.jl:50-55).  Linear
    constraints go straight to the solver in the reference (constrain.jl) and never reach the
    evaluator; only ``AbstractNonlinearConstraint``s are kept here."""

    def __init__(self, trajectory, objective, integrators, constraints=()):
        if isinstance(integrators, AbstractIntegrator):
            integrators = [integrators]
        self.trajectory = trajectory
        self.objective = objective
        self.integrators = list(integrators)
        self.constraints = list(constraints)

    def nonlinear_constraints(self):
        return [c for c in self.constraints if isinstance(c, AbstractNonlinearConstraint)]

    def objective_terms(self):
        ob = self.objective
        if isinstance(ob, CompositeObjective):
            return list(zip(ob.objectives, ob.weights))
        return [(ob, 1.0)]

    def to_spec(self):
        """Plain-dict problem description shared with the CPU oracle (tests only)."""
        t = self.trajectory
        spec = {
            "N": t.N, "z": t.dim, "timestep": t.timestep,
            "components": {n: (t.components[n].start, len(t.components[n])) for n in t.names},
            "global_dim": t.global_dim,
            "global_components": {n: (t.global_components[n].start, len(t.global_components[n])) for n in t.global_names},
            "integrators": [i.to_spec() for i in self.integrators],
            "objectives": [], "constraints": [c.to_spec(t) for c in self.nonlinear_constraints()],
            "composite": isinstance(self.objective, CompositeObjective),
        }
        for ob, w in self.objective_terms():
            s = ob.to_spec(t)
            s["weight"] = w
            spec["objectives"].append(s)
        return spec


def _dp(a):
    return a.ctypes.data_as(_lib.c_double_p) if a is not None and a.size else None


def _ip(a):
    return a.ctypes.data_as(_lib.c_int32_p) if a is not None and a.size else None


def _f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


class Evaluator:
    """``Evaluator(prob; eval_hessian=true, verbose=false)``.

    Extra keyword arguments (not in the reference): ``batch`` evaluates that many independent
    problems of identical structure per call (vectors become ``(batch, n)``); ``batch_G`` gives
    per-problem bilinear generators ``(batch, m+1, n, n)`` for integrator 0; ``shard=(k0, k1)``
    creates a knot-range shard of one long trajectory; ``device`` picks the GPU."""

    def __init__(self, prob, eval_hessian=True, verbose=False, batch=1, batch_G=None, shard=None, device=-1, Z0=None):
        lib = _lib.load()
        self._lib = lib
        self.prob = prob
        self.trajectory = prob.trajectory
        self.objective = prob.objective
        self.integrators = prob.integrators
        self.constraints = prob.nonlinear_constraints()
        self.eval_hessian = bool(eval_hessian)
        self.batch = int(batch)
        t = prob.trajectory
        keep = []  # keep every array alive until dto_create returns
        programs = []  # (ops, out, consts) of every KnotProgram term, indexed by the descriptors' `program`

        def knot_fn(fn, catalogue, program_id, n_vars):
            """(fn id, program index) of a term's knot function"""
            if isinstance(fn, KnotProgram):
                tape = fn.trace(n_vars)
                programs.append((np.ascontiguousarray(tape.ops), np.ascontiguousarray(tape.out), _f64(tape.consts)))
                return program_id, len(programs) - 1
            return catalogue[fn.name], 0

        ints = (_lib.IntegratorDesc * max(1, len(prob.integrators)))()
        for i, it in enumerate(prob.integrators):
            d = ints[i]
            d.t_off = -1
            if isinstance(it, BilinearIntegrator):
                d.kind = _lib.INT_BILINEAR
                d.x_off, d.x_dim = t.components[it.x_name].start, it.x_dim
                d.u_off, d.u_dim = t.components[it.u_name].start, it.u_dim
                if batch_G is not None and i == 0:
                    G = _f64(np.asarray(batch_G).transpose(0, 1, 3, 2))  # column-major matrices
                    if G.shape != (self.batch, it.u_dim + 1, it.x_dim, it.x_dim):
                        raise ValueError("batch_G must be (batch, m+1, n, n)")
                    d.G_batch_stride = (it.u_dim + 1) * it.x_dim * it.x_dim
                else:
                    G = _f64(it.G.transpose(0, 2, 1))
                keep.append(G)
                d.G = _dp(G)
            elif isinstance(it, DerivativeIntegrator):
                d.kind = _lib.INT_DERIVATIVE
                d.x_off, d.x_dim = t.components[it.x_name].start, it.x_dim
                d.u_off, d.u_dim = t.components[it.xdot_name].start, it.x_dim
            elif isinstance(it, TimeDependentBilinearIntegrator):
                d.kind = _lib.INT_TDBILINEAR
                d.x_off, d.x_dim = t.components[it.x_name].start, it.x_dim
                d.u_off, d.u_dim = t.components[it.u_name].start, it.u_dim
                d.t_off = t.components[it.t_name].start
                d.spline_order = it.spline_order
                d.tdb_steps = it.steps
                g = it.G
                arrs = [_f64(g.G0.T), _f64(g.A.transpose(0, 2, 1)), _f64(g.B.transpose(0, 2, 1)), _f64(g.omega), _f64(g.phi),
                        _f64(g.D.transpose(0, 2, 1)), _f64(g.omega_d), _f64(g.phi_d)]
                keep += arrs
                d.G, d.A, d.B, d.omega, d.phi, d.D, d.omega_d, d.phi_d = [_dp(a) for a in arrs]
                d.n_carrier = g.D.shape[0]
            else:
                raise UnsupportedComponent(f"integrator {type(it).__name__} is outside the device path")

        terms = prob.objective_terms()
        objs = (_lib.ObjectiveDesc * max(1, len(terms)))()
        for i, (ob, w) in enumerate(terms):
            d = objs[i]
            d.weight = w
            if isinstance(ob, QuadraticRegularizer):
                d.kind = _lib.OBJ_QUADREG
                vo = np.asarray(list(t.components[ob.name]), dtype=np.int32)
                tm = np.asarray(ob.times, dtype=np.int32)
                R, base = _f64(ob.R), _f64(ob.baseline.T)  # (N, nv) row-major == nv x N column-major
                keep += [vo, tm, R, base]
                d.n_vars, d.var_offs, d.n_times, d.times, d.R = len(vo), _ip(vo), len(tm), _ip(tm), _dp(R)
                d.baseline = _dp(base) if np.any(base) else None
            elif isinstance(ob, LinearRegularizer):
                d.kind = _lib.OBJ_LINREG
                vo = np.asarray(list(t.components[ob.name]), dtype=np.int32)
                tm = np.asarray(ob.times, dtype=np.int32)
                R = _f64(ob.R)
                keep += [vo, tm, R]
                d.n_vars, d.var_offs, d.n_times, d.times, d.R = len(vo), _ip(vo), len(tm), _ip(tm), _dp(R)
            elif isinstance(ob, MinimumTimeObjective):
                d.kind = _lib.OBJ_MINTIME
                d.D = ob.D
            elif isinstance(ob, KnotPointObjective):
                d.kind = _lib.OBJ_KNOT
                d.fn, d.program = knot_fn(ob.l, _lib.L_FUNCS, _lib.L_PROGRAM, len(ob.var_offs))
                vo, tm = np.asarray(ob.var_offs, np.int32), np.asarray(ob.times, np.int32)
                pr, Qs = _f64(ob.params), _f64(ob.Qs)
                keep += [vo, tm, pr, Qs]
                d.n_vars, d.var_offs, d.n_times, d.times = len(vo), _ip(vo), len(tm), _ip(tm)
                d.n_params, d.params, d.Qs = pr.shape[1], _dp(pr), _dp(Qs)
            elif isinstance(ob, GlobalKnotPointObjective):
                d.kind = _lib.OBJ_GLOBAL_KNOT
                d.fn, d.program = knot_fn(ob.l, _lib.L_FUNCS, _lib.L_PROGRAM, len(ob.var_offs) + len(ob.gvar_offs))
                vo, go, tm = np.asarray(ob.var_offs, np.int32), np.asarray(ob.gvar_offs, np.int32), np.asarray(ob.times, np.int32)
                pr, Qs = _f64(ob.params), _f64(ob.Qs)
                keep += [vo, go, tm, pr, Qs]
                d.n_vars, d.var_offs, d.n_times, d.times = len(vo), _ip(vo), len(tm), _ip(tm)
                d.n_gvars, d.gvar_offs = len(go), _ip(go)
                d.n_params, d.params, d.Qs = pr.shape[1], _dp(pr), _dp(Qs)
                if len(go) == 0:  # no global variables at all: an ordinary knot objective
                    d.kind = _lib.OBJ_KNOT
            elif isinstance(ob, NullObjective):
                d.kind = _lib.OBJ_NULL
            else:
                raise UnsupportedComponent(f"objective {type(ob).__name__} is outside the device path")

        cons = (_lib.ConstraintDesc * max(1, len(self.constraints)))()
        for i, c in enumerate(self.constraints):
            d = cons[i]
            d.fn, d.program = knot_fn(c.g, _lib.G_FUNCS, _lib.G_PROGRAM,
                                      len(c.var_offs) + (len(c.gvar_offs) if isinstance(c, NonlinearGlobalKnotPointConstraint) else 0))
            d.equality = int(c.equality)
            vo, tm, pr = np.asarray(c.var_offs, np.int32), np.asarray(c.times, np.int32), _f64(c.params)
            keep += [vo, tm, pr]
            d.n_vars, d.var_offs, d.n_times, d.times = len(vo), _ip(vo), len(tm), _ip(tm)
            d.g_dim, d.n_params, d.params = c.g_dim, pr.shape[1], _dp(pr)
            if isinstance(c, NonlinearGlobalKnotPointConstraint):
                go = np.asarray(c.gvar_offs, np.int32)
                keep.append(go)
                d.n_gvars, d.gvar_offs = len(go), _ip(go)

        Z0a = _f64(t.vec() if Z0 is None else Z0).reshape(-1)
        keep.append(Z0a)
        desc = _lib.ProblemDesc()
        desc.abi_version = _lib.ABI_VERSION
        desc.N, desc.z, desc.dt_off = t.N, t.dim, t.components[t.timestep].start
        desc.batch, desc.eval_hessian, desc.device = self.batch, int(self.eval_hessian), device
        if shard is not None:
            desc.shard_k0, desc.shard_k1 = int(shard[0]), int(shard[1])
        desc.n_integrators, desc.n_objectives, desc.n_constraints = len(prob.integrators), len(terms), len(self.constraints)
        desc.integrators, desc.objectives, desc.constraints = ints, objs, cons
        desc.Z0 = _dp(Z0a)
        desc.global_dim = t.global_dim
        progs = (_lib.KnotProgramDesc * max(1, len(programs)))()
        for i, (ops, out, consts) in enumerate(programs):
            keep += [ops, out, consts]
            progs[i].n_ops, progs[i].ops = ops.shape[0], _ip(ops)
            progs[i].n_out, progs[i].out = out.size, _ip(out)
            progs[i].n_consts, progs[i].consts = consts.size, _dp(consts)
        desc.n_programs, desc.programs = len(programs), progs
        h = C.c_void_p()
        rc = lib.dto_create(C.byref(desc), C.byref(h))
        if rc != _lib.DTO_OK:
            msg = lib.dto_last_error(None).decode()
            if rc == _lib.DTO_ERR_UNSUPPORTED:
                raise UnsupportedComponent(msg)
            raise _lib.DtoError(rc, msg)
        self._h = h
        si = _lib.SizeInfo()
        _lib.check(lib.dto_sizes(h, C.byref(si)), h)
        self.n_vars = si.n_vars
        self.n_dynamics_constraints = si.n_dynamics_cons
        self.n_nonlinear_constraints = si.n_nonlinear_cons
        self.n_constraints = si.n_cons
        self.nnz_jacobian = si.nnz_jac
        self.nnz_hessian = si.nnz_hess
        self.n_constraint_hessian_elements = si.nnz_hess
        self.sharded = shard is not None
        sl = _lib.ShardLayout()
        _lib.check(lib.dto_shard_info(h, C.byref(sl)), h)
        self.shard_layout = sl
        self.global_dim = t.global_dim
        self.n_z_in = sl.z_halo_end - sl.z_begin + t.global_dim  # doubles of Z one call consumes (per problem)
        self._jac_structure = None
        self._hess_structure = None
        if verbose:
            print(f"      building evaluator: {len(prob.integrators)} integrators, {len(self.constraints)} nonlinear constraints")
            print(f"      dynamics constraints: {self.n_dynamics_constraints}, nonlinear constraints: {self.n_nonlinear_constraints}")
            print(f"      jacobian structure: {self.nnz_jacobian} nonzeros")
            print(f"      hessian structure: {self.nnz_hessian} nonzeros")
            print("      evaluator ready")

    # ---- lifetime ----
    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            self._lib.dto_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- MOI interface ----
    def initialize(self, features=None):
        return None

    def features_available(self):
        return ["Grad", "Jac", "Hess"] if self.eval_hessian else ["Grad", "Jac"]

    def _z(self, Z):
        Z = _f64(Z).reshape(-1)
        if Z.size != self.batch * self.n_z_in:
            raise ValueError(f"Z has {Z.size} entries, expected {self.batch * self.n_z_in}")
        return Z

    def _out(self, out, n):
        if not (isinstance(out, np.ndarray) and out.dtype == np.float64 and out.flags.c_contiguous and out.size == n):
            raise ValueError(f"output must be a contiguous float64 array of {n} entries")
        return out

    def eval_objective(self, Z):
        Z = self._z(Z)
        J = np.empty(self.batch)
        _lib.check(self._lib.dto_eval_objective(self._h, Z.ctypes.data, J.ctypes.data), self._h)
        return float(J[0]) if self.batch == 1 else J

    def eval_objective_gradient(self, grad, Z):
        Z = self._z(Z)
        n = self.shard_layout.z_end - self.shard_layout.z_begin + self.global_dim
        self._out(grad, self.batch * n)
        _lib.check(self._lib.dto_eval_gradient(self._h, Z.ctypes.data, grad.ctypes.data), self._h)

    def eval_constraint(self, g, Z):
        Z = self._z(Z)
        self._out(g, self.batch * self.n_constraints)
        _lib.check(self._lib.dto_eval_constraint(self._h, Z.ctypes.data, g.ctypes.data), self._h)

    def eval_constraint_jacobian(self, J, Z):
        Z = self._z(Z)
        self._out(J, self.batch * self.nnz_jacobian)
        _lib.check(self._lib.dto_eval_jacobian(self._h, Z.ctypes.data, J.ctypes.data), self._h)

    def eval_hessian_lagrangian(self, H, Z, sigma, mu):
        Z = self._z(Z)
        mu = _f64(mu).reshape(-1)
        if mu.size != self.batch * self.n_constraints:
            raise ValueError("mu has the wrong length")
        self._out(H, self.batch * self.nnz_hessian)
        _lib.check(self._lib.dto_eval_hessian(self._h, Z.ctypes.data, float(sigma), mu.ctypes.data, H.ctypes.data), self._h)

    def _w(self, w, n):
        w = _f64(w).reshape(-1)
        if w.size != n:
            raise ValueError(f"w has {w.size} entries, expected {n}")
        return w

    def eval_constraint_jacobian_product(self, y, x, w):
        x, w = self._z(x), self._w(w, self.batch * self.n_vars)
        self._out(y, self.batch * self.n_constraints)
        _lib.check(self._lib.dto_eval_jacobian_product(self._h, x.ctypes.data, w.ctypes.data, y.ctypes.data), self._h)

    def eval_constraint_jacobian_transpose_product(self, y, x, w):
        x, w = self._z(x), self._w(w, self.batch * self.n_constraints)
        self._out(y, self.batch * self.n_vars)
        _lib.check(self._lib.dto_eval_jacobian_transpose_product(self._h, x.ctypes.data, w.ctypes.data, y.ctypes.data), self._h)

    def eval_all(self, Z, sigma=1.0, mu=None, J=None, grad=None, g=None, jac=None, hess=None):
        """One fused pass over one iterate (any output may be None)."""
        Z = self._z(Z)
        mu_p = None
        if mu is not None:
            mu = self._w(mu, self.batch * self.n_constraints)
            mu_p = mu.ctypes.data
        n_grad = self.shard_layout.z_end - self.shard_layout.z_begin + self.global_dim
        for out, n in ((J, 1), (grad, n_grad), (g, self.n_constraints), (jac, self.nnz_jacobian), (hess, self.nnz_hessian)):
            if out is not None:
                self._out(out, self.batch * n)
        p = lambda a: None if a is None else a.ctypes.data
        _lib.check(self._lib.dto_eval_all(self._h, Z.ctypes.data, float(sigma), mu_p, p(J), p(grad), p(g), p(jac), p(hess)), self._h)

    def upload(self, Z):
        """Make ``Z`` the resident iterate without evaluating anything (returns after the copy has completed)."""
        Z = self._z(Z)
        _lib.check(self._lib.dto_upload(self._h, Z.ctypes.data), self._h)

    def cache_stats(self):
        """(hits, misses) of the iterate cache since creation."""
        a, b = C.c_int64(), C.c_int64()
        _lib.check(self._lib.dto_cache_stats(self._h, C.byref(a), C.byref(b)), self._h)
        return a.value, b.value

    def register_outputs(self, jac=None, hess=None):
        """``dto_register_outputs``: page-lock the solver's own value arrays and write their structural constants once;
        callbacks that are handed these arrays afterwards move only the value-dependent entries.  The arrays must
        stay alive and must only be read by the caller until ``unregister_outputs`` / ``close``."""
        if jac is not None:
            self._out(jac, self.nnz_jacobian)
        if hess is not None:
            self._out(hess, self.nnz_hessian)
        self._registered = (jac, hess)  # keep them alive
        p = lambda a: None if a is None else a.ctypes.data
        _lib.check(self._lib.dto_register_outputs(self._h, p(jac), p(hess)), self._h)

    def unregister_outputs(self):
        _lib.check(self._lib.dto_unregister_outputs(self._h), self._h)
        self._registered = None

    def eval_all_dev(self, dZ, sigma=1.0, dmu=0, dJ=0, dgrad=0, dg=0, djac=0, dhess=0):
        """Device-pointer variant: arguments are raw device addresses (e.g. ``tensor.data_ptr()``);
        enqueues on the handle's stream without synchronising."""
        _lib.check(self._lib.dto_eval_all_dev(self._h, dZ, float(sigma), dmu or None, dJ or None, dgrad or None, dg or None,
                                              djac or None, dhess or None), self._h)

    def violation_dev(self, dg, dviol):
        _lib.check(self._lib.dto_violation_dev(self._h, dg, dviol), self._h)

    def synchronize(self):
        _lib.check(self._lib.dto_synchronize(self._h), self._h)

    @property
    def stream(self):
        return self._lib.dto_stream(self._h)

    def jacobian_structure(self):
        """1-based ``(rows, cols)`` int64 arrays in the reference's order (``zip`` them for the
        reference's ``Vector{Tuple{Int,Int}}``)."""
        if self._jac_structure is None:
            r, c = np.empty(self.nnz_jacobian, np.int64), np.empty(self.nnz_jacobian, np.int64)
            _lib.check(self._lib.dto_jac_structure(self._h, r.ctypes.data_as(_lib.c_int64_p), c.ctypes.data_as(_lib.c_int64_p)), self._h)
            self._jac_structure = (r, c)
        return self._jac_structure

    def hessian_lagrangian_structure(self):
        if self._hess_structure is None:
            r, c = np.empty(self.nnz_hessian, np.int64), np.empty(self.nnz_hessian, np.int64)
            _lib.check(self._lib.dto_hess_structure(self._h, r.ctypes.data_as(_lib.c_int64_p), c.ctypes.data_as(_lib.c_int64_p)), self._h)
            self._hess_structure = (r, c)
        return self._hess_structure

    def constraint_bounds(self):
        lo, hi = np.empty(self.n_constraints), np.empty(self.n_constraints)
        _lib.check(self._lib.dto_constraint_bounds(self._h, _dp(lo), _dp(hi)), self._h)
        return lo, hi

    def shard_maps(self):
        """Global 0-based positions of this shard's rows / Jacobian values / Hessian values."""
        r = np.empty(self.n_constraints, np.int64)
        j = np.empty(self.nnz_jacobian, np.int64)
        hh = np.empty(self.nnz_hessian, np.int64)
        i64 = lambda a: a.ctypes.data_as(_lib.c_int64_p)
        _lib.check(self._lib.dto_shard_maps(self._h, i64(r), i64(j), i64(hh)), self._h)
        return r, j, hh

    def shard_export(self):
        """64-byte CUDA-IPC handle of this shard's exchange window."""
        buf = C.create_string_buffer(64)
        _lib.check(self._lib.dto_shard_export(self._h, buf), self._h)
        return buf.raw

    def shard_link(self, rank, world, handles):
        """Map the exchange windows of all ``world`` shards (``handles``: their ``shard_export()`` in rank order)."""
        raw = b"".join(bytes(x) for x in handles)
        if len(raw) != 64 * world:
            raise ValueError("need one 64-byte handle per rank")
        _lib.check(self._lib.dto_shard_link(self._h, int(rank), int(world), C.create_string_buffer(raw, len(raw))), self._h)

    @staticmethod
    def shard_link_local(evaluators):
        """Link several shards that live in this process (rank order)."""
        lib = _lib.load()
        arr = (C.c_void_p * len(evaluators))(*[e._h for e in evaluators])
        rc = lib.dto_shard_link_local(arr, len(evaluators))
        if rc != _lib.DTO_OK:
            raise _lib.DtoError(rc, "; ".join(lib.dto_last_error(e._h).decode() for e in evaluators))

    def upload_dev(self, dZ):
        _lib.check(self._lib.dto_upload_dev(self._h, dZ), self._h)

    def allreduce_scalars_dev(self, dJ, dviol):
        _lib.check(self._lib.dto_allreduce_scalars_dev(self._h, dJ, dviol), self._h)

    def shard_scalars_dev(self, dg, dJ, dviol):
        """Violation of this shard's residuals ``dg`` and the (sum, max) exchange with the other shards in one kernel."""
        _lib.check(self._lib.dto_shard_scalars_dev(self._h, dg, dJ, dviol), self._h)

    @property
    def local_Z_ptr(self):
        return self._lib.dto_local_Z(self._h)

    @property
    def launch_count(self):
        return int(self._lib.dto_launch_count(self._h))

    @property
    def last_d2h_bytes(self):
        """Bytes the last host-pointer evaluation moved device -> host."""
        return int(self._lib.dto_last_download_bytes(self._h))

    def kernel_timing(self, enable=True):
        _lib.check(self._lib.dto_kernel_timing(self._h, int(enable)), self._h)

    def kernel_time_ms(self):
        ms, n = C.c_double(), C.c_int64()
        _lib.check(self._lib.dto_kernel_time_ms(self._h, C.byref(ms), C.byref(n)), self._h)
        return ms.value, n.value

    def kernel_variant(self, i=0):
        return self._lib.dto_kernel_variant(self._h, i).decode()

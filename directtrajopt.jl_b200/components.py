"""Host-side mirror of the reference's problem components for the hot path:
integrators (src/integrators/*.jl), objectives (src/objectives/{regularizers,minimum_time_objective,
knot_point_objectives,_objectives}.jl) and NonlinearKnotPointConstraint
(src/constraints/nonlinear/knot_point_constraint.jl).  Same names and argument meaning; the opaque
Julia closures (G, g, l) are *lowered to data*: a bilinear generator to (G_drift, G_drives) by
probing, knot functions to entries of the device catalogue (``KnotFunction``) or to traced device programs
(``KnotProgram``, knot_program.py).  A component that cannot be lowered raises at construction -- never mid-solve,
never a CPU fallback."""
from __future__ import annotations

import numpy as np

from . import _lib


class UnsupportedComponent(ValueError):
    pass


# ------------------------------------------------------------------------------------------------
# device catalogue entries
# ------------------------------------------------------------------------------------------------
class KnotFunction:
    """One entry of the device catalogue of knot functions; ``params(i)`` gives the parameter block
    for the i-th listed time."""

    def __init__(self, name, params, g_dim=1, per_time=None):
        self.name = name
        self._params = np.atleast_1d(np.asarray(params, float))
        self.g_dim = g_dim
        self._per_time = per_time  # optional (n_times, np) array overriding the shared block

    def param_table(self, n_times):
        if self._per_time is not None:
            t = np.asarray(self._per_time, float).reshape(n_times, -1)
            return np.ascontiguousarray(t)
        return np.ascontiguousarray(np.tile(self._params, (n_times, 1)))


def NormMinus(c=1.0):
    """g(v) = [norm(v) - c]"""
    return KnotFunction("norm_minus_c", [c])


def NormSqMinus(c=1.0):
    """g(v) = [norm(v)^2 - c]"""
    return KnotFunction("normsq_minus_c", [c])


def SqDistMinus(target, c=0.0):
    """g(v) = [norm(v - target)^2 - c]"""
    return KnotFunction("sqdist_minus_c", np.concatenate([[c], np.asarray(target, float)]))


def LinearMap(A, b=None):
    """g(v) = A v - b"""
    A = np.atleast_2d(np.asarray(A, float))
    b = np.zeros(A.shape[0]) if b is None else np.asarray(b, float)
    return KnotFunction("linear", np.concatenate([[A.shape[0]], A.reshape(-1, order="F"), b]), g_dim=A.shape[0])


def NormSqPlus(p=0.0, per_time=None):
    """l(v, p) = norm(v)^2 + p"""
    return KnotFunction("normsq_plus_p", [p], per_time=None if per_time is None else np.asarray(per_time, float).reshape(-1, 1))


def SqDist(target, per_time=None):
    """l(v) = norm(v - target)^2"""
    return KnotFunction("sqdist", target, per_time=per_time)


def LinearCost(c):
    """l(v) = c' v"""
    return KnotFunction("linear", c)


def SplitSqDist():
    """l(v) = norm(v[:h] - v[h:])^2, h = len(v)/2: e.g. a state against a goal held in a global variable
    (global_objectives.jl:364-369)"""
    return KnotFunction("split_sqdist", [0.0])


def NormProduct(n1, c1=1.0, c2=1.0):
    """g(v) = [norm(v1) - c1; norm(v1) norm(v2) - c2] with v = [v1 (n1 entries); v2]: the reference's test function
    for knot + global variables (global_knot_point_constraint.jl:267-270)"""
    return KnotFunction("norm_product", [c1, c2, float(n1)], g_dim=2)


def IsoInfidelity(goal):
    """l(psi_iso) = 1 - |<goal|psi>|^2 for iso-vectors [re; im]"""
    return KnotFunction("iso_infidelity", goal)


def _knot_function(fn, catalogue, who, n_vars, objective):
    """Check the knot function of a term: a catalogue ``KnotFunction`` or a ``KnotProgram`` (traced here, where the
    term's variable count is known).  A bare callable is refused: it has to be wrapped so that it is clear it will be
    traced.  Returns the term's g_dim."""
    from .knot_program import KnotProgram

    if isinstance(fn, KnotProgram):
        gd = fn.g_dim(n_vars)
        if objective and gd != 1:
            raise UnsupportedComponent(f"{who}: a KnotProgram objective must return one value, not {gd}")
        return gd
    if not isinstance(fn, KnotFunction) or fn.name not in catalogue:
        kind = "objective" if objective else "constraint"
        raise UnsupportedComponent(f"{who}: expected a KnotProgram or a KnotFunction from the device {kind} catalogue")
    return fn.g_dim


def _spec_fn(fn):
    """What the CPU oracle receives as the term's function: the catalogue name, or the KnotProgram (a callable)."""
    return fn.name if isinstance(fn, KnotFunction) else fn


def _offsets(traj, names):
    if isinstance(names, str):
        names = [names]
    offs = []
    for n in names:
        offs += list(traj.components[n])
    return list(names), np.asarray(offs, dtype=np.int32)


# ------------------------------------------------------------------------------------------------
# integrators
# ------------------------------------------------------------------------------------------------
class AbstractIntegrator:
    pass


class BilinearIntegrator(AbstractIntegrator):
    """``BilinearIntegrator(G, x, u, traj)``: x_{k+1} - exp(dt_k G(u_k)) x_k = 0
    (bilinear_integrator.jl:61-85).  ``G`` is either a callable ``u -> matrix`` that is affine in u
    (checked, then lowered to data) or a pair ``(G_drift, G_drives)``."""

    kind = "bilinear"

    def __init__(self, G, x, u, traj):
        self.x_name, self.u_name = x, u
        self.x_dim, self.u_dim = traj.dims[x], traj.dims[u]
        self.var_dim = 2 * self.x_dim + self.u_dim + 1
        self.dim = self.x_dim * (traj.N - 1)
        n, m = self.x_dim, self.u_dim
        if callable(G):
            G0 = np.asarray(G(np.zeros(m)), float)
            drives = [np.asarray(G(np.eye(m)[i]), float) - G0 for i in range(m)]
            utest = np.random.default_rng(0).standard_normal(m)
            Gt = G0 + sum(utest[i] * drives[i] for i in range(m))
            if not np.allclose(np.asarray(G(utest), float), Gt, rtol=1e-12, atol=1e-12 * (1 + np.abs(Gt).max())):
                raise UnsupportedComponent("BilinearIntegrator: G(u) must be affine in u to be lowered to (G_drift, G_drives)")
        else:
            G0, drives = G
            G0 = np.asarray(G0, float)
            drives = [np.asarray(d, float) for d in drives]
        if G0.shape != (n, n) or len(drives) != m or any(d.shape != (n, n) for d in drives):
            raise ValueError("generator shapes do not match the state/drive dimensions")
        self.G = np.stack([G0] + drives) if m else G0[None]
        self.batch_G = None  # optional (batch, m+1, n, n) per-problem generators

    def to_spec(self):
        return {"kind": "bilinear", "x": self.x_name, "u": self.u_name, "G": self.G}


class DerivativeIntegrator(AbstractIntegrator):
    """``DerivativeIntegrator(x, xdot, traj)``: x_{k+1} - x_k - dt_k xdot_k = 0 (derivative_integrator.jl:26-49)."""

    kind = "derivative"

    def __init__(self, x, xdot, traj):
        self.x_name, self.xdot_name = x, xdot
        self.x_dim = traj.dims[x]
        if traj.dims[xdot] != self.x_dim:
            raise ValueError("derivative component must have the variable's dimension")
        self.var_dim = 3 * self.x_dim + 1
        self.dim = self.x_dim * (traj.N - 1)

    def to_spec(self):
        return {"kind": "derivative", "x": self.x_name, "xdot": self.xdot_name}


class CarrierGenerator:
    """Data form of a time-dependent generator
    ``G(u, t) = G0 + sum_i u_i (cos(w_i t + phi_i) A_i + sin(w_i t + phi_i) B_i) + sum_j cos(wd_j t + phd_j) D_j``
    (the family the device kernel integrates; replaces the closure of
    time_dependent_bilinear_integrator.jl:70-78)."""

    def __init__(self, G0, A, B=None, omega=None, phi=None, D=None, omega_d=None, phi_d=None):
        self.G0 = np.asarray(G0, float)
        n = self.G0.shape[0]
        self.A = np.asarray(A, float).reshape(-1, n, n)
        m = self.A.shape[0]
        self.B = np.zeros_like(self.A) if B is None else np.asarray(B, float).reshape(m, n, n)
        self.omega = np.zeros(m) if omega is None else np.asarray(omega, float).reshape(m)
        self.phi = np.zeros(m) if phi is None else np.asarray(phi, float).reshape(m)
        self.D = np.zeros((0, n, n)) if D is None else np.asarray(D, float).reshape(-1, n, n)
        nc = self.D.shape[0]
        self.omega_d = np.zeros(nc) if omega_d is None else np.asarray(omega_d, float).reshape(nc)
        self.phi_d = np.zeros(nc) if phi_d is None else np.asarray(phi_d, float).reshape(nc)

    def __call__(self, u, t):
        G = self.G0.copy()
        for i in range(self.A.shape[0]):
            G += u[i] * (np.cos(self.omega[i] * t + self.phi[i]) * self.A[i] + np.sin(self.omega[i] * t + self.phi[i]) * self.B[i])
        for j in range(self.D.shape[0]):
            G += np.cos(self.omega_d[j] * t + self.phi_d[j]) * self.D[j]
        return G


class TimeDependentBilinearIntegrator(AbstractIntegrator):
    """``TimeDependentBilinearIntegrator(G, x, u, t, traj; spline_order=1)``
    (time_dependent_bilinear_integrator.jl:60-132).  ``G`` must be a ``CarrierGenerator``.
    ``steps`` fixes the number of RK steps per interval of the device integrator (the reference uses
    adaptive Tsit5; see DESIGN.md)."""

    kind = "tdbilinear"

    def __init__(self, G, x, u, t, traj, spline_order=1, steps=0):
        if not isinstance(G, CarrierGenerator):
            raise UnsupportedComponent("TimeDependentBilinearIntegrator: G(u, t) must be given as a CarrierGenerator")
        if spline_order not in (0, 1):
            raise UnsupportedComponent(f"Unsupported spline order: {spline_order}")
        if traj.N <= 1:
            raise ValueError("Trajectory must have at least two timesteps.")
        self.G = G
        self.x_name, self.u_name, self.t_name = x, u, t
        self.spline_order = spline_order
        self.x_dim, self.u_dim = traj.dims[x], traj.dims[u]
        if traj.dims[t] != 1 or G.G0.shape != (self.x_dim, self.x_dim) or G.A.shape[0] != self.u_dim:
            raise ValueError("generator shapes do not match the trajectory")
        self.dim = self.x_dim * (traj.N - 1)
        self.steps = steps

    def to_spec(self):
        g = self.G
        return {"kind": "tdbilinear", "x": self.x_name, "u": self.u_name, "t": self.t_name, "spline_order": self.spline_order,
                "G0": g.G0, "A": g.A, "B": g.B, "omega": g.omega, "phi": g.phi, "D": g.D, "omega_d": g.omega_d, "phi_d": g.phi_d,
                "steps": self.steps}


# ------------------------------------------------------------------------------------------------
# objectives
# ------------------------------------------------------------------------------------------------
class AbstractObjective:
    def __add__(self, other):
        o1, w1 = (self.objectives, self.weights) if isinstance(self, CompositeObjective) else ([self], [1.0])
        o2, w2 = (other.objectives, other.weights) if isinstance(other, CompositeObjective) else ([other], [1.0])
        return CompositeObjective(list(o1) + list(o2), list(w1) + list(w2))

    def __mul__(self, num):
        if isinstance(self, CompositeObjective):
            return CompositeObjective(self.objectives, [float(num) * w for w in self.weights])
        return CompositeObjective([self], [float(num)])

    __rmul__ = __mul__


class CompositeObjective(AbstractObjective):
    """Flat weighted sum (``+`` flattens, ``*`` scales weights; _objectives.jl:106-187)."""

    def __init__(self, objectives, weights):
        self.objectives, self.weights = list(objectives), [float(w) for w in weights]


class NullObjective(AbstractObjective):
    def __init__(self, traj=None):
        pass

    def to_spec(self, traj):
        return {"kind": "null"}


class QuadraticRegularizer(AbstractObjective):
    """``QuadraticRegularizer(name, traj, R; baseline, times)``:
    J = sum_t 1/2 (dt (v_t - baseline_t))' R (dt (v_t - baseline_t))   (regularizers.jl:38-90)."""

    def __init__(self, name, traj, R, baseline=None, times=None):
        d = traj.dims[name]
        self.name = name
        self.R = np.full(d, float(R)) if np.isscalar(R) else np.asarray(R, float)
        if self.R.shape != (d,):
            raise ValueError("length(R) must equal the component dimension")
        self.baseline = np.zeros((d, traj.N)) if baseline is None else np.asarray(baseline, float).reshape(d, traj.N)
        self.times = list(range(1, traj.N + 1)) if times is None else [int(t) for t in times]

    def to_spec(self, traj):
        return {"kind": "quadreg", "name": self.name, "R": self.R, "baseline": self.baseline, "times": self.times}


class LinearRegularizer(AbstractObjective):
    """``LinearRegularizer(name, traj, R; times)``: J = sum_t dt_t R'v_t   (regularizers.jl:207-313)."""

    def __init__(self, name, traj, R, times=None):
        d = traj.dims[name]
        self.name = name
        self.R = np.full(d, float(R)) if np.isscalar(R) else np.asarray(R, float)
        if self.R.shape != (d,):
            raise ValueError("length(R) must equal the component dimension")
        self.times = list(range(1, traj.N + 1)) if times is None else [int(t) for t in times]

    def to_spec(self, traj):
        return {"kind": "linreg", "name": self.name, "R": self.R, "times": self.times}


class MinimumTimeObjective(AbstractObjective):
    """``MinimumTimeObjective(traj; D=1.0)``: J = D sum_{k<N} dt_k (minimum_time_objective.jl:24-49)."""

    def __init__(self, traj, D=1.0):
        self.D = float(D)

    def to_spec(self, traj):
        return {"kind": "mintime", "D": self.D}


class KnotPointObjective(AbstractObjective):
    """``KnotPointObjective(l, names, traj; times, Qs)``: J = sum_i Q_i l([vars]_{times[i]}, params_i)
    (knot_point_objectives.jl:65-157); ``l`` is a ``KnotProgram`` or a ``KnotFunction`` of the objective catalogue."""

    def __init__(self, l, names, traj, times=None, Qs=None):
        self.l = l
        self.var_names, self.var_offs = _offsets(traj, names)
        _knot_function(l, _lib.L_FUNCS, "KnotPointObjective", len(self.var_offs), objective=True)
        self.times = list(range(1, traj.N + 1)) if times is None else [int(t) for t in times]
        self.Qs = np.ones(len(self.times)) if Qs is None else np.asarray(Qs, float)
        if self.Qs.shape != (len(self.times),):
            raise ValueError("Qs must have the same length as times")
        self.params = l.param_table(len(self.times))
        self.knot_hvp = None  # optional KnotHVP carrier (knot_hvp.jl)

    def to_spec(self, traj):
        return {"kind": "knot", "fn": _spec_fn(self.l), "names": self.var_names, "times": self.times, "params": self.params, "Qs": self.Qs}


def _global_offsets(traj, global_names):
    if global_names is None:  # auto-detect (global_objectives.jl:167-170)
        global_names = list(traj.global_names)
    if isinstance(global_names, str):
        global_names = [global_names]
    offs = []
    for n in global_names:
        offs += list(traj.global_components[n])
    return list(global_names), np.asarray(offs, dtype=np.int32)


class GlobalKnotPointObjective(AbstractObjective):
    """``GlobalKnotPointObjective(l, names, global_names, traj; times, Qs)``:
    J = sum_i Q_i l([knot vars at times[i]; global vars], params_i)  (global_objectives.jl:139-341).
    ``global_names=None`` takes every global component of the trajectory."""

    def __init__(self, l, names, global_names, traj, times=None, Qs=None):
        self.l = l
        self.var_names, self.var_offs = _offsets(traj, names) if names else ([], np.zeros(0, np.int32))
        self.global_names, self.gvar_offs = _global_offsets(traj, global_names)
        _knot_function(l, _lib.L_FUNCS, "GlobalKnotPointObjective", len(self.var_offs) + len(self.gvar_offs), objective=True)
        self.times = list(range(1, traj.N + 1)) if times is None else [int(t) for t in times]
        self.Qs = np.ones(len(self.times)) if Qs is None else np.asarray(Qs, float)
        if self.Qs.shape != (len(self.times),):
            raise ValueError("Qs must have the same length as times")
        self.params = l.param_table(len(self.times))
        self.knot_hvp = None

    def to_spec(self, traj):
        return {"kind": "global_knot", "fn": _spec_fn(self.l), "names": self.var_names, "global_names": self.global_names,
                "times": self.times, "params": self.params, "Qs": self.Qs}


class GlobalObjective(GlobalKnotPointObjective):
    """``GlobalObjective(l, global_names, traj; Q)``: J = Q l(global vars)  (global_objectives.jl:35-130).  Lowered to
    a global-knot term without knot variables, listed once."""

    def __init__(self, l, global_names, traj, Q=1.0):
        super().__init__(l, [], global_names, traj, times=[1], Qs=[Q])
        self.Q = float(Q)


def TerminalObjective(l, names, traj, global_names=None, Q=1.0):
    """``TerminalObjective(l, name(s), traj; Q)`` = KnotPointObjective at ``times=[N]`` (knot_point_objectives.jl:120-157);
    with ``global_names`` the GlobalKnotPointObjective form (global_objectives.jl:347-389)."""
    if global_names is not None:
        return GlobalKnotPointObjective(l, names, global_names, traj, times=[traj.N], Qs=[Q])
    return KnotPointObjective(l, names, traj, times=[traj.N], Qs=[Q])


# ---- KnotHVP: declarable per-knot Hessian-vector-product capability (knot_hvp.jl:45-148) -------
# The reference defines only the carriers and the trait; the apply-math belongs to the consumer.
class KnotHVP:
    pass


class ConstantLowRankHVP(KnotHVP):
    """``ConstantLowRankHVP(A, core)``: per-knot Hessian H = A' G A with constant A (knot_hvp.jl:84-87)."""

    def __init__(self, A, core):
        self.A = np.asarray(A, float)
        if self.A.ndim != 2:
            raise ValueError("A must be a matrix")
        self.core = str(core)


class CustomKnotHVP(KnotHVP):
    """``CustomKnotHVP(apply!, on_device)`` (knot_hvp.jl:122-125)."""

    def __init__(self, apply, on_device):
        self.apply = apply
        self.on_device = bool(on_device)


def knot_hvp(obj, traj):
    """Trait: the declared per-knot HVP capability of ``obj``, or ``None`` (knot_hvp.jl:148 and the
    KnotPointObjective method below it)."""
    return getattr(obj, "knot_hvp", None)


# ------------------------------------------------------------------------------------------------
# constraints
# ------------------------------------------------------------------------------------------------
class AbstractNonlinearConstraint:
    pass


class NonlinearKnotPointConstraint(AbstractNonlinearConstraint):
    """``NonlinearKnotPointConstraint(g, names, traj; times, equality)`` (knot_point_constraint.jl:27-107);
    ``g`` is a ``KnotProgram`` or a ``KnotFunction`` of the constraint catalogue."""

    def __init__(self, g, names, traj, times=None, equality=True):
        self.g = g
        self.var_names, self.var_offs = _offsets(traj, names)
        self.g_dim = _knot_function(g, _lib.G_FUNCS, "NonlinearKnotPointConstraint", len(self.var_offs), objective=False)
        self.equality = bool(equality)
        self.times = list(range(1, traj.N + 1)) if times is None else [int(t) for t in times]
        self.params = g.param_table(len(self.times))
        self.var_dim = len(self.var_offs)
        self.dim = self.g_dim * len(self.times)

    def to_spec(self, traj):
        return {"kind": "knot", "fn": _spec_fn(self.g), "names": self.var_names, "times": self.times, "params": self.params,
                "equality": self.equality}


class NonlinearGlobalKnotPointConstraint(AbstractNonlinearConstraint):
    """``NonlinearGlobalKnotPointConstraint(g, names, global_names, traj; times, equality)``: g([knot vars; global vars])
    at every listed time (global_knot_point_constraint.jl:30-256)."""

    def __init__(self, g, names, global_names, traj, times=None, equality=True):
        self.g = g
        self.var_names, self.var_offs = _offsets(traj, names) if names else ([], np.zeros(0, np.int32))
        self.global_names, self.gvar_offs = _global_offsets(traj, global_names)
        self.g_dim = _knot_function(g, _lib.G_FUNCS, "NonlinearGlobalKnotPointConstraint", len(self.var_offs) + len(self.gvar_offs),
                                    objective=False)
        self.equality = bool(equality)
        self.times = list(range(1, traj.N + 1)) if times is None else [int(t) for t in times]
        self.params = g.param_table(len(self.times))
        self.var_dim = len(self.var_offs)
        self.global_dim = len(self.gvar_offs)
        self.combined_dim = self.var_dim + self.global_dim
        self.dim = self.g_dim * len(self.times)

    def to_spec(self, traj):
        return {"kind": "global_knot", "fn": _spec_fn(self.g), "names": self.var_names, "global_names": self.global_names,
                "times": self.times, "params": self.params, "equality": self.equality}


class NonlinearGlobalConstraint(NonlinearGlobalKnotPointConstraint):
    """``NonlinearGlobalConstraint(g, global_names, traj; equality)``: g(global vars) (global_constraint.jl:24-159).
    Lowered to a global-knot constraint without knot variables, listed once (rows = g_dim)."""

    def __init__(self, g, global_names, traj, equality=True):
        super().__init__(g, [], global_names, traj, times=[1], equality=equality)

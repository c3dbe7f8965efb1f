"""User-written knot functions as traced device programs.

The reference's users pass closures ``g(v)`` / ``g(v, p)`` / ``l(v)`` to ``NonlinearKnotPointConstraint``,
``KnotPointObjective`` and the global variants (knot_point_constraint.jl:76-83, knot_point_objectives.jl:65-72).
``KnotProgram(f)`` makes such a closure runnable on the device: when the term is constructed (the first moment the
number of variables is known) ``f`` is called once on arrays of tracers, and the operations it performs are recorded as
an SSA tape of the operations of include/dto_b200.h (``DTO_OP_*``).  The library compiles that tape and differentiates
it on the GPU with the same hyper-dual templates as the catalogue, so values, Jacobians, Hessians and the
value-dependent stored sparsity pattern all come from one device implementation.

What ``f`` may do: ``+ - * /``, unary minus, ``** c`` for a number ``c``, ``v @ w`` and ``sum`` over tracer arrays, and the
NumPy ufuncs ``np.sqrt, np.exp, np.log, np.sin, np.cos, np.tanh`` (for object arrays NumPy calls the element's method of
the same name).  A data-dependent branch (``if x > 0``, ``abs``, ``min``/``max``), a traced exponent and any other
ufunc raise ``UnsupportedComponent`` at construction.
"""
from __future__ import annotations

import struct

import numpy as np

from .components import UnsupportedComponent

OP_VAR, OP_PARAM, OP_CONST = 1, 2, 3
OP_ADD, OP_SUB, OP_MUL, OP_DIV = 4, 5, 6, 7
OP_NEG, OP_SQRT, OP_EXP, OP_LOG, OP_SIN, OP_COS, OP_TANH = 8, 9, 10, 11, 12, 13, 14
OP_POWC = 15
UNARY = {"sqrt": OP_SQRT, "exp": OP_EXP, "log": OP_LOG, "sin": OP_SIN, "cos": OP_COS, "tanh": OP_TANH}


class Tape:
    """SSA tape: ``ops`` is an (n, 3) int32 array of {opcode, a, b}, ``out`` the output value indices, ``consts`` the
    constants.  Identical operations on identical operands are recorded once (common subexpressions are shared)."""

    def __init__(self):
        self._ops, self._memo, self._consts, self._cmemo = [], {}, [], {}
        self.out = None

    def node(self, op, a, b=0):
        key = (op, a, b)
        i = self._memo.get(key)
        if i is None:
            i = self._memo[key] = len(self._ops)
            self._ops.append(key)
        return Tracer(self, i)

    def const_index(self, x):
        x = float(x)
        key = struct.pack("<d", x)
        if key not in self._cmemo:
            self._cmemo[key] = len(self._consts)
            self._consts.append(x)
        return self._cmemo[key]

    def const(self, x):
        return self.node(OP_CONST, self.const_index(x))

    @property
    def ops(self):
        return np.asarray(self._ops, dtype=np.int32).reshape(-1, 3)

    @property
    def consts(self):
        return np.asarray(self._consts, dtype=np.float64)

    def replay(self, v, p=()):
        """Evaluate the tape on floats (NumPy semantics of every operation)."""
        val = []
        c = self._consts
        for op, a, b in self._ops:
            if op == OP_VAR: r = float(v[a])
            elif op == OP_PARAM: r = float(p[a])
            elif op == OP_CONST: r = c[a]
            elif op == OP_ADD: r = val[a] + val[b]
            elif op == OP_SUB: r = val[a] - val[b]
            elif op == OP_MUL: r = val[a] * val[b]
            elif op == OP_DIV: r = val[a] / val[b]
            elif op == OP_NEG: r = -val[a]
            elif op == OP_POWC: r = float(np.float64(val[a]) ** c[b])
            else: r = float(getattr(np, {v_: k for k, v_ in UNARY.items()}[op])(val[a]))
            val.append(r)
        return np.array([val[i] for i in self.out])


def _unsupported(what):
    raise UnsupportedComponent(f"KnotProgram: {what} cannot be traced into a device program")


class Tracer:
    """A value of the traced function: an index into its tape."""

    __slots__ = ("tape", "i")
    __array_priority__ = 100  # `ndarray (op) Tracer` defers to the tracer's reflected operator

    def __init__(self, tape, i):
        self.tape, self.i = tape, i

    def _arg(self, x):
        if isinstance(x, Tracer):
            if x.tape is not self.tape:
                _unsupported("mixing values of two traces")
            return x
        if isinstance(x, (int, float, np.integer, np.floating)) and not isinstance(x, bool):
            return self.tape.const(x)
        if isinstance(x, np.ndarray) and x.ndim == 0:
            return self._arg(x.item())
        return NotImplemented

    def _bin(self, op, x, reflected=False):
        y = self._arg(x)
        if y is NotImplemented:
            return NotImplemented
        a, b = (y, self) if reflected else (self, y)
        return self.tape.node(op, a.i, b.i)

    def __add__(self, x):
        return self._bin(OP_ADD, x)

    def __radd__(self, x):
        if isinstance(x, int) and x == 0:  # sum() starts from the integer 0
            return self
        return self._bin(OP_ADD, x, True)

    def __sub__(self, x):
        return self._bin(OP_SUB, x)

    def __rsub__(self, x):
        return self._bin(OP_SUB, x, True)

    def __mul__(self, x):
        return self._bin(OP_MUL, x)

    def __rmul__(self, x):
        return self._bin(OP_MUL, x, True)

    def __truediv__(self, x):
        return self._bin(OP_DIV, x)

    def __rtruediv__(self, x):
        return self._bin(OP_DIV, x, True)

    def __neg__(self):
        return self.tape.node(OP_NEG, self.i)

    def __pos__(self):
        return self

    def __pow__(self, c):
        if isinstance(c, Tracer):
            _unsupported("x ** y with a traced exponent")
        if isinstance(c, np.ndarray) and c.ndim == 0:
            c = c.item()
        if not isinstance(c, (int, float, np.integer, np.floating)) or isinstance(c, bool):
            return NotImplemented
        return self.tape.node(OP_POWC, self.i, self.tape.const_index(c))

    def __rpow__(self, x):
        _unsupported("x ** y with a traced exponent")

    def sqrt(self):
        return self.tape.node(OP_SQRT, self.i)

    def exp(self):
        return self.tape.node(OP_EXP, self.i)

    def log(self):
        return self.tape.node(OP_LOG, self.i)

    def sin(self):
        return self.tape.node(OP_SIN, self.i)

    def cos(self):
        return self.tape.node(OP_COS, self.i)

    def tanh(self):
        return self.tape.node(OP_TANH, self.i)

    # a scalar tracer passed to a ufunc directly (np.sqrt(v[0]))
    def __array_ufunc__(self, ufunc, method, *inputs, **kwargs):
        if method == "__call__" and not kwargs:
            if ufunc.__name__ in UNARY and len(inputs) == 1:
                return getattr(self, ufunc.__name__)()
            binary = {"add": "__add__", "subtract": "__sub__", "multiply": "__mul__", "true_divide": "__truediv__", "divide": "__truediv__"}
            if ufunc.__name__ in binary and len(inputs) == 2:
                a, b = inputs
                if isinstance(a, Tracer):
                    return getattr(a, binary[ufunc.__name__])(b)
                return getattr(b, "__r" + binary[ufunc.__name__][2:])(a)
            if ufunc.__name__ == "negative":
                return -self
            if ufunc.__name__ == "power" and len(inputs) == 2 and inputs[0] is self:
                return self ** inputs[1]
        _unsupported(f"the ufunc {ufunc.__name__}")

    # branches on traced values: the tape has no control flow
    def __bool__(self):
        _unsupported("a data-dependent branch (truth value of a traced value)")

    def _cmp(self, x):
        _unsupported("a comparison of traced values (data-dependent branch)")

    __lt__ = __le__ = __gt__ = __ge__ = __eq__ = __ne__ = _cmp
    __hash__ = object.__hash__

    def __abs__(self):
        _unsupported("abs (not smooth)")

    def __float__(self):
        _unsupported("converting a traced value to a number")

    def __getattr__(self, name):
        # NumPy applies a ufunc to an object array by calling the element's method of the ufunc's name
        if name.startswith("__"):
            raise AttributeError(name)
        _unsupported(f"the function {name}")


class KnotProgram:
    """``KnotProgram(f, params=None, per_time=None)``: a user knot function for any knot term constructor
    (``NonlinearKnotPointConstraint``, ``KnotPointObjective``, ``TerminalObjective``, ``GlobalObjective``,
    ``GlobalKnotPointObjective``, ``NonlinearGlobalKnotPointConstraint``, ``NonlinearGlobalConstraint``).

    ``f(v)`` -- or ``f(v, p)`` when parameters are given -- receives the term's variables concatenated in the order of
    ``names`` (then the global variables) and returns a sequence of ``g_dim`` values (a constraint) or one value (an
    objective).  ``params`` is one parameter vector for every listed time, ``per_time`` an ``(n_times, n_params)``
    table of one row per listed time (as in the catalogue's ``KnotFunction``)."""

    def __init__(self, f, params=None, per_time=None):
        if not callable(f):
            raise TypeError("KnotProgram needs a callable f(v) or f(v, p)")
        self.f = f
        self.with_params = params is not None or per_time is not None
        self._params = np.atleast_1d(np.asarray([] if params is None else params, float))
        self._per_time = None if per_time is None else np.asarray(per_time, float)
        self.n_params = self._per_time.reshape(self._per_time.shape[0], -1).shape[1] if per_time is not None else self._params.size
        self._tapes = {}

    def param_table(self, n_times):
        if self._per_time is not None:
            return np.ascontiguousarray(self._per_time.reshape(n_times, -1))
        return np.ascontiguousarray(np.tile(self._params, (n_times, 1)))

    def trace(self, n_vars):
        """The tape of ``f`` on ``n_vars`` variables (traced once per variable count)."""
        tape = self._tapes.get(n_vars)
        if tape is None:
            tape = Tape()
            v = np.empty(n_vars, dtype=object)
            for i in range(n_vars):
                v[i] = tape.node(OP_VAR, i)
            p = np.empty(self.n_params, dtype=object)
            for i in range(self.n_params):
                p[i] = tape.node(OP_PARAM, i)
            try:
                res = self.f(v, p) if self.with_params else self.f(v)
            except TypeError as e:
                # a ufunc applied to an object array looks up the element's method of its name; NumPy turns the tracer's
                # refusal into a TypeError
                if isinstance(e.__cause__ or e.__context__, UnsupportedComponent) or "loop of ufunc" in str(e):
                    raise UnsupportedComponent(f"KnotProgram: {e}") from e
                raise
            outs = [res] if isinstance(res, (Tracer, int, float, np.integer, np.floating)) else list(np.asarray(res, dtype=object).reshape(-1))
            if not outs:
                raise UnsupportedComponent("KnotProgram: f returned no values")
            idx = []
            for o in outs:
                if isinstance(o, Tracer):
                    if o.tape is not tape:
                        _unsupported("a value of another trace")
                    idx.append(o.i)
                elif isinstance(o, (int, float, np.integer, np.floating)):
                    idx.append(tape.const(o).i)
                else:
                    raise UnsupportedComponent(f"KnotProgram: f returned a {type(o).__name__}, not a number")
            tape.out = np.asarray(idx, dtype=np.int32)
            self._tapes[n_vars] = tape
        return tape

    def g_dim(self, n_vars):
        return int(self.trace(n_vars).out.size)

    def __call__(self, v, p=()):
        """``f`` itself on the term's variables and one parameter row (the CPU oracle differentiates this call)."""
        return self.f(v, p) if self.with_params else self.f(v)

"""Second-order jets of user knot functions (KnotProgram terms) for the CPU oracle.

The oracle's knot-function table (`dto_oracle._cfun` / `_lfun`) holds closed forms of the device catalogue.  A
KnotProgram carries the user's own function instead; the reference value, gradient and Hessian of such a term come from
calling that function on an object array of `Jet`s: every operation applies its exact chain rule to the whole gradient
vector and Hessian matrix at once.  This is independent of the tracer (it never sees the tape) and of the device's
seeded hyper-dual pairs.  `with_user_functions(monkeypatch)` routes the oracle's callable terms through it and leaves
every catalogue entry to the oracle's own closed forms."""
import numpy as np


class Jet:
    """value, gradient vector and Hessian matrix of a scalar in vd variables"""

    __slots__ = ("v", "g", "H")

    def __init__(self, v, g, H):
        self.v, self.g, self.H = v, g, H

    @staticmethod
    def of(x, like):
        if isinstance(x, Jet):
            return x
        return Jet(float(x), np.zeros_like(like.g), np.zeros_like(like.H))

    def chain(self, f, f1, f2):
        """f(self) given f, f' and f'' at self.v"""
        return Jet(f, f1 * self.g, f1 * self.H + f2 * np.outer(self.g, self.g))

    def __add__(self, x):
        x = Jet.of(x, self)
        return Jet(self.v + x.v, self.g + x.g, self.H + x.H)

    __radd__ = __add__

    def __sub__(self, x):
        x = Jet.of(x, self)
        return Jet(self.v - x.v, self.g - x.g, self.H - x.H)

    def __rsub__(self, x):
        return Jet.of(x, self) - self

    def __mul__(self, x):
        x = Jet.of(x, self)
        o = np.outer(self.g, x.g)
        return Jet(self.v * x.v, self.g * x.v + self.v * x.g, self.H * x.v + self.v * x.H + o + o.T)

    __rmul__ = __mul__

    def __truediv__(self, x):
        x = Jet.of(x, self)
        r = self * x.chain(1 / x.v, -1 / x.v**2, 2 / x.v**3)
        r.v = self.v / x.v
        return r

    def __rtruediv__(self, x):
        return Jet.of(x, self) / self

    def __neg__(self):
        return Jet(-self.v, -self.g, -self.H)

    def __pos__(self):
        return self

    def __pow__(self, c):
        c = float(c)
        x = np.float64(self.v)
        d1 = 0.0 if c == 0 else c * x ** (c - 1)
        d2 = 0.0 if c in (0.0, 1.0) else c * (c - 1) * x ** (c - 2)
        return self.chain(x**c, d1, d2)

    def sqrt(self):
        r = np.sqrt(self.v)
        return self.chain(r, 0.5 / r, -0.25 / (r * self.v))

    def exp(self):
        e = np.exp(self.v)
        return self.chain(e, e, e)

    def log(self):
        return self.chain(np.log(self.v), 1 / self.v, -1 / self.v**2)

    def sin(self):
        return self.chain(np.sin(self.v), np.cos(self.v), -np.sin(self.v))

    def cos(self):
        return self.chain(np.cos(self.v), -np.sin(self.v), -np.cos(self.v))

    def tanh(self):
        t = np.tanh(self.v)
        return self.chain(t, 1 - t * t, -2 * t * (1 - t * t))


def jets(fn, v, p):
    """value, Jacobian and Hessians of a user function fn(v, p) -> (val[gd], J[gd, vd], H[gd, vd, vd])"""
    v = np.asarray(v, float)
    vd = v.size
    x = np.empty(vd, dtype=object)
    for i in range(vd):
        e = np.zeros(vd)
        e[i] = 1.0
        x[i] = Jet(float(v[i]), e, np.zeros((vd, vd)))
    res = fn(x, np.asarray(p, float))
    outs = [res] if isinstance(res, (Jet, int, float, np.floating)) else list(np.asarray(res, dtype=object).reshape(-1))
    zero = Jet(0.0, np.zeros(vd), np.zeros((vd, vd)))
    outs = [Jet.of(o, zero) for o in outs]
    return (np.array([o.v for o in outs]), np.array([o.g for o in outs]).reshape(len(outs), vd),
            np.array([o.H for o in outs]).reshape(len(outs), vd, vd))


def with_user_functions(monkeypatch, orc):
    """let the oracle module evaluate KnotProgram terms (their spec's "fn" is the callable KnotProgram)"""
    c0, l0 = orc._cfun, orc._lfun
    monkeypatch.setattr(orc, "_cfun", lambda fn, v, p: jets(fn, v, p) if callable(fn) else c0(fn, v, p))

    def l(fn, v, p):
        if callable(fn):
            val, J, H = jets(fn, v, p)
            return val[0], J[0], H[0]
        return l0(fn, v, p)

    monkeypatch.setattr(orc, "_lfun", l)

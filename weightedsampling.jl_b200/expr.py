"""Per-particle expressions: the host-side form of what ``vectorize`` builds in the reference
(``src/rewrites.jl:146-219``): constants become one value per particle, a particle variable becomes
its column, calls become elementwise operations.  Here an expression is a small tree that is
serialised to postfix tokens (``ws_tok``) and compiled to device micro-ops by the runtime; anything
that cannot be expressed is rejected with :class:`UnsupportedModelError` when the model is built.

Vector-valued columns (``x .= [0.0, 0.0]``) are ``d`` scalar planes; arithmetic on them is
component-wise, which covers the reference's uses (``x{t} + v``, ``0.1 * I2`` is a build-time
constant).
"""
from __future__ import annotations

import ctypes as C
import struct
import math
import numbers

import numpy as np

from . import _lib as L
from ._lib import UnsupportedModelError


def _unsupported(msg):
    return UnsupportedModelError(L.WS_EUNSUPPORTED, msg)


class Expr:
    """Base class; operators build the tree."""

    def __add__(self, o): return Bin(L.TOK_ADD, self, wrap(o))
    def __radd__(self, o): return Bin(L.TOK_ADD, wrap(o), self)
    def __sub__(self, o): return Bin(L.TOK_SUB, self, wrap(o))
    def __rsub__(self, o): return Bin(L.TOK_SUB, wrap(o), self)
    def __mul__(self, o): return Bin(L.TOK_MUL, self, wrap(o))
    def __rmul__(self, o): return Bin(L.TOK_MUL, wrap(o), self)
    def __truediv__(self, o): return Bin(L.TOK_DIV, self, wrap(o))
    def __rtruediv__(self, o): return Bin(L.TOK_DIV, wrap(o), self)
    def __pow__(self, o): return Bin(L.TOK_POW, self, wrap(o))
    def __rpow__(self, o): return Bin(L.TOK_POW, wrap(o), self)
    def __neg__(self): return Un(L.TOK_NEG, self)
    def __pos__(self): return self
    def __abs__(self): return Un(L.TOK_ABS, self)
    def __getitem__(self, j): return Index(self, j)

    # comparisons give 1.0 / 0.0 per particle (the device form of the reference's Bool columns)
    def __lt__(self, o): return Bin(L.TOK_LT, self, wrap(o))
    def __le__(self, o): return Bin(L.TOK_LE, self, wrap(o))
    def __gt__(self, o): return Bin(L.TOK_LT, wrap(o), self)
    def __ge__(self, o): return Bin(L.TOK_LE, wrap(o), self)
    def eq(self, o): return Bin(L.TOK_EQ, self, wrap(o))
    def __or__(self, o): return Bin(L.TOK_MAX, self, wrap(o))      # a || b on 0/1 values
    def __ror__(self, o): return Bin(L.TOK_MAX, wrap(o), self)
    def __and__(self, o): return Bin(L.TOK_MIN, self, wrap(o))     # a && b
    def __rand__(self, o): return Bin(L.TOK_MIN, wrap(o), self)
    def __invert__(self): return Un(L.TOK_NOT, self)               # !a

    # truthiness would silently build wrong programs: use where(cond, a, b)
    def __bool__(self):
        raise _unsupported("a particle-dependent value cannot be used as a Python condition; use where(cond, a, b)")


class Const(Expr):
    def __init__(self, v):
        self.v = v  # float or 1-d ndarray


class Col(Expr):
    """A particle variable (column) by name: ``getcol(state.store, :name)``."""

    def __init__(self, name):
        self.name = str(name)

    def __repr__(self):
        return f"col({self.name!r})"


class Index(Expr):
    """``x[j]`` on a vector-valued column; ``j`` is 0-based here (the @model front-end converts)."""

    def __init__(self, base, j):
        if isinstance(j, Expr):
            raise _unsupported("particle-dependent indices are outside the device-op set")
        self.base, self.j = base, int(j)


class Bin(Expr):
    def __init__(self, op, a, b):
        self.op, self.a, self.b = op, a, b


class Un(Expr):
    def __init__(self, op, a):
        self.op, self.a = op, a


class Select(Expr):
    """``cond ? a : b`` per particle (``ifelse.(cond, a, b)``, rewrites.jl:193-199); both branches are evaluated."""

    def __init__(self, cond, a, b):
        self.cond, self.a, self.b = wrap(cond), wrap(a), wrap(b)


class Rand(Expr):
    """A fresh standard variate per particle inside a sampler expression: 'n' normal, 'u' uniform [0,1),
    'e' exponential."""

    def __init__(self, kind):
        self.kind = kind


class Param(Expr):
    """Placeholder for a build-time constant that is supplied later (``WS_TOK_PARAM``): the loop variable of a loop
    body that is described once and replayed per element (core.Loop / ``ws_exec``)."""

    def __init__(self, index):
        self.index = int(index)


class RandP(Expr):
    """A variate with a (per-particle) parameter inside a sampler expression: kind 'gamma' = standard
    Gamma(shape), 'poisson' = Poisson(rate) (device rejection samplers on Philox sub-counters)."""

    def __init__(self, kind, arg):
        self.kind, self.arg = kind, wrap(arg)


class NotAProbabilityVector(ValueError):
    """A Categorical argument whose rows are not probability vectors (Distributions' ``isprobvec``)."""


class Table:
    """A build-time constant vector or matrix that particle values index (``ws_table``): ``T[s]`` on a vector,
    ``T[s, k]`` on a matrix, and the row ``T[s, :]`` as the argument of ``Categorical``.  Indices are Julia's,
    1-based.  An index that is not an integer in range reads NaN and counts an index fault, which :func:`run`
    reports as ``IndexError`` when the run ends (the reference throws ``BoundsError`` at the statement)."""

    def __init__(self, values):
        a = np.array(values, dtype=np.float64)
        if a.ndim not in (1, 2) or a.size == 0:
            raise ValueError(f"a table is a non-empty vector or matrix (got shape {a.shape})")
        self.is_vector = a.ndim == 1
        self.values = np.ascontiguousarray(a[None, :] if self.is_vector else a)
        self._probvec = None

    @property
    def shape(self):
        return self.values.shape

    def __getitem__(self, idx):
        idx = idx if isinstance(idx, tuple) else (idx,)
        if self.is_vector:
            if len(idx) != 1:
                raise _unsupported("a vector table takes one index")
            return TableRead(self, 1.0, idx[0])
        if len(idx) != 2:
            raise _unsupported("a matrix table takes two indices, `T[s, k]` (or `T[s, :]` as a Categorical argument)")
        if isinstance(idx[1], slice):
            if idx[1] != slice(None):
                raise _unsupported("only a whole row `T[s, :]` can be sliced out of a table")
            return TableRow(self, idx[0])
        return TableRead(self, idx[0], idx[1])

    def check_probabilities(self):
        """every row >= 0 and summing to 1 within sqrt(eps) (Distributions' ``isprobvec``), else NotAProbabilityVector"""
        if self._probvec is None:
            v = self.values
            sums = v.sum(axis=1)
            bad = np.flatnonzero(~(np.all(v >= 0.0, axis=1) & (np.abs(sums - 1.0) <= math.sqrt(np.finfo(np.float64).eps))))
            self._probvec = bad.size == 0
            self._bad_row = int(bad[0]) + 1 if bad.size else 0
        if not self._probvec:
            raise NotAProbabilityVector(f"row {self._bad_row} of the Categorical probabilities is not a probability vector "
                                        f"(entries must be >= 0 and sum to 1): {self.values[self._bad_row - 1]}")


def table(values):
    """``ws.table(array)``: see :class:`Table`."""
    return values if isinstance(values, Table) else Table(values)


class TableRead(Expr):
    """``T[row, col]`` (1-based, per particle)."""

    def __init__(self, tab, row, col):
        self.table, self.row, self.col = tab, wrap(row), wrap(col)


class TableRow:
    """``T[row, :]``: a row of a table, the argument of ``Categorical`` (not a value of its own)."""

    def __init__(self, tab, row):
        self.table, self.row = tab, wrap(row)


def _cat_row(p):
    """The argument of Categorical as a table row: ``T[s, :]`` or a constant probability vector (a one-row table)."""
    if isinstance(p, TableRow):
        row = p
    elif isinstance(p, Expr) and not isinstance(p, Const):
        raise _unsupported("Categorical with per-particle probability vectors is outside the device-op set (the "
                           "probabilities must be a constant vector or a row `P[s, :]` of a build-time matrix)")
    else:
        v = np.asarray(p.v if isinstance(p, Const) else p, dtype=np.float64)
        if v.ndim != 1:
            raise _unsupported("Categorical takes a probability vector")
        row = TableRow(Table(v), 1.0)
    row.table.check_probabilities()
    return row


class RandCat(Expr):
    """A draw of ``Categorical(row)`` inside a sampler expression (one uniform per particle)."""

    def __init__(self, p):
        self.p = _cat_row(p)


class CatLogp(Expr):
    """``logpdf(Categorical(row), x)``: log p[x] for x in 1..K, -Inf for any other value."""

    def __init__(self, p, x):
        self.p, self.x = _cat_row(p), wrap(x)


def randcat(p): return RandCat(p)
def cat_logpdf(p, x): return CatLogp(p, x)


def randgamma(shape): return RandP("gamma", shape)
def randpoisson(rate): return RandP("poisson", rate)
def randn(): return Rand("n")
def randu(): return Rand("u")
def randexp(): return Rand("e")


def where(cond, a, b):
    if not isinstance(cond, Expr):
        return a if cond else b
    return Select(cond, a, b)


class Vec(Expr):
    """``[e1, e2, ...]`` with per-particle entries."""

    def __init__(self, items):
        self.items = [wrap(i) for i in items]


def wrap(v):
    if isinstance(v, Expr):
        return v
    if isinstance(v, (bool, np.bool_)):
        return Const(1.0 if v else 0.0)  # Bool -> 1.0 / 0.0
    if isinstance(v, numbers.Real):
        return Const(float(v))
    if isinstance(v, (list, tuple)):
        if any(isinstance(i, Expr) for i in v):
            return Vec(v)
        return Const(np.asarray(v, dtype=np.float64))
    if isinstance(v, np.ndarray):
        if v.ndim == 0:
            return Const(float(v))
        if v.ndim == 1:
            return Const(np.asarray(v, dtype=np.float64))
        raise _unsupported(f"{v.ndim}-d array as a particle value is outside the device-op set")
    raise _unsupported(f"value of type {type(v).__name__} is outside the device-op set")


def col(name):
    return Col(name)


def _fn(op):
    def f(x):
        if isinstance(x, Expr):
            return Un(op, x)
        return {L.TOK_EXP: math.exp, L.TOK_LOG: math.log, L.TOK_SQRT: math.sqrt, L.TOK_SIN: math.sin,
                L.TOK_COS: math.cos, L.TOK_ABS: abs, L.TOK_SQUARE: lambda t: t * t, L.TOK_LGAMMA: math.lgamma,
                L.TOK_LOG1P: math.log1p, L.TOK_EXPM1: math.expm1, L.TOK_TAN: math.tan, L.TOK_ATAN: math.atan,
                L.TOK_TANH: math.tanh, L.TOK_FLOOR: math.floor, L.TOK_NOT: lambda t: 0.0 if t else 1.0}[op](x)
    return f


def _fn2(op, py):
    def f(a, b):
        if isinstance(a, Expr) or isinstance(b, Expr):
            return Bin(op, wrap(a), wrap(b))
        return py(a, b)
    return f


exp = _fn(L.TOK_EXP)
log = _fn(L.TOK_LOG)
sqrt = _fn(L.TOK_SQRT)
sin = _fn(L.TOK_SIN)
cos = _fn(L.TOK_COS)
abs2 = _fn(L.TOK_SQUARE)
lgamma = _fn(L.TOK_LGAMMA)
log1p = _fn(L.TOK_LOG1P)
expm1 = _fn(L.TOK_EXPM1)
tan = _fn(L.TOK_TAN)
atan = _fn(L.TOK_ATAN)
tanh = _fn(L.TOK_TANH)
floor = _fn(L.TOK_FLOOR)
minimum = _fn2(L.TOK_MIN, min)
maximum = _fn2(L.TOK_MAX, max)


# ------------------------------------------------------------------------------------------------
# Julia Base functions that have no micro-op of their own: compositions of the ones above, written to give Julia's
# result (signed zeros, NaN propagation, ties) on particle expressions and plain Python arithmetic on build-time numbers.
# (`vectorize` broadcasts ANY Julia function over particle columns, rewrites.jl:150-163; the device-op set is closed,
# so the common scalar ones are spelled out here.)
# ------------------------------------------------------------------------------------------------
_LN2, _LN10 = math.log(2.0), math.log(10.0)


def _is_expr(*xs):
    return any(isinstance(x, Expr) for x in xs)


def _has_draw(e):
    if isinstance(e, (Rand, RandP, RandCat)):
        return True
    return isinstance(e, Expr) and any(_has_draw(v) for v in vars(e).values() if isinstance(v, (Expr, list, tuple))) or \
        (isinstance(e, (list, tuple)) and any(_has_draw(v) for v in e))


def _reuses_args(fn):
    """These compositions mention an argument more than once; an expression is a TREE, so a fresh variate inside it
    (`randn()` in a sampler closure) would be drawn once per mention.  Refuse instead of sampling wrongly."""
    def f(*a):
        if any(_has_draw(x) for x in a):
            raise _unsupported(f"{fn.__name__}() of an expression that contains a fresh variate: assign the draw to a "
                               "particle variable first (the composition would evaluate it more than once)")
        return fn(*a)
    f.__name__ = fn.__name__
    f.__doc__ = fn.__doc__
    return f


@_reuses_args
def isnan(x):
    return ~(x.eq(x)) if isinstance(x, Expr) else math.isnan(x)


def isinf(x):
    return abs(x).eq(math.inf) if isinstance(x, Expr) else math.isinf(x)


def isfinite(x):
    return (abs(x) < math.inf) if isinstance(x, Expr) else math.isfinite(x)


@_reuses_args
def sign(x):
    if isinstance(x, Expr):
        return where(x > 0.0, 1.0, where(x < 0.0, -1.0, x))   # sign(±0.0) = ±0.0, sign(NaN) = NaN
    return math.copysign(1.0, x) if x != 0 and not math.isnan(x) else x


def ceil(x):
    return -floor(-x) if isinstance(x, Expr) else float(math.ceil(x))


@_reuses_args
def trunc(x):
    if isinstance(x, Expr):
        return where(x < 0.0, -floor(-x), floor(x))
    return float(math.trunc(x))


@_reuses_args
def round_even(x):
    """Julia's `round(x)`: to the nearest integer, ties to even — by the classic (|x| + 2^52) - 2^52, which the
    round-to-nearest-even addition itself performs exactly for |x| < 2^52 (larger values are integers already).
    (An expression is a tree, so every reuse of a sub-expression is a copy: the compositions are kept short — a pass
    holds 96 micro-ops.)"""
    if isinstance(x, Expr):
        # (the min is there for the lowering, which folds x + c1 - c2 into x + (c1 - c2): it must not see one linear chain)
        t = minimum(abs(x) + 4503599627370496.0, math.inf) - 4503599627370496.0
        # the sign goes back on by a product with ±1 (a negation would be folded into the linear chain and lose -0.0):
        # round(-0.3) = -0.0 as Julia's (round(-0.0) gives +0.0)
        return where(abs(x) < 4503599627370496.0, t * where(x < 0.0, -1.0, 1.0), x)
    return float(round(x))   # Python rounds ties to even, too


@_reuses_args
def clamp(x, lo, hi):
    if _is_expr(x, lo, hi):
        x, lo, hi = wrap(x), wrap(lo), wrap(hi)
        return where(x > hi, hi, where(x < lo, lo, x))   # Base.clamp: ifelse(x > hi, hi, ifelse(x < lo, lo, x))
    return hi if x > hi else (lo if x < lo else x)


def log2(x):
    return log(x) / _LN2 if isinstance(x, Expr) else math.log2(x)


def log10(x):
    return log(x) / _LN10 if isinstance(x, Expr) else math.log10(x)


def logb(*a):
    """`log(x)` or `log(b, x)`"""
    if len(a) == 1:
        return log(a[0])
    b, x = a
    return log(x) / log(b)


def exp2(x):
    return exp(x * _LN2) if isinstance(x, Expr) else 2.0 ** x


def exp10(x):
    return exp(x * _LN10) if isinstance(x, Expr) else 10.0 ** x


@_reuses_args
def sinh(x):
    return (expm1(x) - expm1(-x)) * 0.5 if isinstance(x, Expr) else math.sinh(x)


@_reuses_args
def cosh(x):
    return (exp(x) + exp(-x)) * 0.5 if isinstance(x, Expr) else math.cosh(x)


@_reuses_args
def asin(x):
    return atan(x / sqrt((1.0 - x) * (1.0 + x))) if isinstance(x, Expr) else math.asin(x)


@_reuses_args
def acos(x):
    return 2.0 * atan(sqrt((1.0 - x) / (1.0 + x))) if isinstance(x, Expr) else math.acos(x)


@_reuses_args
def atan2(*a):
    """`atan(x)` or the two-argument `atan(y, x)`"""
    if len(a) == 1:
        return atan(a[0])
    y, x = a
    if not _is_expr(y, x):
        return math.atan2(y, x)
    # atan(y / x) moved into the right quadrant.  Kept short (see round_even): exactly-zero arguments follow the unsigned
    # convention (atan(0, 0) = 0, atan(y, ±0.0) = ±π/2 by the sign of y, atan(-0.0, x < 0) = +π) and atan(±Inf, ±Inf) is
    # NaN, where Julia distinguishes signed zeros and returns ±π/4, ±3π/4.
    y, x = wrap(y), wrap(x)
    on_axis = where(y > 0.0, math.pi / 2, where(y < 0.0, -math.pi / 2, y * 0.0))
    return where(x.eq(0.0), on_axis, atan(y / x) + where(x < 0.0, where(y < 0.0, -math.pi, math.pi), 0.0))


@_reuses_args
def hypot(x, y):
    """sqrt(x^2 + y^2) without overflow of the squares: m sqrt(1 + (n / m)^2), m = max(|x|, |y|), n = min(|x|, |y|)
    (hypot(Inf, Inf) and hypot(Inf, NaN) come out NaN; Julia returns Inf)."""
    if not _is_expr(x, y):
        return math.hypot(x, y)
    ax, ay = abs(wrap(x)), abs(wrap(y))
    m = maximum(ax, ay)
    return where(m.eq(0.0), 0.0, m * sqrt(1.0 + abs2(minimum(ax, ay) / m)))


@_reuses_args
def cbrt(x):
    return sign(x) * abs(x) ** (1.0 / 3.0) if isinstance(x, Expr) else math.copysign(abs(x) ** (1.0 / 3.0), x)


def inv(x):
    return 1.0 / x


def fld(x, y):
    return floor(x / y) if _is_expr(x, y) else float(math.floor(x / y))


def cld(x, y):
    return ceil(x / y)


def div(x, y):
    """Julia's `÷` / `div`: the quotient truncated towards zero."""
    return trunc(x / y) if _is_expr(x, y) else (float(math.trunc(x / y)) if isinstance(x, float) or isinstance(y, float)
                                                else int(math.trunc(x / y)))


@_reuses_args
def rem(x, y):
    """Julia's `%` / `rem`: remainder with the sign of the dividend (x - y trunc(x / y); on particle values the
    quotient is formed in floating point, which is exact while |x / y| < 2^53)."""
    if _is_expr(x, y):
        x, y = wrap(x), wrap(y)
        return x - y * trunc(x / y)
    return math.fmod(x, y) if isinstance(x, float) or isinstance(y, float) else int(math.fmod(x, y))


@_reuses_args
def mod(x, y):
    """Julia's `mod`: remainder with the sign of the divisor (x - y floor(x / y))."""
    if _is_expr(x, y):
        x, y = wrap(x), wrap(y)
        return x - y * floor(x / y)
    return x % y   # Python's % is the floored one


def nmin(*a):
    out = a[0]
    for b in a[1:]:
        out = minimum(out, b)
    return out


def nmax(*a):
    out = a[0]
    for b in a[1:]:
        out = maximum(out, b)
    return out


def to_float(x):
    return x if isinstance(x, Expr) else float(x)


def _int_first(fn):
    """`floor(Int, x)` / `round(Int, x)`: the type argument is dropped — every particle value is a Float64 plane"""
    def f(*a):
        if len(a) == 2 and isinstance(a[0], type):
            return fn(a[1])
        if len(a) != 1:
            raise _unsupported(f"{fn.__name__}() with {len(a)} arguments (digits / base keywords are outside the device-op set)")
        return fn(a[0])
    return f


# ------------------------------------------------------------------------------------------------
# lowering to postfix tokens
# ------------------------------------------------------------------------------------------------
class Tokens:
    """A scalar expression as a Python list of (op, col, comp, val)."""

    __slots__ = ("toks",)

    def __init__(self, toks):
        self.toks = toks

    @staticmethod
    def const(v):
        return Tokens([(L.TOK_CONST, 0, 0, float(v))])

    def is_const(self):
        return len(self.toks) == 1 and self.toks[0][0] == L.TOK_CONST

    def const_value(self):
        return self.toks[0][3]


def lower(e, store):
    """Expr -> Tokens (scalar) or list[Tokens] (vector).  ``store`` resolves column names."""
    e = wrap(e)
    if isinstance(e, Const):
        if isinstance(e.v, np.ndarray):
            return [Tokens.const(x) for x in e.v]
        return Tokens.const(e.v)
    if isinstance(e, Col):
        cid, width = store._lookup(e.name)
        if cid < 0:
            raise KeyError(f"particle variable {e.name!r} does not exist yet")
        if width == 1:
            return Tokens([(L.TOK_PLANE, cid, 0, 0.0)])
        return [Tokens([(L.TOK_PLANE, cid, k, 0.0)]) for k in range(width)]
    if isinstance(e, Vec):
        items = [lower(i, store) for i in e.items]
        if any(isinstance(i, list) for i in items):
            raise _unsupported("nested vectors are outside the device-op set")
        return items
    if isinstance(e, Index):
        base = lower(e.base, store)
        if not isinstance(base, list):
            raise _unsupported("indexing a scalar particle variable")
        if not (0 <= e.j < len(base)):
            raise IndexError(f"index {e.j} out of range for a vector of length {len(base)}")
        return base[e.j]
    if isinstance(e, Rand):
        return Tokens([({"n": L.TOK_RANDN, "u": L.TOK_RANDU, "e": L.TOK_RANDEXP}[e.kind], 0, 0, 0.0)])
    if isinstance(e, Param):
        return Tokens([(L.TOK_PARAM, e.index, 0, 0.0)])
    if isinstance(e, RandP):
        a = lower(e.arg, store)
        if isinstance(a, list):
            raise _unsupported("vector-valued distribution parameters are outside the device-op set")
        return Tokens(a.toks + [({"gamma": L.TOK_RANDGAMMA, "poisson": L.TOK_RANDPOISSON}[e.kind], 0, 0, 0.0)])
    if isinstance(e, TableRead):
        r, c = lower(e.row, store), lower(e.col, store)
        if isinstance(r, list) or isinstance(c, list):
            raise _unsupported("table indices must be scalar-valued")
        return Tokens(r.toks + c.toks + [(L.TOK_TABLE, store._table_id(e.table), 0, 0.0)])
    if isinstance(e, CatLogp):
        r, x = lower(e.p.row, store), lower(e.x, store)
        if isinstance(r, list) or isinstance(x, list):
            raise _unsupported("Categorical values and rows must be scalar-valued")
        return Tokens(r.toks + x.toks + [(L.TOK_TABLE, store._table_id(e.p.table), 1, 0.0)])
    if isinstance(e, RandCat):
        r = lower(e.p.row, store)
        if isinstance(r, list):
            raise _unsupported("a Categorical row index must be scalar-valued")
        return Tokens(r.toks + [(L.TOK_RANDCAT, store._table_id(e.p.table), 0, 0.0)])
    if isinstance(e, Select):
        c, a, b = lower(e.cond, store), lower(e.a, store), lower(e.b, store)
        if isinstance(c, list) or isinstance(a, list) or isinstance(b, list):
            raise _unsupported("vector-valued conditionals are outside the device-op set")
        return Tokens(c.toks + a.toks + b.toks + [(L.TOK_SELECT, 0, 0, 0.0)])
    if isinstance(e, Un):
        a = lower(e.a, store)
        if isinstance(a, list):
            if e.op == L.TOK_NEG:
                return [Tokens(t.toks + [(L.TOK_NEG, 0, 0, 0.0)]) for t in a]
            raise _unsupported("elementwise functions of vector-valued variables are outside the device-op set")
        return Tokens(a.toks + [(e.op, 0, 0, 0.0)])
    if isinstance(e, Bin):
        a, b = lower(e.a, store), lower(e.b, store)
        va, vb = isinstance(a, list), isinstance(b, list)
        if not va and not vb:
            return Tokens(a.toks + b.toks + [(e.op, 0, 0, 0.0)])
        if va and vb:
            if e.op not in (L.TOK_ADD, L.TOK_SUB):
                raise _unsupported("only + and - are defined between vector-valued variables")
            if len(a) != len(b):
                raise ValueError(f"vector lengths differ ({len(a)} vs {len(b)})")
            return [Tokens(x.toks + y.toks + [(e.op, 0, 0, 0.0)]) for x, y in zip(a, b)]
        # vector (*|/) scalar, scalar * vector
        if va and e.op in (L.TOK_MUL, L.TOK_DIV):
            return [Tokens(x.toks + b.toks + [(e.op, 0, 0, 0.0)]) for x in a]
        if vb and e.op == L.TOK_MUL:
            return [Tokens(a.toks + y.toks + [(e.op, 0, 0, 0.0)]) for y in b]
        raise _unsupported("this mix of scalar and vector operands is outside the device-op set")
    raise _unsupported(f"cannot lower {type(e).__name__}")


_tok_structs = {}
_expr_structs = {}
_TOK_BYTES = 24   # sizeof(ws_tok): int32 op, col, comp, reserved; double val


def _EXPR_STRUCT(n):
    st = _expr_structs.get(n)
    if st is None:
        st = _expr_structs[n] = struct.Struct("<" + "Qii" * n)   # ws_expr: const ws_tok* toks; int32 n, reserved
    return st


def _TOK_STRUCT(n):
    st = _tok_structs.get(n)
    if st is None:
        st = _tok_structs[n] = struct.Struct("<" + "iiiid" * n)
    return st


class CExprs:
    """Owns the ctypes arrays behind one or more ``ws_expr`` (keeps them alive for the call)."""

    def __init__(self, token_lists):
        # One packed token buffer for all expressions of the statement and one packed ws_expr array pointing into it:
        # two struct copies instead of four ctypes attribute stores per token and a cast per expression (the host
        # walker lowers every statement of every loop iteration: this is on the per-step path).
        flat, counts = [], []
        for t in token_lists:
            for op, c, comp, val in t.toks:
                flat += (op, c, comp, 0, val)
            counts.append(len(t.toks))
        n_tok = sum(counts)
        self._toks = (L.ws_tok * max(1, n_tok)).from_buffer_copy(_TOK_STRUCT(n_tok).pack(*flat) if n_tok else b"\0" * _TOK_BYTES)
        base = C.addressof(self._toks)
        head, off = [], 0
        for k in counts:
            head += (base + off * _TOK_BYTES, k, 0)
            off += k
        self.arr = (L.ws_expr * len(counts)).from_buffer_copy(_EXPR_STRUCT(len(counts)).pack(*head))

    def ptr(self, i=0):
        p = C.cast(C.byref(self.arr, i * C.sizeof(L.ws_expr)), C.POINTER(L.ws_expr))
        p._owner = self      # whoever keeps the pointer (a recorded loop body) keeps the token buffers alive
        return p

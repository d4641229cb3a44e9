"""``@model`` front-end: the reference's probabilistic-program DSL (``src/rewrites.jl``) accepted as
Julia SOURCE TEXT and lowered to the transformer tree of :mod:`core` (whose ``apply`` bodies are the
device ops).  ``model(src)`` plays the role of macro expansion: the statement forms, the particle-
variable bookkeeping and the error cases follow ``walk_body`` / ``gen_step`` / ``vectorize``
(rewrites.jl:146-219, 500-558, 643-752); anything outside the fixed device-op set raises
:class:`UnsupportedModelError` here, before any particle exists.

    ssm = model('''
    @model function ssm(obs)
        x{1} .= 0.0
        v .= 0.0
        for (t, o) in enumerate(obs)
            x{t + 1} .= x{t} + v
            dv ~ Normal(0.0, 0.1)
            v .= v + dv
            o => Normal(x{t + 1}, 1.0)
        end
    end
    ''')
    run(ssm(obs), SMCState(1000))

Supported statements (rewrites.jl:7-36): ``x .= e``, ``x ~ f(a...)``, ``_ ~ f(a...)``, ``e => f(a...)``,
``x << q(a...; diversity=d)``, ``(x, y) << q(...)``, build-time ``=`` / ``+=`` ..., ``for``, ``if`` (no
else; ``resampled`` allowed), ``Resample()``; dynamic families ``x{e}`` (column ``x_e``), accessors
``x[e]`` on vector-valued columns.  A ``Resample()`` is auto-inserted after every ``~`` and ``=>``
(rewrites.jl:707-711).  The signature is a Julia signature (rewrites.jl:776-806): ``function f(a, b::T=default;
kw=default, required_kw)`` — annotations are skipped, defaults are build-time expressions evaluated left to right —
and loop variables destructure as nested tuples (``for (i, (x, y)) in enumerate(data)``, rewrites.jl:652-664).
Build-time statements (rewrites.jl:717-733) include tuple assignment (``a, b = 1.0, 2.0``), local functions
(``g(u) = 2u + 1``) and anonymous functions (``h = (u, v) -> u * v``), which trace into the device expression when
called on particle variables; ``a[end]``, ``√x``, and Julia's truncated ``÷`` / ``%``.  Scalar Base functions without a
micro-op of their own (``sign clamp ceil trunc round isnan isinf isfinite log2 log10 log(b, x) exp2 exp10 sinh cosh
asin acos atan(y, x) hypot cbrt inv fld cld div rem mod``, n-ary ``min`` / ``max``, ``floor(Int, x)``) are compositions
of the micro-ops (``expr.py``; their conventions at signed zeros / infinities are stated there).
"""
from __future__ import annotations

import math
import re

import numpy as np

from . import _lib as L
from . import core, expr
from ._lib import UnsupportedModelError
from .expr import Col, Expr, Index, Vec


class ModelSyntaxError(ValueError):
    """The reference raises ``error(...)`` at macro expansion for these."""


def _unsupported(msg):
    return UnsupportedModelError(L.WS_EUNSUPPORTED, msg)


# ---------------------------------------------------------------------------------------------
# tokenizer
# ---------------------------------------------------------------------------------------------
_TOKEN_RE = re.compile(r"""
    (?P<ws>[ \t\r]+)
  | (?P<comment>\#=.*?=\#|\#[^\n]*)
  | (?P<nl>\n)
  | (?P<num>(?:\d[\d_]*\.?\d*(?:[eE][+-]?\d+)?|\.\d+(?:[eE][+-]?\d+)?))
  | (?P<name>@?[^\W\d][\w!′]*)
  | (?P<op>\.\+=|\.-=|\.\*=|\./=|\.=|=>|<<|==|!=|<=|>=|&&|\|\||\+=|-=|\*=|/=|\.\+|\.-|\.\*|\./|\.\^|->|[-+*/^%÷√=<>!~:,;()\[\]{}.'?&|])
""", re.X | re.S)


def tokenize(src):
    toks, pos = [], 0
    while pos < len(src):
        m = _TOKEN_RE.match(src, pos)
        if not m:
            raise ModelSyntaxError(f"cannot tokenize at: {src[pos:pos + 20]!r}")
        pos = m.end()
        k = m.lastgroup
        if k in ("ws", "comment"):
            continue
        toks.append((k, m.group(k)))
    toks.append(("eof", ""))
    return toks


# ---------------------------------------------------------------------------------------------
# parser -> AST (tuples)
# ---------------------------------------------------------------------------------------------
_STMT_OPS = {".=", "~", "=>", "<<", "=", "+=", "-=", "*=", "/=", ".+=", ".-=", ".*=", "./="}


class Parser:
    def __init__(self, toks):
        self.t, self.i = toks, 0
        self.depth = 0  # bracket depth: newlines are ignored inside brackets
        self.no_range = 0  # > 0 while parsing the middle operand of a ternary (`:` belongs to the ternary)
        self.in_index = 0  # > 0 inside `a[...]`: `end` is the last index there, not a block terminator

    def peek(self, skip_nl=False):
        j = self.i
        while (skip_nl or self.depth > 0) and self.t[j][0] == "nl":
            j += 1
        return self.t[j]

    def next(self, skip_nl=False):
        while (skip_nl or self.depth > 0) and self.t[self.i][0] == "nl":
            self.i += 1
        tok = self.t[self.i]
        self.i += 1
        return tok

    def accept(self, kind, val=None, skip_nl=False):
        k, v = self.peek(skip_nl)
        if k == kind and (val is None or v == val):
            return self.next(skip_nl)
        return None

    def expect(self, kind, val=None, skip_nl=False):
        tok = self.accept(kind, val, skip_nl)
        if tok is None:
            raise ModelSyntaxError(f"expected {val or kind}, got {self.peek(skip_nl)[1]!r}")
        return tok

    def skip_newlines(self):
        while self.t[self.i][0] == "nl" or self.t[self.i] == ("op", ";"):
            self.i += 1

    # ---- top level ----------------------------------------------------------------------------
    def parse_model(self):
        self.skip_newlines()
        if self.accept("name", "@model"):
            pass
        self.expect("name", "function", skip_nl=True)
        name = self.expect("name")[1]
        self.expect("op", "(")
        self.depth += 1
        # `function name(args...; kwargs...)` (rewrites.jl:776-787 splices both lists into the generated function
        # verbatim): positional and keyword parameters, each with an optional type annotation and default value
        params, defaults, kwonly = [], {}, set()
        after_semicolon = False
        while not self.accept("op", ")"):
            if self.accept("op", ";"):
                after_semicolon = True
                continue
            pname = self.expect("name")[1]
            params.append(pname)
            if after_semicolon:
                kwonly.add(pname)
            if self.peek() == ("op", ":") and self.t[self.i + 1] == ("op", ":"):
                # `T::Int`, `data::Vector{Float64}`, `m::Base.Matrix`: a Julia type annotation on a model argument
                # (test/macro_test.jl:12) restricts dispatch and nothing else — skipped
                self.next()
                self.next()
                self.expect("name")
                while self.accept("op", "."):
                    self.expect("name")
                if self.accept("op", "{"):
                    nest = 1
                    while nest > 0:
                        k, v = self.next()
                        if k == "eof":
                            raise ModelSyntaxError("unterminated type parameters in the model signature")
                        nest += (k, v) == ("op", "{")
                        nest -= (k, v) == ("op", "}")
            if self.accept("op", "="):
                defaults[pname] = self.parse_expr()
            self.accept("op", ",")
        self.signature = (defaults, kwonly)
        self.depth -= 1
        body = self.parse_block()
        self.expect("name", "end")
        self.skip_newlines()
        if self.peek()[0] != "eof":
            raise ModelSyntaxError(f"unexpected text after the model function: {self.peek()[1]!r}")
        return name, params, body

    def parse_block(self):
        stmts = []
        while True:
            self.skip_newlines()
            k, v = self.peek()
            if k == "eof" or (k == "name" and v in ("end", "else", "elseif")):
                return stmts
            stmts.append(self.parse_stmt())

    def parse_stmt(self):
        k, v = self.peek()
        if k == "name" and v == "for":
            self.next()
            pat = self.parse_pattern()
            if not (self.accept("name", "in") or self.accept("op", "=") or self.accept("name", "∈")):
                raise ModelSyntaxError("expected `in` in for loop")
            it = self.parse_expr()
            body = self.parse_block()
            self.expect("name", "end")
            return ("for", pat, it, body)
        if k == "name" and v == "if":
            self.next()
            cond = self.parse_expr()
            body = self.parse_block()
            if self.peek()[1] in ("else", "elseif"):
                raise ModelSyntaxError("`if` with an else branch is not supported by @model (rewrites.jl:671-682)")
            self.expect("name", "end")
            return ("if", cond, body)
        lhs = self.parse_expr()
        if self.peek() == ("op", ","):
            # `a, b = 1.0, 2.0`: a tuple on either side of a plain `=` may be written without parentheses
            items = [lhs]
            while self.accept("op", ","):
                items.append(self.parse_expr())
            lhs = ("tuple", items)
            if self.peek() != ("op", "="):
                raise ModelSyntaxError("unexpected token ','")
        k, v = self.peek()
        if k == "op" and v in _STMT_OPS:
            self.next()
            rhs = self.parse_expr()
            if v == "=" and self.peek() == ("op", ","):
                items = [rhs]
                while self.accept("op", ","):
                    items.append(self.parse_expr())
                rhs = ("tuple", items)
            if v == "=" and lhs[0] == "call" and lhs[1][0] == "name" and not lhs[3] and all(a[0] == "name" for a in lhs[2]):
                # `g(u, v) = body`: a local function (a build-time `=` like any other, rewrites.jl:717-733)
                return ("stmt", "=", lhs[1], ("lambda", [a[1] for a in lhs[2]], rhs))
            return ("stmt", v, lhs, rhs)
        return ("expr", lhs)

    def parse_pattern(self):
        # `x`, `(x, y)`, `(i, (x, y))`: the loop variable becomes the single destructuring argument of the body
        # closure (rewrites.jl:652-664), so patterns nest as Julia's do
        if self.accept("op", "("):
            self.depth += 1
            names = []
            while not self.accept("op", ")"):
                names.append(self.parse_pattern())
                self.accept("op", ",")
            self.depth -= 1
            return names
        return self.expect("name")[1]

    # ---- expressions (precedence climbing) ------------------------------------------------------
    def parse_expr(self):
        c = self.parse_or()
        if self.peek() == ("op", "->"):
            # `u -> body`, `(u, v) -> body`
            params = [c] if c[0] == "name" else (c[1] if c[0] == "tuple" else None)
            if params is None or not all(a[0] == "name" for a in params):
                raise ModelSyntaxError("the parameters of an anonymous function must be names")
            self.next()
            return ("lambda", [a[1] for a in params], self.parse_expr())
        if self.peek() == ("op", "?"):
            # ternary `cond ? a : b` (vectorised to ifelse.(cond, a, b) when cond is per-particle, rewrites.jl:193-199)
            self.next()
            self.no_range += 1
            a = self.parse_expr()
            self.no_range -= 1
            self.expect("op", ":")
            b = self.parse_expr()
            return ("if", c, a, b)
        return c

    def parse_or(self):
        a = self.parse_and()
        while self.accept("op", "||"):
            a = ("bin", "||", a, self.parse_and())
        return a

    def parse_and(self):
        a = self.parse_cmp()
        while self.accept("op", "&&"):
            a = ("bin", "&&", a, self.parse_cmp())
        return a

    def parse_cmp(self):
        a = self.parse_range()
        while self.peek() in (("op", "=="), ("op", "!="), ("op", "<"), ("op", ">"), ("op", "<="), ("op", ">=")):
            op = self.next()[1]
            a = ("bin", op, a, self.parse_range())
        return a

    def parse_range(self):
        a = self.parse_add()
        if self.peek() == ("op", ":") and self.no_range == 0:
            self.next()
            b = self.parse_add()
            if self.peek() == ("op", ":"):
                self.next()
                c = self.parse_add()
                return ("range", a, c, b)
            return ("range", a, b, None)
        return a

    def parse_add(self):
        a = self.parse_mul()
        while self.peek() in (("op", "+"), ("op", "-"), ("op", ".+"), ("op", ".-"), ("op", "|")):
            op = self.next()[1].lstrip(".")
            a = ("bin", "||" if op == "|" else op, a, self.parse_mul())
        return a

    def parse_mul(self):
        a = self.parse_unary()
        while self.peek() in (("op", "*"), ("op", "/"), ("op", "%"), ("op", "÷"), ("op", ".*"), ("op", "./"), ("op", "&")):
            op = self.next()[1].lstrip(".")
            a = ("bin", "&&" if op == "&" else op, a, self.parse_unary())
        return a

    def parse_unary(self):
        if self.accept("op", "-"):
            return ("un", "-", self.parse_unary())
        if self.accept("op", "+"):
            return self.parse_unary()
        if self.accept("op", "!"):
            return ("un", "!", self.parse_unary())
        if self.accept("op", "√"):
            return ("call", ("name", "sqrt"), [self.parse_unary()], {})
        return self.parse_pow()

    def parse_pow(self):
        a = self.parse_postfix()
        if self.peek() in (("op", "^"), ("op", ".^")):
            self.next()
            return ("bin", "^", a, self.parse_unary())  # right associative, binds tighter than unary minus on its left
        return a

    def parse_args(self, close):
        """comma separated expressions with optional `; kw=val` / `kw=val` keyword arguments"""
        args, kwargs = [], {}
        self.depth += 1
        in_kw = False
        while True:
            if self.accept("op", close):
                break
            if self.accept("op", ";"):
                in_kw = True
                continue
            if self.accept("op", ","):
                continue
            k, v = self.peek()
            k2 = self.t[self._index_after_peek()]
            if k == "name" and k2 == ("op", "="):
                self.next()
                self.next()
                kwargs[v] = self.parse_expr()
                continue
            if in_kw:
                raise ModelSyntaxError("expected keyword argument after `;`")
            args.append(self.parse_expr())
        self.depth -= 1
        return args, kwargs

    def _index_after_peek(self):
        j = self.i
        while self.t[j][0] == "nl":
            j += 1
        j += 1
        while self.t[j][0] == "nl":
            j += 1
        return j

    def parse_postfix(self):
        a = self.parse_atom()
        while True:
            k, v = self.t[self.i]  # no newline skipping: a call paren must follow directly
            if (k, v) == ("op", "("):
                self.next()
                args, kwargs = self.parse_args(")")
                a = ("call", a, args, kwargs)
            elif (k, v) == ("op", "["):
                self.next()
                self.in_index += 1
                args, _ = self.parse_args("]")
                self.in_index -= 1
                if len(args) == 2:
                    a = ("index2", a, args[0], args[1])   # `P[s, k]` / `P[s, :]`: a row or entry of a build-time matrix
                elif len(args) != 1:
                    raise ModelSyntaxError("only `x[e]` and `P[i, j]` indices are supported (rewrites.jl:170-171)")
                else:
                    a = ("index", a, args[0])
            elif (k, v) == ("op", "{"):
                self.next()
                args, _ = self.parse_args("}")
                if len(args) != 1 or a[0] != "name":
                    raise ModelSyntaxError("unsupported dynamic-variable expression (expected `x{e}`)")
                a = ("curly", a[1], args[0])
            elif (k, v) == ("op", "."):
                self.next()
                fld = self.expect("name")[1]
                a = ("field", a, fld)
            elif (k, v) == ("op", "'"):
                self.next()
                a = ("call", ("name", "transpose"), [a], {})
            else:
                return a

    def parse_atom(self):
        k, v = self.next()
        if k == "num":
            txt = v.replace("_", "")
            is_int = re.fullmatch(r"\d+", txt) is not None
            node = ("num", int(txt) if is_int else float(txt))
            # numeric-literal coefficient: 2x, 2(x + 1)
            k2, v2 = self.t[self.i]
            if k2 == "name" and v2 not in ("in", "end", "for", "if", "else", "elseif"):
                return ("bin", "*", node, self.parse_postfix())
            if (k2, v2) == ("op", "("):
                return ("bin", "*", node, self.parse_atom_paren())
            return node
        if k == "name":
            if v == "end" and self.in_index > 0:
                return ("name", "__end__")   # `a[end]`: bound to the length of `a` when the index is evaluated
            return ("name", v)
        if (k, v) == ("op", "("):
            self.i -= 1
            return self.parse_atom_paren()
        if (k, v) == ("op", "["):
            return self.parse_bracket()
        if (k, v) == ("op", ":") and self.in_index > 0 and self.t[self.i] in (("op", ","), ("op", "]")):
            return ("colon",)   # `P[s, :]`: the whole row
        if (k, v) == ("op", ":"):
            # symbol literal :x
            nm = self.expect("name")[1]
            return ("sym", nm)
        raise ModelSyntaxError(f"unexpected token {v!r}")

    def parse_atom_paren(self):
        self.expect("op", "(")
        self.depth += 1
        items = []
        trailing_comma = False
        while not self.accept("op", ")"):
            items.append(self.parse_expr())
            trailing_comma = self.accept("op", ",") is not None
        self.depth -= 1
        if len(items) == 1 and not trailing_comma:
            return items[0]
        return ("tuple", items)

    def parse_bracket(self):
        """[a, b, c] vector  |  [a b; c d] matrix  (newlines inside act like `;`)"""
        rows, row = [], []
        is_matrix = False
        saved_depth = self.depth
        self.depth = 0  # newlines are significant inside a matrix literal
        while True:
            k, v = self.t[self.i]
            if k == "nl":
                self.i += 1
                if row and is_matrix:
                    rows.append(row)
                    row = []
                continue
            if (k, v) == ("op", "]"):
                self.i += 1
                break
            if (k, v) == ("op", ","):
                self.i += 1
                continue
            if (k, v) == ("op", ";"):
                self.i += 1
                is_matrix = True
                rows.append(row)
                row = []
                continue
            before = self.i
            row.append(self.parse_expr())
            # space separated entries => matrix row
            k2, v2 = self.t[self.i]
            if (k2, v2) not in (("op", ","), ("op", "]"), ("op", ";")) and k2 != "nl" and self.i > before:
                is_matrix = True
        self.depth = saved_depth
        if is_matrix:
            if row:
                rows.append(row)
            return ("matrix", rows)
        return ("vect", row)


# ---------------------------------------------------------------------------------------------
# static checks ("macro expansion"): particle-variable bookkeeping and error cases
# ---------------------------------------------------------------------------------------------
def _names_in(ast):
    """(plain names, curly bases) referenced anywhere in an AST"""
    names, curlies = set(), set()

    def rec(a):
        if not isinstance(a, tuple):
            if isinstance(a, list):
                for x in a:
                    rec(x)
            elif isinstance(a, dict):
                for x in a.values():
                    rec(x)
            return
        if a[0] == "name":
            names.add(a[1])
        elif a[0] == "curly":
            curlies.add(a[1])
            rec(a[2])
        else:
            for x in a[1:]:
                rec(x)
    rec(ast)
    return names, curlies


def _contains_particle(ast, pv):
    names, curlies = _names_in(ast)
    return bool(curlies) or bool(names & pv)


def _root_of(lhs):
    """(kind, base) with kind in plain / curly / accessor"""
    if lhs[0] == "name":
        return "plain", lhs[1]
    if lhs[0] == "curly":
        return "curly", lhs[1]
    if lhs[0] in ("index", "field"):
        k, b = _root_of(lhs[1])
        return "accessor", b
    raise ModelSyntaxError(f"unsupported assignment target")


def _check_expr(ast, pv, fam, stmt):
    """walk an expression that may contain particle variables (the `vectorize` error cases)"""
    if not isinstance(ast, tuple):
        return
    tag = ast[0]
    if tag == "curly":
        if _contains_particle(ast[2], pv):
            raise ModelSyntaxError(f"Dynamic-variable index in `{ast[1]}{{...}}` must not depend on a particle variable "
                                   "(a column name cannot vary per particle)")
        if ast[1] not in fam:
            raise ModelSyntaxError(f"`{ast[1]}` is not a registered dynamic-variable family; assign `{ast[1]}{{...}} .= ...` "
                                   "(or `~`) first")
        return
    if tag == "field" and _contains_particle(ast[1], pv):
        raise _unsupported("struct-valued particle columns (`x.p`) are outside the device-op set")
    if tag == "tuple" and _contains_particle(ast, pv):
        raise ModelSyntaxError("Unsupported expression containing a particle variable (tuple)")
    if tag in ("index", "index2") and any(_contains_particle(i, pv) for i in ast[2:]):
        # a build-time array indexed by a particle value is a table (expr.Table); a particle variable is not
        if _contains_particle(ast[1], pv):
            raise _unsupported("particle-dependent indices into a particle variable are outside the device-op set")
    for x in ast[1:]:
        if isinstance(x, tuple):
            _check_expr(x, pv, fam, stmt)
        elif isinstance(x, list):
            for y in x:
                if isinstance(y, list):
                    for z in y:
                        _check_expr(z, pv, fam, stmt)
                else:
                    _check_expr(y, pv, fam, stmt)
        elif isinstance(x, dict):
            for y in x.values():
                _check_expr(y, pv, fam, stmt)


def _pattern_names(pat):
    if isinstance(pat, list):
        return [n for p in pat for n in _pattern_names(p)]
    return [pat]


def _destructure(pat, x, out):
    """bind the loop element `x` to the (possibly nested) pattern, as Julia's tuple destructuring does"""
    if isinstance(pat, list):
        xs = tuple(x)
        if len(xs) < len(pat):
            raise ValueError(f"cannot destructure {len(xs)} value(s) into {len(pat)} loop variables")
        for p, v in zip(pat, xs):
            _destructure(p, v, out)
    else:
        out[pat] = x
    return out


def _static_check(stmts, pv, fam, locals_):
    for s in stmts:
        if s[0] == "for":
            _, pat, it, body = s
            if _contains_particle(it, pv):
                raise ModelSyntaxError("a `for` collection must not depend on a particle variable")
            loc = set(locals_) | set(_pattern_names(pat))
            _static_check(body, pv, fam, loc)
        elif s[0] == "if":
            _, cond, body = s
            names, curl = _names_in(cond)
            if curl or (names - {"resampled"}) & pv:
                raise ModelSyntaxError("an `if` condition must not reference a particle variable "
                                       "(it may reference `resampled`)")
            _static_check(body, pv, fam, locals_)
        elif s[0] == "expr":
            e = s[1]
            if e[0] == "call" and e[1] == ("name", "Resample") and not e[2]:
                continue
            raise ModelSyntaxError("unsupported statement (expected .=, ~, =>, <<, =, for, if or Resample())")
        else:
            _, op, lhs, rhs = s
            if op in (".+=", ".-=", ".*=", "./="):
                raise ModelSyntaxError(f"Dotted compound assignment `{op}` is not supported; write `x .= x {op[1]} ...`")
            if op in ("=", "+=", "-=", "*=", "/="):
                targets = [lhs]
                if lhs[0] == "tuple" and op == "=":
                    targets = lhs[1]                    # `(a, b) = ...` / `a, b = ...`: build-time destructuring
                for t in targets:
                    if t[0] != "name":
                        raise ModelSyntaxError("a plain `=` target must be a local variable name")
                    if t[1] in pv or t[1] in fam:
                        raise ModelSyntaxError(f"`{t[1]}` is a particle variable; use `.=` instead of `{op}`")
                if _contains_particle(rhs, pv):
                    raise ModelSyntaxError("the right-hand side of a plain `=` runs once at build time and cannot read a "
                                           "particle variable; use `.=` / `~`")
                locals_ = set(locals_) | {t[1] for t in targets}
                continue
            if op == "<<":
                targets = lhs[1] if lhs[0] == "tuple" else [lhs]
                for t in targets:
                    kind, base = _root_of(t)
                    if kind == "accessor":
                        raise ModelSyntaxError("a move target must be a whole particle variable (or dynamic family member), "
                                               "not a value-level accessor `x[e]` / `x.p`")
                    if kind == "plain" and base not in pv:
                        raise ModelSyntaxError(f"move target `{base}` is not a particle variable")
                    if kind == "curly":
                        _check_expr(t, pv, fam, s)
                if rhs[0] != "call" or rhs[1][0] != "name":
                    raise ModelSyntaxError("`<<` expects a proposal call, e.g. `x << RW(0.1)`")
                for a in rhs[2]:
                    if _contains_particle(a, pv):
                        raise ModelSyntaxError("proposal arguments must not depend on particle variables")
                continue
            # .=, ~, =>
            if rhs[0] == "call" and op in ("~", "=>"):
                if rhs[1][0] != "name":
                    raise ModelSyntaxError("kernel must be named")
                kname = rhs[1][1]
                if kname in core._REFERENCE_ONLY_KERNELS:
                    raise _unsupported(f"kernel {kname} is in the reference's default_kernels but outside the device-op "
                                       "set (Normal, MvNormal, Exponential)")
                for a in rhs[2]:
                    _check_expr(a, pv, fam, s)
            elif op in ("~", "=>"):
                raise ModelSyntaxError(f"`{op}` expects a kernel call on its right-hand side")
            else:
                _check_expr(rhs, pv, fam, s)
            if op == "=>":
                _check_expr(lhs, pv, fam, s)
                continue
            if op == "~" and lhs == ("name", "_"):
                continue
            kind, base = _root_of(lhs)
            if kind == "plain":
                if base in fam:
                    raise ModelSyntaxError(f"`{base}` is a dynamic-variable family; it cannot also be a plain particle variable")
                if base in locals_:
                    raise ModelSyntaxError(f"`{base}` is a build-time local; it cannot also be a particle variable")
                pv.add(base)
            elif kind == "curly":
                if _contains_particle(lhs[2], pv):
                    raise ModelSyntaxError(f"Dynamic-variable index in `{base}{{...}}` must not depend on a particle variable")
                if base in pv:
                    raise ModelSyntaxError(f"`{base}` is already a plain particle variable; it cannot also be used as a "
                                           f"dynamic-variable family `{base}{{...}}`")
                fam.add(base)
            else:
                if lhs[0] == "field":
                    raise _unsupported("struct-valued particle columns (`x.p`) are outside the device-op set")
                if base not in pv and base not in fam:
                    raise ModelSyntaxError(f"accessor write into `{base}`, which is not a particle variable yet")
                _check_expr(lhs[1], pv, fam, s)
                if _contains_particle(lhs[2], pv):
                    raise _unsupported("particle-dependent indices are outside the device-op set")


# ---------------------------------------------------------------------------------------------
# evaluation of build-time expressions / construction of particle expressions
# ---------------------------------------------------------------------------------------------
def dynname(base, idx):
    """rewrites.jl:93: x{7} -> :x_7"""
    if isinstance(idx, float) and idx.is_integer():
        idx = int(idx)
    return f"{base}_{idx}"


class _Range:
    def __init__(self, a, b, step=1):
        self.a, self.b, self.step = a, b, step

    def __iter__(self):
        if all(isinstance(v, (int, np.integer)) for v in (self.a, self.b, self.step)):
            return iter(range(self.a, self.b + (1 if self.step > 0 else -1), self.step))
        return iter(np.arange(self.a, self.b + self.step / 2, self.step).tolist())

    def __len__(self):
        return len(list(iter(self)))


def _enumerate1(xs):
    return [(i + 1, x) for i, x in enumerate(xs)]


def _jl_zeros(*dims):
    return np.zeros(tuple(int(d) for d in dims))


def _jl_ones(*dims):
    return np.ones(tuple(int(d) for d in dims))


_BUILTINS = {
    "sqrt": expr.sqrt, "exp": expr.exp, "log": expr.log, "sin": expr.sin, "cos": expr.cos, "abs2": expr.abs2,
    "tan": expr.tan, "atan": expr.atan, "tanh": expr.tanh, "log1p": expr.log1p, "expm1": expr.expm1, "lgamma": expr.lgamma,
    "loggamma": expr.lgamma, "floor": expr.floor, "min": expr.minimum, "max": expr.maximum, "ifelse": expr.where,
    "abs": lambda x: abs(x), "zeros": _jl_zeros, "ones": _jl_ones, "length": len, "enumerate": _enumerate1,
    "zip": lambda *a: list(zip(*a)), "collect": list, "sum": lambda x: float(np.sum(x)), "Inf": math.inf,
    "NaN": math.nan, "pi": math.pi, "π": math.pi, "true": True, "false": False, "nothing": None,
    "Float64": float, "Int": int, "float": float, "fill": lambda v, n: np.full(int(n), v),
    "transpose": lambda m: np.asarray(m).T, "size": lambda a, d=None: np.shape(a) if d is None else np.shape(a)[d - 1],
    "minimum": lambda x: float(np.min(x)), "maximum": lambda x: float(np.max(x)), "mean": lambda x: float(np.mean(x)),
    "Diagonal": lambda v: np.diag(np.asarray(v, dtype=float)), "diagm": lambda v: np.diag(np.asarray(v, dtype=float)),
    "eachindex": lambda x: _Range(1, len(x)), "first": lambda x: x[0], "last": lambda x: x[-1],
    # scalar Base functions without a micro-op of their own: compositions (expr.py), Julia's results on particle values
    "sign": expr.sign, "clamp": expr.clamp, "ceil": expr._int_first(expr.ceil), "trunc": expr._int_first(expr.trunc),
    "round": expr._int_first(expr.round_even), "isnan": expr.isnan, "isinf": expr.isinf, "isfinite": expr.isfinite,
    "log2": expr.log2, "log10": expr.log10, "exp2": expr.exp2, "exp10": expr.exp10, "sinh": expr.sinh, "cosh": expr.cosh,
    "asin": expr.asin, "acos": expr.acos, "hypot": expr.hypot, "cbrt": expr.cbrt, "inv": expr.inv, "fld": expr.fld,
    "cld": expr.cld, "div": expr.div, "rem": expr.rem, "mod": expr.mod, "one": lambda x: 1.0, "zero": lambda x: 0.0,
    "iszero": lambda x: x.eq(0.0) if isinstance(x, Expr) else x == 0, "isone": lambda x: x.eq(1.0) if isinstance(x, Expr) else x == 1,
    "prod": lambda x: float(np.prod(x)), "abs": lambda x: abs(x), "reverse": lambda x: x[::-1], "range": lambda a, b=None, length=None, step=None, stop=None: _jl_range(a, b, length, step, stop),
}
_BUILTINS.update({"floor": expr._int_first(expr.floor), "atan": expr.atan2, "log": expr.logb, "min": expr.nmin, "max": expr.nmax,
                  "Float64": expr.to_float, "float": expr.to_float})


def _jl_range(start, stop=None, length=None, step=None, stop_kw=None):
    """`range(a, b; length=n)` / `range(a, b; step=s)` / `range(a; stop=b, length=n)` as a list of floats"""
    if stop is None:
        stop = stop_kw
    if length is not None:
        return [float(v) for v in np.linspace(float(start), float(stop), int(length))]
    step = 1 if step is None else step
    n = int(math.floor((stop - start) / step + 1e-12)) + 1
    return [start + k * step for k in range(max(0, n))]


class _Env:
    def __init__(self, values, particle_vars, families, parent=None):
        self.values, self.pv, self.fam, self.parent = values, particle_vars, families, parent

    def lookup(self, name):
        e = self
        while e is not None:
            if name in e.values:
                return e.values[name]
            e = e.parent
        if name in self.pv:
            return Col(name)
        if name in _BUILTINS:
            return _BUILTINS[name]
        raise ModelSyntaxError(f"undefined name `{name}` in model body")

    def child(self, values):
        return _Env(dict(values), self.pv, self.fam, self)

    def snapshot(self):
        """the bindings visible now, frozen: later rebinding of a build-time local does not reach a body built lazily"""
        chain, e = [], self
        while e is not None:
            chain.append(e.values)
            e = e.parent
        merged = {}
        for d in reversed(chain):
            merged.update(d)
        return _Env(merged, self.pv, self.fam, None)

    def set_local(self, name, v):
        # Julia closure scoping: assigning a name that exists in an enclosing scope rebinds it there
        e = self
        while e is not None:
            if name in e.values:
                e.values[name] = v
                return
            e = e.parent
        self.values[name] = v


def _binop(op, a, b):
    if op == "+": return a + b
    if op == "-": return a - b
    if op == "*":
        if isinstance(a, np.ndarray) and isinstance(b, np.ndarray) and a.ndim == 2:
            return a @ b
        return a * b
    if op == "/": return a / b
    if op == "^": return a ** b
    if op == "%": return expr.rem(a, b)    # Julia: remainder with the sign of the dividend
    if op == "÷": return expr.div(a, b)    # Julia: quotient truncated towards zero
    if op == "==": return a.eq(b) if isinstance(a, Expr) else (b.eq(a) if isinstance(b, Expr) else a == b)
    if op == "!=": return ~(a.eq(b)) if isinstance(a, Expr) else (~(b.eq(a)) if isinstance(b, Expr) else a != b)
    if op == "<": return a < b
    if op == ">": return a > b
    if op == "<=": return a <= b
    if op == ">=": return a >= b
    if op == "&&": return (a & b) if (isinstance(a, Expr) or isinstance(b, Expr)) else (bool(a) and bool(b))
    if op == "||": return (a | b) if (isinstance(a, Expr) or isinstance(b, Expr)) else (bool(a) or bool(b))
    raise ModelSyntaxError(f"unsupported operator {op}")


_COLON = object()   # a bare `:` index


def ev(ast, env):
    tag = ast[0]
    if tag == "num":
        return ast[1]
    if tag == "name":
        return env.lookup(ast[1])
    if tag == "sym":
        return ast[1]
    if tag == "bin":
        return _binop(ast[1], ev(ast[2], env), ev(ast[3], env))
    if tag == "un":
        v = ev(ast[2], env)
        if ast[1] == "!":
            return ~v if isinstance(v, Expr) else (not v)
        return -v
    if tag == "if":
        return expr.where(ev(ast[1], env), ev(ast[2], env), ev(ast[3], env))
    if tag == "range":
        a, b = ev(ast[1], env), ev(ast[2], env)
        step = 1 if ast[3] is None else ev(ast[3], env)
        return _Range(a, b, step)
    if tag == "vect":
        items = [ev(x, env) for x in ast[1]]
        if any(isinstance(i, Expr) for i in items):
            return Vec(items)
        return np.asarray(items, dtype=np.float64) if all(isinstance(i, (int, float)) for i in items) else items
    if tag == "matrix":
        return np.asarray([[float(ev(x, env)) for x in row] for row in ast[1]], dtype=np.float64)
    if tag == "tuple":
        return tuple(ev(x, env) for x in ast[1])
    if tag == "curly":
        idx = ev(ast[2], env)
        return Col(dynname(ast[1], idx))
    if tag == "lambda":
        params, body, defenv = ast[1], ast[2], env

        def fn(*a):
            if len(a) != len(params):
                raise TypeError(f"function takes {len(params)} argument(s) but {len(a)} were given")
            return ev(body, defenv.child(dict(zip(params, a))))   # (the defining scope stays live, as a Julia closure's does)
        return fn
    if tag == "index":
        base = ev(ast[1], env)
        ienv = env
        if "__end__" in _names_in(ast[2])[0]:
            if isinstance(base, Expr):
                if not isinstance(base, Vec):
                    raise _unsupported("`end` in the index of a particle variable (its length is not known when the model is built)")
                ienv = env.child({"__end__": len(base.items)})
            else:
                ienv = env.child({"__end__": len(base)})
        idx = ev(ast[2], ienv)
        if isinstance(base, Expr):
            return Index(base, int(idx) - 1)  # Julia is 1-based
        if isinstance(idx, Expr) or isinstance(base, expr.Table):
            return expr.table(base)[idx]      # `mu[s]`: a build-time vector indexed by a particle value
        if isinstance(idx, _Range):
            return np.asarray(base)[[int(i) - 1 for i in idx]]
        return base[int(idx) - 1]
    if tag == "index2":
        base, i, j = ev(ast[1], env), ev(ast[2], env), ev(ast[3], env)
        if isinstance(base, Expr):
            raise _unsupported("two indices into a particle variable are outside the device-op set")
        if isinstance(i, Expr) or isinstance(j, Expr):
            return expr.table(base)[i, slice(None) if j is _COLON else j]
        a = base.values if isinstance(base, expr.Table) else np.asarray(base)
        return a[int(i) - 1, :] if j is _COLON else a[int(i) - 1, int(j) - 1]
    if tag == "colon":
        return _COLON
    if tag == "field":
        raise _unsupported("property access in a model body is outside the device-op set")
    if tag == "call":
        fn = ev(ast[1], env)
        args = [ev(a, env) for a in ast[2]]
        kwargs = {k: ev(v, env) for k, v in ast[3].items()}
        if not callable(fn):
            raise ModelSyntaxError(f"`{ast[1][1] if ast[1][0] == 'name' else '?'}` is not callable")
        return fn(*args, **kwargs)
    raise ModelSyntaxError(f"unsupported expression node {tag}")


# ---------------------------------------------------------------------------------------------
# statements -> transformer tree  (walk_body / gen_step)
# ---------------------------------------------------------------------------------------------
def _lhs_target(lhs, env):
    """-> column name or (name, j0) accessor target"""
    if lhs[0] == "name":
        return lhs[1]
    if lhs[0] == "curly":
        return dynname(lhs[1], ev(lhs[2], env))
    if lhs[0] == "index":
        base = _lhs_target(lhs[1], env)
        if isinstance(base, tuple):
            raise _unsupported("chained accessors are outside the device-op set")
        return (base, int(ev(lhs[2], env)) - 1)
    raise ModelSyntaxError("unsupported assignment target")


_ast_cache = {}


def _uses_resampled(cond):
    k = ("r", id(cond))
    v = _ast_cache.get(k)
    if v is None:
        v = _ast_cache[k] = (cond, "resampled" in _names_in(cond)[0])   # the AST is kept alive with its id
    return v[1]


def _build_is_pure(stmts):
    """True if constructing these statements assigns no build-time local (plain `=`, `+=`, ...), at any depth:
    then WHEN the transformers are constructed cannot be observed."""
    k = ("p", id(stmts))
    v = _ast_cache.get(k)
    if v is None:
        def pure(ss):
            for s in ss:
                if s[0] == "for":
                    if not pure(s[3]):
                        return False
                elif s[0] == "if":
                    if not pure(s[2]):
                        return False
                elif s[0] != "expr" and s[1] in ("=", "+=", "-=", "*=", "/="):
                    return False
            return True
        v = _ast_cache[k] = (stmts, pure(stmts))
    return v[1]


def _build(stmts, env, kernels, proposals):
    steps = []
    for s in stmts:
        if s[0] == "for":
            _, pat, it, body = s
            coll = ev(it, env)

            def bodyfn(x, pat=pat, body=body):
                vals = _destructure(pat, x, {})
                return core.Sequence(*_build(body, env.child(vals), kernels, proposals))
            steps.append(core.Loop(lambda state, coll=coll: coll, bodyfn))
        elif s[0] == "if":
            _, cond, body = s
            cenv = env

            uses_resampled = _uses_resampled(cond)

            def predfn(state, cond=cond, cenv=cenv, uses_resampled=uses_resampled):
                # `resampled` -> state.resampled (rewrites.jl:360-368); anything else is build-time
                vals = {"resampled": state.resampled} if uses_resampled else {}
                return bool(ev(cond, cenv.child(vals)))
            predfn.only_resampled = cond == ("name", "resampled")   # `if resampled`: lets a loop run its steps in blocks (core.Loop)
            if _build_is_pure(body):
                steps.append(core.Cond(predfn, lazy_body=lambda body=body, benv=env.snapshot(): core.Sequence(
                    *_build(body, benv, kernels, proposals))))
            else:   # build-time locals are assigned inside: construct now, as the reference does
                steps.append(core.Cond(predfn, core.Sequence(*_build(body, env.child({}), kernels, proposals))))
        elif s[0] == "expr":
            steps.append(core.Resample())
        else:
            _, op, lhs, rhs = s
            if op in ("=", "+=", "-=", "*=", "/="):
                v = ev(rhs, env)
                if lhs[0] == "tuple":
                    vals = tuple(v)
                    if len(vals) < len(lhs[1]):
                        raise ModelSyntaxError(f"cannot destructure {len(vals)} value(s) into {len(lhs[1])} names")
                    for t, x in zip(lhs[1], vals):
                        env.set_local(t[1], x)
                    continue
                if op != "=":
                    v = _binop(op[0], env.lookup(lhs[1]), v)
                env.set_local(lhs[1], v)
            elif op == ".=":
                steps.append(core.Assign(_lhs_target(lhs, env), ev(rhs, env)))
            elif op == "~":
                kernel = _resolve(rhs[1][1], kernels, env)
                args = tuple(ev(a, env) for a in rhs[2])
                if lhs == ("name", "_"):
                    core_k = kernel
                    steps.append(core.Weight(core_k, args))
                else:
                    steps.append(core.Sample(_lhs_target(lhs, env), kernel, args))
                steps.append(core.Resample())
            elif op == "=>":
                kernel = _resolve(rhs[1][1], kernels, env)
                args = tuple(ev(a, env) for a in rhs[2])
                steps.append(core.Observe(ev(lhs, env), kernel, args))
                steps.append(core.Resample())
            elif op == "<<":
                targets = lhs[1] if lhs[0] == "tuple" else [lhs]
                names = [_lhs_target(t, env) for t in targets]
                pname = rhs[1][1]
                table = dict(core.default_proposals)
                table.update(proposals or {})
                if pname not in table:
                    raise ModelSyntaxError(f"unknown proposal `{pname}`")
                args = tuple(ev(a, env) for a in rhs[2])
                kw = {k: ev(v, env) for k, v in rhs[3].items()}
                div = kw.pop("diversity", None)
                if kw:
                    raise ModelSyntaxError(f"unsupported proposal keyword(s) {sorted(kw)} (only `diversity`)")
                steps.append(core.Move(names, table[pname], args, div))
    return steps


def _resolve(name, kernels, env):
    if kernels and name in kernels:
        return core.resolve_kernel(kernels[name])
    try:
        v = env.lookup(name)
        if isinstance(v, core.WeightedKernel):
            return v
    except ModelSyntaxError:
        pass
    return core.resolve_kernel(name, kernels)


def model(src, particle_vars=(), scope=None):
    """``@model function f(args...) ... end`` -> Python function ``f(*args, kernels=None, proposals=None)``
    that builds (but does not run) the transformer ``Sequence``.

    ``particle_vars`` pre-registers columns that already exist on the state the model will run on (a
    continuation model applied to an existing SMCState, as benchmarks/ssm/bench_single_update does).
    ``scope`` supplies the names the Julia source takes from its enclosing module: helper functions written
    over particle expressions (``oscillator(t, A, ω, γ, ϕ)``) and user-defined ``WeightedKernel``s."""
    parser = Parser(tokenize(src))
    name, params, body = parser.parse_model()
    defaults, kwonly = parser.signature
    positional = [p for p in params if p not in kwonly]
    n_required = sum(1 for p in positional if p not in defaults)
    pv, fam = set(particle_vars), set()
    _static_check(body, pv, fam, set(params))

    def build(*args, kernels=None, proposals=None, **kwargs):
        if not (n_required <= len(args) <= len(positional)):
            takes = str(len(positional)) if n_required == len(positional) else f"from {n_required} to {len(positional)}"
            raise TypeError(f"{name}() takes {takes} positional arguments but {len(args)} were given")
        unknown = set(kwargs) - kwonly
        if unknown:
            raise TypeError(f"{name}() got unexpected keyword argument(s) {sorted(unknown)}")
        env = _Env(dict(zip(positional, args)), pv, fam, parent=_Env(dict(scope or {}), pv, fam))
        # defaults are evaluated left to right with the earlier parameters in scope, as Julia does
        for p in params:
            if p in kwonly and p in kwargs:
                env.values[p] = kwargs[p]
            elif p not in env.values:
                if p not in defaults:
                    raise TypeError(f"{name}(): keyword argument `{p}` not assigned")   # Julia: UndefKeywordError
                env.values[p] = ev(defaults[p], env)
        seq = core.Sequence(*_build(body, env, kernels, proposals))
        seq._has_moves = has_moves  # lets run() skip score-tape recording for move-free models
        return seq

    has_moves = "<<" in src
    build.__name__ = name
    build.particle_vars = frozenset(pv)
    build.dynamic_families = frozenset(fam)
    build.has_moves = has_moves
    return build

"""AMPL .nl reader and batched NLP evaluator (SURVEY.md section 8f-2).

The reference reads its test problems through Ipopt's AmplTNLP + ASL (src/SQPTNLP.cpp:13-132, test/simple_test.cpp:72-78;
format sample test/CUTE_examples/hs071.nl:1-75); neither library is available here, so this module restates what that
layer delivers to Algorithm.cpp for the text ("g") .nl format of the Hock-Schittkowski files:

  * Get_nlp_info / Get_bounds_info / Get_starting_point            (SQPTNLP.cpp:31-62)
  * Eval_f, Eval_gradient, Eval_constraints                        (SQPTNLP.cpp:67-92)
  * Eval_Jacobian / Get_Strucutre_Jacobian   FORTRAN-style triplets in ASL's column-major order       (:94-111)
  * Eval_Hessian  / Get_Structure_Hessian    upper triangle, column by column; the caller passes -lambda (:113-132)

All instances of a batch share the model and differ in x, so every evaluation is a straight-line program over
[batch]-long vectors.  The expression DAG is differentiated symbolically once (first and second order, with constant
folding so that structural zeros vanish) and emitted three times from one table of outputs: as numpy source for the host
mirror, by `cuda_source()` as CUDA kernels (one thread per instance) for a device-resident outer loop, and by `c_source()`
as C for one instance, the evaluator of the CPU oracle.
"""
import math
import os

import numpy as np

from .sqp_types import NLPInfo

_BIN = {0: "add", 1: "sub", 2: "mul", 3: "div", 5: "pow"}
# comparison opcodes -> (node kind, operands swapped, result negated): LT, LE, EQ, GE, GT, NE
_CMP = {22: ("lt", False, False), 23: ("le", False, False), 24: ("eq", False, False), 28: ("le", True, False), 29: ("lt", True, False),
        30: ("eq", False, True)}
_UN = {16: "neg", 39: "sqrt", 41: "sin", 43: "log", 44: "exp", 46: "cos", 15: "abs", 38: "tan", 49: "atan", 37: "tanh",
       40: "sinh", 45: "cosh", 42: "log10", 53: "acos", 51: "asin"}


class Graph:
    """Hash-consed expression DAG with local simplification.  Node = tuple; ids are positions in self.nodes."""

    def __init__(self):
        self.nodes, self.index = [], {}
        self._dep = {}  # node -> variables it depends on (nodes are immutable, so the memo lives as long as the graph)
        self.ZERO, self.ONE = self.const(0.0), self.const(1.0)

    def _mk(self, t):
        i = self.index.get(t)
        if i is None:
            i = len(self.nodes)
            self.nodes.append(t)
            self.index[t] = i
        return i

    def const(self, c):
        c = float(c)
        return self._mk(("const", c if c != 0.0 else 0.0))

    def var(self, i):
        return self._mk(("var", int(i)))

    def cval(self, a):
        t = self.nodes[a]
        return t[1] if t[0] == "const" else None

    def add(self, a, b):
        ca, cb = self.cval(a), self.cval(b)
        if ca is not None and cb is not None:
            return self.const(ca + cb)
        if ca == 0.0:
            return b
        if cb == 0.0:
            return a
        return self._mk(("add", a, b))

    def sub(self, a, b):
        ca, cb = self.cval(a), self.cval(b)
        if ca is not None and cb is not None:
            return self.const(ca - cb)
        if cb == 0.0:
            return a
        if ca == 0.0:
            return self.neg(b)
        if a == b:
            return self.ZERO
        return self._mk(("sub", a, b))

    def mul(self, a, b):
        ca, cb = self.cval(a), self.cval(b)
        if ca is not None and cb is not None:
            return self.const(ca * cb)
        if ca == 0.0 or cb == 0.0:
            return self.ZERO
        if ca == 1.0:
            return b
        if cb == 1.0:
            return a
        if ca == -1.0:
            return self.neg(b)
        if cb == -1.0:
            return self.neg(a)
        return self._mk(("mul", a, b))

    def div(self, a, b):
        ca, cb = self.cval(a), self.cval(b)
        if ca is not None and cb is not None and cb != 0.0:
            return self.const(ca / cb)
        if ca == 0.0:
            return self.ZERO
        if cb == 1.0:
            return a
        return self._mk(("div", a, b))

    def pow(self, a, b):
        ca, cb = self.cval(a), self.cval(b)
        if cb == 0.0:
            return self.ONE
        if cb == 1.0:
            return a
        if ca is not None and cb is not None:
            try:
                return self.const(math.pow(ca, cb))
            except (ValueError, OverflowError):
                pass
        return self._mk(("pow", a, b))

    def neg(self, a):
        ca = self.cval(a)
        if ca is not None:
            return self.const(-ca)
        if self.nodes[a][0] == "neg":
            return self.nodes[a][1]
        return self._mk(("neg", a))

    def un(self, op, a):
        if op == "neg":
            return self.neg(a)
        ca = self.cval(a)
        if ca is not None:
            try:
                if op == "ncdf":
                    return self.const(0.5 * math.erfc(-ca * 0.7071067811865476))
                return self.const(getattr(math, {"abs": "fabs"}.get(op, op))(ca))
            except (ValueError, OverflowError):
                pass
        return self._mk((op, a))

    # ---- non-smooth operators of the CUTE models beyond the HS set: comparisons give 1.0 / 0.0, `if` selects
    def cmp(self, op, a, b):
        ca, cb = self.cval(a), self.cval(b)
        if ca is not None and cb is not None:
            return self.ONE if {"le": ca <= cb, "lt": ca < cb, "eq": ca == cb}[op] else self.ZERO
        return self._mk((op, a, b))

    def ifelse(self, c, a, b):
        cc = self.cval(c)
        if cc is not None:
            return a if cc != 0.0 else b
        if a == b:
            return a
        return self._mk(("if", c, a, b))

    def min2(self, a, b):
        return self.ifelse(self.cmp("le", a, b), a, b)

    def max2(self, a, b):
        return self.ifelse(self.cmp("le", b, a), a, b)

    def sum(self, args):
        out = self.ZERO
        for a in args:
            out = self.add(out, a)
        return out

    # ---- differentiation (memoised per variable)
    def diff(self, a, v, memo):
        """d node / d x_v.  Post-order over an explicit stack: a sum of a thousand terms is a chain of a thousand `add` nodes
        (the CUTE models beyond the HS set), which a recursive walk cannot descend."""
        if (a, v) in memo:
            return memo[(a, v)]
        stack = [a]
        while stack:
            node = stack[-1]
            if (node, v) in memo:
                stack.pop()
                continue
            if v not in self.depends(node, self._dep):  # structurally zero: no walk through the subtree (the local
                memo[(node, v)] = self.ZERO             # simplifications would reduce it to ZERO anyway)
                stack.pop()
                continue
            t = self.nodes[node]
            missing = [k for k in t[1:] if (k, v) not in memo] if t[0] not in ("const", "var") else []
            if missing:
                stack.extend(missing)
                continue
            memo[(node, v)] = self._diff_node(node, v, memo)  # every child is in the memo: the calls below return at once
            stack.pop()
        return memo[(a, v)]

    def _diff_node(self, a, v, memo):
        key = (a, v)
        if key in memo:
            return memo[key]
        t = self.nodes[a]
        op = t[0]
        if op == "const":
            r = self.ZERO
        elif op == "var":
            r = self.ONE if t[1] == v else self.ZERO
        elif op == "add":
            r = self.add(self.diff(t[1], v, memo), self.diff(t[2], v, memo))
        elif op == "sub":
            r = self.sub(self.diff(t[1], v, memo), self.diff(t[2], v, memo))
        elif op == "mul":
            r = self.add(self.mul(self.diff(t[1], v, memo), t[2]), self.mul(t[1], self.diff(t[2], v, memo)))
        elif op == "div":
            da, db = self.diff(t[1], v, memo), self.diff(t[2], v, memo)
            r = self.sub(self.div(da, t[2]), self.div(self.mul(a, db), t[2]))  # (a/b)' = a'/b - (a/b) b'/b
        elif op == "pow":
            base, ex = t[1], t[2]
            db, de = self.diff(base, v, memo), self.diff(ex, v, memo)
            ce = self.cval(ex)
            if ce is not None:
                r = self.mul(self.mul(ex, self.pow(base, self.const(ce - 1.0))), db)
            else:
                r = self.mul(a, self.add(self.mul(de, self.un("log", base)), self.div(self.mul(ex, db), base)))
        elif op == "neg":
            r = self.neg(self.diff(t[1], v, memo))
        elif op in ("le", "lt", "eq"):
            r = self.ZERO  # piecewise constant
        elif op == "if":
            r = self.ifelse(t[1], self.diff(t[2], v, memo), self.diff(t[3], v, memo))  # derivative of the selected branch
        else:
            u, du = t[1], self.diff(t[1], v, memo)
            if du == self.ZERO:
                r = self.ZERO
            elif op == "sqrt":
                r = self.div(du, self.mul(self.const(2.0), a))
            elif op == "sin":
                r = self.mul(self.un("cos", u), du)
            elif op == "cos":
                r = self.neg(self.mul(self.un("sin", u), du))
            elif op == "log":
                r = self.div(du, u)
            elif op == "log10":
                r = self.div(du, self.mul(u, self.const(math.log(10.0))))
            elif op == "exp":
                r = self.mul(a, du)
            elif op == "tan":
                r = self.mul(self.add(self.ONE, self.mul(a, a)), du)
            elif op == "atan":
                r = self.div(du, self.add(self.ONE, self.mul(u, u)))
            elif op == "tanh":
                r = self.mul(self.sub(self.ONE, self.mul(a, a)), du)
            elif op == "sinh":
                r = self.mul(self.un("cosh", u), du)
            elif op == "cosh":
                r = self.mul(self.un("sinh", u), du)
            elif op == "asin":
                r = self.div(du, self.un("sqrt", self.sub(self.ONE, self.mul(u, u))))
            elif op == "acos":
                r = self.neg(self.div(du, self.un("sqrt", self.sub(self.ONE, self.mul(u, u)))))
            elif op == "abs":
                r = self.mul(self.div(u, a), du)
            elif op == "ncdf":  # standard normal distribution function: Phi'(u) = exp(-u^2/2) / sqrt(2 pi)
                r = self.mul(self.mul(self.const(0.3989422804014327), self.un("exp", self.mul(self.const(-0.5), self.mul(u, u)))), du)
            else:
                raise NotImplementedError(op)
        memo[key] = r
        return r

    def depends(self, a, memo):
        """frozenset of variable indices the node depends on (explicit stack, see diff)"""
        stack = [a]
        while stack:
            node = stack[-1]
            if node in memo:
                stack.pop()
                continue
            t = self.nodes[node]
            if t[0] == "const":
                memo[node] = frozenset()
            elif t[0] == "var":
                memo[node] = frozenset([t[1]])
            else:
                missing = [k for k in t[1:] if k not in memo]
                if missing:
                    stack.extend(missing)
                    continue
                memo[node] = frozenset().union(*[memo[k] for k in t[1:]])
            stack.pop()
        return memo[a]


class _Tokens:
    def __init__(self, text):
        self.lines = [ln.split("#")[0].rstrip() for ln in text.splitlines()]
        self.pos = 0

    def next(self):
        ln = self.lines[self.pos]
        self.pos += 1
        return ln

    def more(self):
        while self.pos < len(self.lines) and not self.lines[self.pos].strip():
            self.pos += 1
        return self.pos < len(self.lines)


# Imported functions (F segments).  The reference's HS models declare one, `myerf` (hs068, hs069), implemented by an AMPL function
# library that is not part of the reference; Hock-Schittkowski 68 / 69 define it as the standard normal distribution function
# Phi (with it the tabulated solution of hs068 satisfies x3 = 2 Phi(-x2) to all printed digits).
_IMPORTED = {"myerf": "ncdf"}


def _read_expr(tok, G, defined, funcs=None):
    ln = tok.next().strip()
    k = ln[0]
    if k == "f":
        idx, nargs = (int(t) for t in ln[1:].split())
        args = [_read_expr(tok, G, defined, funcs) for _ in range(nargs)]
        name = (funcs or {}).get(idx)
        if name not in _IMPORTED or nargs != 1:
            raise NotImplementedError("imported function %r with %d arguments" % (name, nargs))
        return G.un(_IMPORTED[name], args[0])
    if k == "n":
        return G.const(float(ln[1:]))
    if k == "v":
        i = int(ln[1:])
        return defined[i] if i in defined else G.var(i)
    if k == "o":
        op = int(ln[1:])
        if op in _BIN:
            a = _read_expr(tok, G, defined, funcs)
            b = _read_expr(tok, G, defined, funcs)
            return getattr(G, _BIN[op])(a, b)
        if op in _UN:
            return G.un(_UN[op], _read_expr(tok, G, defined, funcs))
        if op == 54:
            cnt = int(tok.next().strip())
            return G.sum([_read_expr(tok, G, defined, funcs) for _ in range(cnt)])
        if op in (11, 12):  # MINLIST / MAXLIST
            cnt = int(tok.next().strip())
            args = [_read_expr(tok, G, defined, funcs) for _ in range(cnt)]
            out = args[0]
            for a in args[1:]:
                out = G.min2(out, a) if op == 11 else G.max2(out, a)
            return out
        if op in _CMP:  # comparisons: 1.0 / 0.0
            a = _read_expr(tok, G, defined, funcs)
            b = _read_expr(tok, G, defined, funcs)
            kind, swap, negate = _CMP[op]
            r_ = G.cmp(kind, b, a) if swap else G.cmp(kind, a, b)
            return G.sub(G.ONE, r_) if negate else r_
        if op in (20, 21):  # OR, AND on 0 / 1 values
            a = _read_expr(tok, G, defined, funcs)
            b = _read_expr(tok, G, defined, funcs)
            return G.mul(a, b) if op == 21 else G.sub(G.add(a, b), G.mul(a, b))
        if op == 34:  # NOT
            return G.sub(G.ONE, _read_expr(tok, G, defined, funcs))
        if op == 35:  # if c then a else b
            c = _read_expr(tok, G, defined, funcs)
            a = _read_expr(tok, G, defined, funcs)
            b = _read_expr(tok, G, defined, funcs)
            return G.ifelse(c, a, b)
        raise NotImplementedError("nl opcode o%d" % op)
    raise NotImplementedError("nl expression token %r" % ln)


def _read_bounds(tok, count):
    lo, hi = np.empty(count), np.empty(count)
    for i in range(count):
        f = tok.next().split()
        kind = int(f[0])
        if kind == 0:
            lo[i], hi[i] = float(f[1]), float(f[2])
        elif kind == 1:
            lo[i], hi[i] = -np.inf, float(f[1])
        elif kind == 2:
            lo[i], hi[i] = float(f[1]), np.inf
        elif kind == 3:
            lo[i], hi[i] = -np.inf, np.inf
        elif kind == 4:
            lo[i] = hi[i] = float(f[1])
        else:
            raise NotImplementedError("complementarity constraints")
    return lo, hi


class NLModel:
    """Parsed .nl problem: expression ids in a Graph plus bounds, start and the linear parts."""

    def __init__(self, path):
        with open(path) as f:
            text = f.read()
        if not text.startswith("g"):
            raise ValueError("only the text ('g') .nl format is read")
        tok = _Tokens(text)
        hdr = [tok.next().split() for _ in range(10)]
        self.name = os.path.splitext(os.path.basename(path))[0]
        self.n, self.m, self.n_obj = int(hdr[1][0]), int(hdr[1][1]), int(hdr[1][2])
        funcs = {}
        self.nzJ = int(hdr[7][0])
        G = self.G = Graph()
        n, m = self.n, self.m
        self.con_nl = [G.ZERO] * m
        self.obj_nl, self.obj_sense = G.ZERO, 0
        self.con_lin = [dict() for _ in range(m)]
        self.obj_lin = {}
        self.x0 = np.zeros(n)
        self.lam0 = np.zeros(m)
        self.x_l, self.x_u = np.full(n, -np.inf), np.full(n, np.inf)
        self.c_l, self.c_u = np.full(m, -np.inf), np.full(m, np.inf)
        defined = {}
        while tok.more():
            ln = tok.next().strip()
            k, rest = ln[0], ln[1:].split()
            if k == "F":
                funcs[int(rest[0])] = rest[3]
            elif k == "C":
                self.con_nl[int(rest[0])] = _read_expr(tok, G, defined, funcs)
            elif k == "O":
                if int(rest[0]) == 0:
                    self.obj_sense = int(rest[1])
                    self.obj_nl = _read_expr(tok, G, defined, funcs)
                else:
                    _read_expr(tok, G, defined, funcs)
            elif k == "V":
                idx, nlin = int(rest[0]), int(rest[1])
                e = G.ZERO
                for _ in range(nlin):
                    f = tok.next().split()
                    j = int(f[0])
                    e = G.add(e, G.mul(G.const(float(f[1])), defined[j] if j in defined else G.var(j)))
                defined[idx] = G.add(e, _read_expr(tok, G, defined, funcs))
            elif k == "r":
                self.c_l, self.c_u = _read_bounds(tok, m)
            elif k == "b":
                self.x_l, self.x_u = _read_bounds(tok, n)
            elif k == "x":
                for _ in range(int(rest[0])):
                    f = tok.next().split()
                    self.x0[int(f[0])] = float(f[1])
            elif k == "d":
                for _ in range(int(rest[0])):
                    f = tok.next().split()
                    self.lam0[int(f[0])] = float(f[1])
            elif k == "k":
                for _ in range(int(rest[0])):
                    tok.next()
            elif k == "J":
                i = int(rest[0])
                for _ in range(int(rest[1])):
                    f = tok.next().split()
                    self.con_lin[i][int(f[0])] = float(f[1])
            elif k == "G":
                i = int(rest[0])
                for _ in range(int(rest[1])):
                    f = tok.next().split()
                    if i == 0:
                        self.obj_lin[int(f[0])] = float(f[1])
            elif k == "S":
                for _ in range(int(rest[1])):
                    tok.next()
            else:
                raise NotImplementedError("nl segment %r" % ln)


_INFIX = {"add": "+", "sub": "-", "mul": "*", "div": "/"}
_CMP_C = {"le": "<=", "lt": "<", "eq": "=="}
_MATH_NAMES = ("pow", "sqrt", "sin", "cos", "log", "exp", "tan", "atan", "tanh", "sinh", "cosh", "log10", "acos", "asin")
# the functions each dialect of _emit calls (a name missing from a table is called as is); "nl" is C whose transcendental
# functions go through __noinline__ wrappers (emitted once by cuda_source for the chunked form): inlined, every pow() is a few
# hundred instructions and the kernels of hs025 / hs105 reach 5 MB of SASS
_FUN = {"py": {"pow": "np.power", "sqrt": "np.sqrt", "sin": "np.sin", "cos": "np.cos", "log": "np.log", "exp": "np.exp", "abs": "np.abs",
               "tan": "np.tan", "atan": "np.arctan", "tanh": "np.tanh", "sinh": "np.sinh", "cosh": "np.cosh", "log10": "np.log10",
               "acos": "np.arccos", "asin": "np.arcsin", "ncdf": "_ncdf"},
        "c": {"abs": "fabs"}}
_FUN["nl"] = dict(_FUN["c"], **{f: "nl_" + f for f in _MATH_NAMES})
_MATH_WRAPPERS = (["static __device__ __noinline__ double nl_pow(double a, double b) { return pow(a, b); }"] +
                  ["static __device__ __noinline__ double nl_%s(double a) { return %s(a); }" % (f, f) for f in _MATH_NAMES if f != "pow"])


def _emit(G, roots, lang):
    """Straight-line code computing the nodes `roots` in dialect `lang` ("py", "c" or "nl", see _FUN); returns (lines,
    name_of(node), the compute nodes in the order of `lines`, the sorted indices of the variables the program reads)."""
    order, seen = [], set()

    def visit(a):
        stack = [(a, False)]
        while stack:
            node, done = stack.pop()
            if done:
                order.append(node)
                continue
            if node in seen:
                continue
            seen.add(node)
            stack.append((node, True))
            t = G.nodes[node]
            if t[0] not in ("const", "var"):
                for k in t[1:]:
                    if k not in seen:
                        stack.append((k, False))

    for r in roots:
        visit(r)
    py, fun = lang == "py", _FUN[lang]
    name, lines, compute, xs = {}, [], [], []
    for a in order:
        t = G.nodes[a]
        if t[0] == "const":
            name[a] = repr(t[1]) if t[1] >= 0 else "(%r)" % t[1]
            continue
        if t[0] == "var":
            name[a] = "x%d" % t[1]
            xs.append(t[1])
            continue
        nm = "t%d" % a
        if t[0] in _INFIX:
            rhs = "%s %s %s" % (name[t[1]], _INFIX[t[0]], name[t[2]])
        elif t[0] == "pow":
            ce = G.cval(t[2])
            if ce == 2.0:
                rhs = "%s * %s" % (name[t[1]], name[t[1]])
            else:
                rhs = "%s(%s, %s)" % (fun.get("pow", "pow"), name[t[1]], name[t[2]])
        elif t[0] == "neg":
            rhs = "-%s" % name[t[1]]
        elif t[0] in _CMP_C:
            rhs = ("(%s %s %s) * 1.0" if py else "(%s %s %s ? 1.0 : 0.0)") % (name[t[1]], _CMP_C[t[0]], name[t[2]])
        elif t[0] == "if":
            rhs = ("np.where(%s != 0.0, %s, %s)" if py else "(%s != 0.0 ? %s : %s)") % (name[t[1]], name[t[2]], name[t[3]])
        else:
            rhs = "%s(%s)" % (fun.get(t[0], t[0]), name[t[1]])
        lines.append(("%s = %s" if py else "const double %s = %s;") % (nm, rhs))
        name[a] = nm
        compute.append(a)
    return lines, name, compute, sorted(xs)


def _emit_chunked_cuda(G, roots, tag, chunk, n):
    """The straight-line program of `roots` cut into consecutive pieces of `chunk` statements, each a __noinline__ device
    function: NVRTC's time grows much faster than linearly with the length of one function (hs105, 20 k statements in one
    kernel: 47 s), while the sum over pieces of a few thousand statements stays linear.  Values that cross a piece boundary go
    through a per-thread scratch array T (local memory); evaluation order and arithmetic are exactly those of the one-piece
    program.  Returns (source lines of the device functions, body lines of the kernel after `b` / bounds check, name_of(root))."""
    lines, name, order, _ = _emit(G, roots, "nl")
    pos = {a: i // chunk for i, a in enumerate(order)}
    npieces = (len(order) + chunk - 1) // chunk
    last_use = {}  # node -> last piece that reads it (npieces = the kernel epilogue)
    for a in order:
        t = G.nodes[a]
        for k in t[1:]:
            if k in pos and pos[a] > last_use.get(k, -1):
                last_use[k] = pos[a]
    for r_ in roots:
        if r_ in pos:
            last_use[r_] = npieces
    cross = [a for a in order if last_use.get(a, -1) > pos[a]]
    tidx = {a: i for i, a in enumerate(cross)}
    funcs, calls = [], []
    for pc in range(npieces):
        seg = order[pc * chunk:(pc + 1) * chunk]
        segset = set(seg)
        ins, xs = [], set()
        for a in seg:
            for k in G.nodes[a][1:]:
                tk = G.nodes[k]
                if tk[0] == "var":
                    xs.add(tk[1])
                elif k in pos and k not in segset and k not in ins:
                    ins.append(k)
        fn = "nlp_piece_%s_%d" % (tag, pc)
        funcs.append("static __device__ __noinline__ void %s(const double* __restrict__ xv, double* __restrict__ T) {" % fn)
        funcs += ["    const double x%d = xv[%d];" % (j, j) for j in sorted(xs)]
        funcs += ["    const double t%d = T[%d];" % (k, tidx[k]) for k in ins]
        funcs += ["    " + lines[i] for i in range(pc * chunk, min((pc + 1) * chunk, len(order)))]
        funcs += ["    T[%d] = t%d;" % (tidx[a], a) for a in seg if a in tidx]
        funcs += ["}", ""]
        calls.append("    %s(xv, T);" % fn)
    body = ["    double xv[%d];" % max(n, 1), "    double T[%d];" % max(len(cross), 1)]
    body += ["    for (int j = 0; j < %d; j++) xv[j] = x[(size_t)b * %d + j];" % (n, n)] + calls
    rname = {}
    for r_ in roots:
        if r_ in tidx:
            rname[r_] = "T[%d]" % tidx[r_]
        else:
            nm = name[r_]
            rname[r_] = ("xv[%s]" % nm[1:]) if G.nodes[r_][0] == "var" else nm
    return funcs, body, rname


class AmplNLP:
    """The SQPTNLP-shaped view of an NLModel, batched over instances (x is [batch][n])."""

    def __init__(self, path):
        md = self.model = NLModel(path) if not isinstance(path, NLModel) else path
        G, n, m = md.G, md.n, md.m
        self.n, self.m, self.name = n, m, md.name
        sgn = -1.0 if md.obj_sense == 1 else 1.0  # AmplTNLP minimises -f for "maximize"
        f = G.add(md.obj_nl, G.sum([G.mul(G.const(c), G.var(j)) for j, c in sorted(md.obj_lin.items())]))
        self.f_node = G.mul(G.const(sgn), f)
        self.c_nodes = [G.add(md.con_nl[i], G.sum([G.mul(G.const(c), G.var(j)) for j, c in sorted(md.con_lin[i].items())]))
                        for i in range(m)]
        memo = {}
        dep = G._dep
        self.grad_nodes = [G.diff(self.f_node, j, memo) for j in range(n)]
        # Jacobian structure: the J segments (every variable that appears in a row), column-major like ASL's goff
        ent = sorted((j, i) for i in range(m) for j in md.con_lin[i])
        self.J_col1 = np.array([j + 1 for j, i in ent], np.int32)
        self.J_row1 = np.array([i + 1 for j, i in ent], np.int32)
        self.jac_nodes = [G.diff(self.c_nodes[i], j, memo) for j, i in ent]
        for i in range(m):
            extra = G.depends(self.c_nodes[i], dep) - set(md.con_lin[i])
            if extra:
                raise ValueError("constraint %d depends on variables missing from its J segment: %s" % (i, sorted(extra)))
        # Hessian of the Lagrangian: upper triangle, column by column; structure = union of structural non-zeros
        funcs = [self.f_node] + self.c_nodes
        hess = {}
        for k, fn in enumerate(funcs):  # only the variables a function depends on can carry a derivative (same entries, same order)
            for j in sorted(G.depends(fn, dep)):
                dj = G.diff(fn, j, memo)
                if dj == G.ZERO:
                    continue
                for i in sorted(v for v in G.depends(dj, dep) if v <= j):
                    d2 = G.diff(dj, i, memo)
                    if d2 != G.ZERO:
                        hess.setdefault((j, i), []).append((k, d2))
        hk = sorted(hess)
        self.H_col1 = np.array([j + 1 for j, i in hk], np.int32)
        self.H_row1 = np.array([i + 1 for j, i in hk], np.int32)
        self._hess_terms = [hess[k] for k in hk]
        # what every evaluator stores, in store order, keyed by the name of the output array (and of the numpy function, eval_<key>):
        # an entry is a sum of terms (k, node), the node times lam[k-1] when k > 0
        self._outputs = {"f": [[(0, self.f_node)]], "c": [[(0, a)] for a in self.c_nodes], "grad": [[(0, a)] for a in self.grad_nodes],
                         "jac": [[(0, a)] for a in self.jac_nodes], "hess": self._hess_terms}
        self._compile()

    # ---- code generation
    def _roots(self, outs):
        """The nodes the outputs `outs` store, in store order."""
        return [a for o in outs for terms in self._outputs[o] for _, a in terms]

    def _stores(self, outs, nm, store, lam):
        """Statements writing the outputs `outs` from the program's values nm: store(output, entry, value) is one statement of
        the dialect, lam(k) the multiplier of constraint k."""
        return ["    " + store(o, e, " + ".join(nm[a] if k == 0 else "%s * %s" % (lam(k - 1), nm[a]) for k, a in terms))
                for o in outs for e, terms in enumerate(self._outputs[o])]

    def _compile(self):
        src = ["import numpy as np", "from scipy.special import ndtr as _ncdf", ""]
        store = lambda o, e, v: "return np.zeros(B) + %s" % v if o == "f" else "out[:, %d] = %s" % (e, v)
        for o, entries in self._outputs.items():
            lines, nm, _, _ = _emit(self.model.G, self._roots([o]), "py")
            src += ["def eval_%s(x%s):" % (o, ", lam" if o == "hess" else ""), "    B = x.shape[0]"]
            src += ["    x%d = x[:, %d]" % (j, j) for j in range(self.n)] + ["    " + ln for ln in lines]
            stores = self._stores([o], nm, store, lambda k: "lam[:, %d]" % k)
            src += stores if o == "f" else ["    out = np.empty((B, %d))" % len(entries)] + stores + ["    return out"]
            src.append("")
        self.source = "\n".join(src)
        ns = {}
        exec(compile(self.source, "<nl:%s>" % self.name, "exec"), ns)
        self._f, self._c, self._g, self._j, self._h = (ns["eval_" + o] for o in self._outputs)

    CUDA_PIECE = 1500  # statements per device function of the chunked form (large DAGs)

    def cuda_source(self, piece=None):
        """The same straight-line programs as two CUDA kernels, one thread per instance, instance-major outputs:
        nlp_eval_fc (f, c at trial points) and nlp_eval_all (f, c, grad f, Jacobian and Lagrangian-Hessian triplet
        values).  Compiled at run time by sqpb200_nlp_compile (NVRTC, sm_100a, --fmad=false).  Programs longer than `piece`
        statements are cut into __noinline__ device functions of that length (_emit_chunked_cuda)."""
        G, n = self.model.G, self.n
        piece = self.CUDA_PIECE if piece is None else piece
        chunked = sum(1 for t in G.nodes if t[0] not in ("const", "var")) > piece
        src = ["// generated by restartsqp_b200/nl_reader.py from %s.nl" % self.name +
               (" (chunked: %d statements per device function)" % piece if chunked else ""),
               "static __device__ __forceinline__ double ncdf(double u) { return 0.5 * erfc(-u * 0.7071067811865476); }"]
        if chunked:
            src += _MATH_WRAPPERS + [""]
        store = lambda o, e, v: ("f[b] = %s;" % v if o == "f" else
                                 "%s[(size_t)b * %d + %d] = %s;" % (o, len(self._outputs[o]), e, v))
        lam = lambda k: "lam[(size_t)b * %d + %d]" % (self.m, k)
        kernels = []
        for tag, outs, sig in (
                ("fc", ("f", "c"),
                 ['extern "C" __global__ void nlp_eval_fc(int B, const double* __restrict__ x, double* __restrict__ f, double* __restrict__ c) {']),
                ("all", tuple(self._outputs),
                 ['extern "C" __global__ void nlp_eval_all(int B, const double* __restrict__ x, const double* __restrict__ lam,',
                  "                                        double* __restrict__ f, double* __restrict__ c, double* __restrict__ grad,",
                  "                                        double* __restrict__ jac, double* __restrict__ hess) {"])):
            if chunked:  # the device functions go ahead of both kernels
                funcs, body, nm = _emit_chunked_cuda(G, self._roots(outs), tag, piece, n)
                src += funcs
            else:
                lines, nm, _, xs = _emit(G, self._roots(outs), "c")
                body = ["    const double x%d = x[(size_t)b * %d + %d];" % (j, n, j) for j in xs] + ["    " + ln for ln in lines]
            kernels += sig + ["    const int b = blockIdx.x * blockDim.x + threadIdx.x;", "    if (b >= B) return;"] + body
            kernels += self._stores(outs, nm, store, lam) + ["}", ""]
        return "\n".join(src + kernels[:-1])  # no blank line after the last kernel

    def c_source(self):
        """The straight-line programs as plain C for ONE instance (nlp_fc, nlp_all): used by the CPU oracle's SQP loop
        (oracle/oracle_sqp.c), i.e. by tests and by bench.py's CPU figure, never by the product path."""
        src = ["#include <math.h>", "/* generated by restartsqp_b200/nl_reader.py from %s.nl */" % self.name,
               "static double ncdf(double u) { return 0.5 * erfc(-u * 0.7071067811865476); }"]
        store = lambda o, e, v: "*f = %s;" % v if o == "f" else "%s[%d] = %s;" % (o, e, v)
        for sig, outs in (("void nlp_fc(const double* x, double* f, double* c) {", ("f", "c")),
                          ("void nlp_all(const double* x, const double* lam, double* f, double* c, double* grad, double* jac, double* hess) {",
                           tuple(self._outputs))):
            lines, nm, _, xs = _emit(self.model.G, self._roots(outs), "c")
            src += [sig] + ["    const double x%d = x[%d];" % (j, j) for j in xs] + ["    " + ln for ln in lines]
            src += self._stores(outs, nm, store, lambda k: "lam[%d]" % k) + ["}", ""]
        return "\n".join(src[:-1])  # no blank line after the last function

    # ---- SQPTNLP interface (src/SQPTNLP.cpp)
    def Get_nlp_info(self):
        return NLPInfo(nCon=self.m, nVar=self.n, nnz_jac_g=len(self.jac_nodes), nnz_h_lag=len(self._hess_terms))

    def Get_bounds_info(self):
        md = self.model
        big = 1.0e19  # Ipopt's nlp_{lower,upper}_bound_inf as AmplTNLP reports infinite bounds
        cv = lambda v: np.where(np.isinf(v), np.sign(v) * big, v)
        return cv(md.x_l), cv(md.x_u), cv(md.c_l), cv(md.c_u)

    def Get_starting_point(self):
        return self.model.x0.copy(), self.model.lam0.copy()

    def _x(self, x):
        return np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)

    def Eval_f(self, x):
        with np.errstate(all="ignore"):
            return self._f(self._x(x))

    def Eval_constraints(self, x):
        with np.errstate(all="ignore"):
            return self._c(self._x(x))

    def Eval_gradient(self, x):
        with np.errstate(all="ignore"):
            return self._g(self._x(x))

    def Eval_Jacobian(self, x):
        with np.errstate(all="ignore"):
            return self._j(self._x(x))

    def Eval_Hessian(self, x, lam):
        with np.errstate(all="ignore"):
            return self._h(self._x(x), np.ascontiguousarray(np.atleast_2d(lam), dtype=np.float64))


def write_model_file(nlp, path, x0=None):
    """Hand a model to the C++ batched driver (restartsqp_b200/csrc/driver/batched_sqp_main.cpp -> BatchedAlgorithm): sizes,
    bounds, starting point, 1-based sparsity patterns, the starting points [B][n] and the CUDA source of the batched evaluator.
    Doubles are written as C99 hex floats: the hand-over is exact."""
    h = nlp if isinstance(nlp, AmplNLP) else AmplNLP(nlp)
    xl, xu, cl, cu = h.Get_bounds_info()
    xs, ls = h.Get_starting_point()
    x0 = np.atleast_2d(np.asarray(xs if x0 is None else x0, dtype=np.float64))
    hx = lambda a: " ".join(("inf" if v == np.inf else "-inf" if v == -np.inf else float(v).hex()) for v in np.asarray(a, dtype=np.float64).ravel())
    ints = lambda a: " ".join(str(int(v)) for v in a)
    with open(path, "w") as f:
        f.write("%d %d %d %d %d\n" % (h.n, h.m, len(h.J_row1), len(h.H_row1), x0.shape[0]))
        for a in (xl, xu, cl, cu, xs, np.asarray(ls, dtype=np.float64).reshape(-1)[:h.m]):
            f.write(hx(a) + "\n")
        for a in (h.J_row1, h.J_col1, h.H_row1, h.H_col1):
            f.write(ints(a) + "\n")
        f.write(hx(x0) + "\n---SOURCE---\n")
        f.write(h.cuda_source())


class DeviceNLP:
    """AmplNLP whose evaluations run on the GPU: the generated CUDA source is compiled with NVRTC through the C ABI
    (sqpb200_nlp_compile / _load / _eval).  Same SQPTNLP-shaped interface plus the fused calls the batched driver prefers
    (Eval_f_c for trial points, Eval_all for accepted points).  There is no CPU fallback: constructing it without a CUDA
    device raises."""

    MAX_NODES = 200000  # large DAGs are compiled in pieces (AmplNLP.cuda_source); hs092, the largest HS model, has 121 k nodes

    def __init__(self, path, device=0, max_nodes=None):
        import ctypes as C
        from . import _capi as capi
        self.host = path if isinstance(path, AmplNLP) else AmplNLP(path)
        h = self.host
        limit = self.MAX_NODES if max_nodes is None else max_nodes
        if len(h.model.G.nodes) > limit:
            raise ValueError("%s: expression DAG of %d nodes exceeds the device-evaluator limit of %d (NVRTC compile time)"
                             % (h.name, len(h.model.G.nodes), limit))
        self.n, self.m, self.name = h.n, h.m, h.name
        self.J_row1, self.J_col1, self.H_row1, self.H_col1 = h.J_row1, h.J_col1, h.H_row1, h.H_col1
        self.zJ, self.zH = len(h.J_row1), len(h.H_row1)
        self._C, self._capi, self.L = C, capi, capi.lib()
        self.h = C.c_void_p()
        log = C.create_string_buffer(4096)
        rc = self.L.sqpb200_nlp_compile(h.cuda_source().encode(), self.n, self.m, self.zJ, self.zH, log, 4096, C.byref(self.h))
        if rc != 0:
            raise RuntimeError("sqpb200_nlp_compile(%s) failed (%d): %s" % (self.name, rc, self.L.sqpb200_nlp_last_error().decode()))
        rc = self.L.sqpb200_nlp_load(self.h, device)
        if rc != 0:
            raise capi.SqpB200Error("sqpb200_nlp_load failed (%d): %s" % (rc, self.L.sqpb200_nlp_last_error().decode()))

    def close(self):
        if self.h:
            self.L.sqpb200_nlp_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def Get_nlp_info(self): return self.host.Get_nlp_info()
    def Get_bounds_info(self): return self.host.Get_bounds_info()
    def Get_starting_point(self): return self.host.Get_starting_point()
    def launch_count(self): return int(self.L.sqpb200_nlp_launch_count(self.h))

    def _eval(self, which, x, lam=None):
        C = self._C
        x = np.ascontiguousarray(np.atleast_2d(x), dtype=np.float64)
        B = x.shape[0]
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
        f, c = np.empty(B), np.empty((B, self.m))
        g = jv = hv = None
        if which == 1:
            lam = np.ascontiguousarray(np.atleast_2d(lam), dtype=np.float64).reshape(B, self.m)
            g, jv, hv = np.empty((B, self.n)), np.empty((B, self.zJ)), np.empty((B, self.zH))
        rc = self.L.sqpb200_nlp_eval(self.h, which, B, p(x), p(lam), p(f), p(c), p(g), p(jv), p(hv), self._capi.LOC_HOST, None)
        if rc != 0:
            raise self._capi.SqpB200Error("sqpb200_nlp_eval failed (%d): %s" % (rc, self.L.sqpb200_nlp_last_error().decode()))
        return f, c, g, jv, hv

    def eval_device(self, which, B, x, lam=None, f=None, c=None, grad=None, jac=None, hess=None, stream=None):
        """Evaluation with every array already in device memory (CUDA tensors); asynchronous on `stream` (a torch.cuda.Stream; None:
        the default stream)."""
        p = lambda t: None if t is None else self._C.c_void_p(t.data_ptr())
        s = None if stream is None else self._C.c_void_p(stream.cuda_stream)
        rc = self.L.sqpb200_nlp_eval(self.h, which, B, p(x), p(lam), p(f), p(c), p(grad), p(jac), p(hess), self._capi.LOC_DEVICE, s)
        if rc != 0:
            raise self._capi.SqpB200Error("sqpb200_nlp_eval failed (%d): %s" % (rc, self.L.sqpb200_nlp_last_error().decode()))

    def Eval_f_c(self, x):
        f, c, _, _, _ = self._eval(0, x)
        return f, c

    def Eval_all(self, x, lam):
        return self._eval(1, x, lam)

    def Eval_f(self, x): return self._eval(0, x)[0]
    def Eval_constraints(self, x): return self._eval(0, x)[1]
    def Eval_gradient(self, x): return self._eval(1, x, np.zeros((np.atleast_2d(x).shape[0], self.m)))[2]
    def Eval_Jacobian(self, x): return self._eval(1, x, np.zeros((np.atleast_2d(x).shape[0], self.m)))[3]
    def Eval_Hessian(self, x, lam): return self._eval(1, x, lam)[4]

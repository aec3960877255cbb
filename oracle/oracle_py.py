"""ctypes bindings for the CPU oracle (oracle/liboracle.so) and, when present, the reference's
own L0 code (oracle/_ref/libref_l0.so).

TEST INFRASTRUCTURE ONLY.  Importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs; the product package restartsqp_b200 never imports it.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None
_REF = None

c_int_p = C.POINTER(C.c_int)
c_dbl_p = C.POINTER(C.c_double)


def _ip(a):
    return None if a is None else a.ctypes.data_as(c_int_p)


def _dp(a):
    return None if a is None else a.ctypes.data_as(c_dbl_p)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def build(force=False):
    """Compile liboracle.so (and _ref/libref_l0.so when /root/reference exists)."""
    so = os.path.join(_HERE, "liboracle.so")
    srcs = [os.path.join(_HERE, f) for f in ("oracle_l0.c", "oracle_qp.c", "oracle_batch.c", "oracle_sqp.c", "oracle.h", "Makefile")]
    stale = (not os.path.exists(so)) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs)
    if force or stale:
        subprocess.run(["make", "-C", _HERE, "liboracle.so"], check=True, capture_output=True)
    if os.path.isdir("/root/reference/src"):
        subprocess.run(["make", "-C", _HERE, "ref"], check=True, capture_output=True)


def lib():
    global _LIB
    if _LIB is None:
        build()
        L = C.CDLL(os.path.join(_HERE, "liboracle.so"))
        L.orc_one_norm.restype = C.c_double
        L.orc_inf_norm.restype = C.c_double
        L.orc_infea_measure_model.restype = C.c_double
        L.orc_qp_create.restype = C.c_void_p
        L.orc_qp_get_flops.restype = C.c_double
        L.orc_qp_get_flops.argtypes = [C.c_void_p]
        L.orc_qp_destroy.argtypes = [C.c_void_p]
        L.orc_qp_get_fell_back.argtypes = [C.c_void_p]
        L.orc_qp_get_max_free.argtypes = [C.c_void_p]
        _LIB = L
    return _LIB


def ref_lib():
    """The reference's own L0 code (None when oracle/_ref has not been built)."""
    global _REF
    if _REF is None:
        p = os.path.join(_HERE, "_ref", "libref_l0.so")
        if not os.path.exists(p):
            return None
        R = C.CDLL(p)
        for f in ("ref_one_norm", "ref_inf_norm", "ref_vector_one_norm", "ref_vector_inf_norm",
                  "ref_const_INF", "ref_const_sqrt_m_eps"):
            getattr(R, f).restype = C.c_double
        _REF = R
    return _REF


# ----------------------------------------------------------------------------- L0
def identity_info(n, m):
    """I_info_A_ of QPhandler::QPhandler, src/QPhandler.cpp:41-51."""
    return (_i32([1, 1]), _i32([n + 1, n + m + 1]), _i32([m, m]), _f64([1.0, -1.0]))


def assemble_A(nrow, ncol, row1, col1, val, iinfo):
    row1, col1, val = _i32(row1), _i32(col1), _f64(val)
    irow, jcol, size, ival = iinfo
    zJ = len(row1)
    z = zJ + int(size.sum())
    er, ec, ev = np.zeros(z, np.int32), np.zeros(z, np.int32), np.zeros(z)
    n = lib().orc_expand_A(zJ, _ip(row1), _ip(col1), _dp(val), len(size), _ip(irow), _ip(jcol), _ip(size),
                           _dp(ival), _ip(er), _ip(ec), _dp(ev))
    assert n == z
    return csc_from_entries(ncol, er, ec, ev)


def assemble_H(n, row1, col1, val, symmetric=True):
    row1, col1, val = _i32(row1), _i32(col1), _f64(val)
    zH = len(row1)
    er, ec, ev = np.zeros(2 * zH, np.int32), np.zeros(2 * zH, np.int32), np.zeros(2 * zH)
    z = lib().orc_expand_H(zH, _ip(row1), _ip(col1), _dp(val), int(symmetric), _ip(er), _ip(ec), _dp(ev))
    return csc_from_entries(n, er[:z].copy(), ec[:z].copy(), ev[:z].copy())


def csc_from_entries(ncol, er, ec, ev):
    z = len(er)
    colptr = np.zeros(ncol + 1, np.int32)
    rowidx, order, val = np.zeros(z, np.int32), np.zeros(z, np.int32), np.zeros(z)
    lib().orc_csc_from_entries(ncol, z, _ip(_i32(er)), _ip(_i32(ec)), _dp(_f64(ev)), _ip(colptr), _ip(rowidx),
                               _dp(val), _ip(order))
    return colptr, rowidx, val, order


def csr_from_entries(nrow, er, ec, ev):
    """Compressed-row branch of SpHbMat::setStructure (src/SpHbMat.cpp:238-250, 324-337): the same sort with the roles of
    row and column exchanged, key (row, col, counter).  Returns (rowptr, colidx, val, order)."""
    return csc_from_entries(nrow, ec, er, ev)


def assemble_A_csr(nrow, ncol, row1, col1, val, iinfo):
    """QOREInterface::set_A -> SpHbMat(nnz, nCon, nVar, isCompressedRow = true)::setStructure(rhs, I_info)
    (src/QOREInterface.cpp:643-650, :205)."""
    row1, col1, val = _i32(row1), _i32(col1), _f64(val)
    irow, jcol, size, ival = iinfo
    zJ = len(row1)
    z = zJ + int(size.sum())
    er, ec, ev = np.zeros(z, np.int32), np.zeros(z, np.int32), np.zeros(z)
    n = lib().orc_expand_A(zJ, _ip(row1), _ip(col1), _dp(val), len(size), _ip(irow), _ip(jcol), _ip(size),
                           _dp(ival), _ip(er), _ip(ec), _dp(ev))
    assert n == z
    return csr_from_entries(nrow, er, ec, ev)


def assemble_H_csr(n, row1, col1, val, symmetric=True):
    """QOREInterface::set_H -> SpHbMat(nVar, nVar, isCompressedRow = true)::setStructure(rhs)
    (src/QOREInterface.cpp:652-659, :212)."""
    row1, col1, val = _i32(row1), _i32(col1), _f64(val)
    zH = len(row1)
    er, ec, ev = np.zeros(2 * zH, np.int32), np.zeros(2 * zH, np.int32), np.zeros(2 * zH)
    z = lib().orc_expand_H(zH, _ip(row1), _ip(col1), _dp(val), int(symmetric), _ip(er), _ip(ec), _dp(ev))
    return csr_from_entries(n, er[:z].copy(), ec[:z].copy(), ev[:z].copy())


def setmatval_A(order, jac_val, csc_val):
    out = _f64(csc_val).copy()
    jac_val = _f64(jac_val)
    lib().orc_setmatval_A(len(jac_val), _ip(_i32(order)), _dp(jac_val), _dp(out))
    return out


def setmatval_H(row1, col1, order, h_val, csc_val, symmetric=True):
    out = _f64(csc_val).copy()
    h_val = _f64(h_val)
    lib().orc_setmatval_H(len(h_val), _ip(_i32(row1)), _ip(_i32(col1)), int(symmetric), _ip(_i32(order)),
                          _dp(h_val), _dp(out))
    return out


def csc_times(nrow, ncol, colptr, rowidx, val, x, transpose=False):
    colptr, rowidx, val, x = _i32(colptr), _i32(rowidx), _f64(val), _f64(x)
    y = np.zeros(ncol if transpose else nrow)
    f = lib().orc_csc_transposed_times if transpose else lib().orc_csc_times
    f(nrow, ncol, _ip(colptr), _ip(rowidx), _dp(val), _dp(x), _dp(y))
    return y


def qp_bounds(mode, n, m, delta, x_l, x_u, x_k, c_l, c_u, c_k, lb, ub, lbA, ubA):
    """In-place on lb, ub, lbA, ubA (float64 contiguous)."""
    lib().orc_qp_bounds(mode, n, m, C.c_double(delta), _dp(_f64(x_l)), _dp(_f64(x_u)), _dp(_f64(x_k)),
                        _dp(_f64(c_l)), _dp(_f64(c_u)), _dp(_f64(c_k)), _dp(lb), _dp(ub), _dp(lbA), _dp(ubA))


def translate_working_set(raw_b, raw_c, x, Ax, lb, ub, lbA, ubA):
    nV, nC = len(raw_b), len(raw_c)
    Wb, Wc = np.zeros(nV, np.int32), np.zeros(nC, np.int32)
    lib().orc_translate_working_set(nV, nC, _ip(_i32(raw_b)), _ip(_i32(raw_c)), _dp(_f64(x)), _dp(_f64(Ax)),
                                    _dp(_f64(lb)), _dp(_f64(ub)), _dp(_f64(lbA)), _dp(_f64(ubA)), _ip(Wb), _ip(Wc))
    return Wb, Wc


def kkt_residuals(nV, nC, A, H, g, lb, ub, lbA, ubA, x, y, Wb, Wc):
    """A, H = (colptr,rowidx,val) tuples; H may be None.  Returns (ok, out[5])."""
    Ap, Ai, Av = _i32(A[0]), _i32(A[1]), _f64(A[2])
    if H is not None:
        Hp, Hi, Hv = _i32(H[0]), _i32(H[1]), _f64(H[2])
    else:
        Hp = Hi = Hv = None
    out = np.zeros(5)
    ok = lib().orc_kkt_residuals(nV, nC, _ip(Ap), _ip(Ai), _dp(Av), _ip(Hp), _ip(Hi), _dp(Hv), _dp(_f64(g)),
                                 _dp(_f64(lb)), _dp(_f64(ub)), _dp(_f64(lbA)), _dp(_f64(ubA)), _dp(_f64(x)),
                                 _dp(_f64(y)), _ip(_i32(Wb)), _ip(_i32(Wc)), _dp(out))
    return bool(ok), out


# ----------------------------------------------------------------------------- row D
class QPOptions(C.Structure):
    _fields_ = [("max_iter", C.c_int), ("refactor_every", C.c_int), ("refine_steps", C.c_int),
                ("enable_flipping", C.c_int), ("enable_drift", C.c_int),
                ("enable_ramping", C.c_int)]


class OracleQP:
    """One QP instance with hot-start state (the oracle's stand-in for qpOASES::SQProblem)."""

    def __init__(self, nV, nC, max_iter=1000):
        self.nV, self.nC = nV, nC
        self.L = lib()
        self.h = C.c_void_p(self.L.orc_qp_create(nV, nC))
        self.opt = QPOptions()
        self.L.orc_qp_default_options(C.byref(self.opt))
        self.opt.max_iter = max_iter

    def __del__(self):
        if getattr(self, "h", None):
            self.L.orc_qp_destroy(self.h)
            self.h = None

    def init(self, H, g, A, lb, ub, lbA, ubA, is_lp=False):
        Ap, Ai, Av = _i32(A[0]), _i32(A[1]), _f64(A[2])
        if H is not None and not is_lp:
            Hp, Hi, Hv = _i32(H[0]), _i32(H[1]), _f64(H[2])
        else:
            Hp = Hi = Hv = None
        return self.L.orc_qp_init(self.h, C.byref(self.opt), _ip(Hp), _ip(Hi), _dp(Hv), _dp(_f64(g)), _ip(Ap),
                                  _ip(Ai), _dp(Av), _dp(_f64(lb)), _dp(_f64(ub)), _dp(_f64(lbA)), _dp(_f64(ubA)),
                                  int(is_lp))

    def hotstart(self, g, lb, ub, lbA, ubA):
        return self.L.orc_qp_hotstart(self.h, C.byref(self.opt), _dp(_f64(g)), _dp(_f64(lb)), _dp(_f64(ub)),
                                      _dp(_f64(lbA)), _dp(_f64(ubA)))

    def hotstart_matrices(self, H_val, A_val, g, lb, ub, lbA, ubA):
        hv = None if H_val is None else _f64(H_val)
        av = None if A_val is None else _f64(A_val)
        return self.L.orc_qp_hotstart_matrices(self.h, C.byref(self.opt), _dp(hv), _dp(av), _dp(_f64(g)),
                                               _dp(_f64(lb)), _dp(_f64(ub)), _dp(_f64(lbA)), _dp(_f64(ubA)))

    def reinit(self, H_val, A_val, g, lb, ub, lbA, ubA):
        """the matrix-status flip of optimizeQP (src/qpOASESInterface.cpp:202-207): init from the previous solution"""
        hv = None if H_val is None else _f64(H_val)
        av = None if A_val is None else _f64(A_val)
        return self.L.orc_qp_reinit(self.h, C.byref(self.opt), _dp(hv), _dp(av), _dp(_f64(g)),
                                    _dp(_f64(lb)), _dp(_f64(ub)), _dp(_f64(lbA)), _dp(_f64(ubA)))

    def solution(self):
        x, y = np.zeros(self.nV), np.zeros(self.nV + self.nC)
        obj, it = C.c_double(0), C.c_int(0)
        self.L.orc_qp_get_solution(self.h, _dp(x), _dp(y), C.byref(obj), C.byref(it))
        return x, y, obj.value, it.value

    def working_set(self):
        wb, wc = np.zeros(self.nV, np.int32), np.zeros(self.nC, np.int32)
        self.L.orc_qp_get_working_set(self.h, _ip(wb), _ip(wc))
        return wb, wc

    def flops(self):
        return self.L.orc_qp_get_flops(self.h)

    def handle_error(self, force_guess=False):
        """qpOASESInterface::handle_error after a solve that did not end OPTIMAL; returns (status, iterations added)."""
        it = C.c_int(0)
        st = self.L.orc_qp_handle_error(self.h, C.byref(self.opt), int(force_guess), C.byref(it))
        return st, it.value


def solve_batch(nV, nC, A, H, g, lb, ub, lbA, ubA, is_lp=False, max_iter=1000, nthreads=0, Avals=None, Hvals=None):
    """Cold-start solve of a batch on the host cores (OpenMP, one oracle object per thread).
    A, H = (colptr,rowidx,val[z]) shared pattern; Avals/Hvals optional [B][z].  Returns dict + threads used."""
    g = _f64(g)
    B = g.shape[0]
    lb, ub, lbA, ubA = _f64(lb), _f64(ub), _f64(lbA), _f64(ubA)
    Ap, Ai = _i32(A[0]), _i32(A[1])
    Av = _f64(A[2] if Avals is None else Avals)
    if H is not None and not is_lp:
        Hp, Hi = _i32(H[0]), _i32(H[1])
        Hv = _f64(H[2] if Hvals is None else Hvals)
    else:
        Hp = Hi = None
        Hv = np.zeros(1)
    x, y = np.empty((B, nV)), np.empty((B, nV + nC))
    obj, st, it = np.empty(B), np.empty(B, np.int32), np.empty(B, np.int32)
    used = lib().orc_qp_solve_batch(B, nV, nC, _ip(Hp), _ip(Hi), _dp(Hv), 0 if Hv.ndim == 1 else Hv.shape[1], _ip(Ap), _ip(Ai),
                                    _dp(Av), 0 if Av.ndim == 1 else Av.shape[1], _dp(g), _dp(lb), _dp(ub), _dp(lbA), _dp(ubA),
                                    int(is_lp), int(max_iter), _dp(x), _dp(y), _dp(obj), _ip(st), _ip(it), int(nthreads))
    return dict(x=x, y=y, obj=obj, status=st, iters=it, threads=used)


# ------------------------------------------------------------------ the caller: SQP outer loop (oracle_sqp.c)
class _SqpProblem(C.Structure):
    _fields_ = ([(k, C.c_int) for k in ("n", "m", "zJ", "zH")] +
                [(k, C.c_void_p) for k in ("J_row1", "J_col1", "H_row1", "H_col1", "x_l", "x_u", "c_l", "c_u", "fc", "all")] +
                [(k, C.c_int) for k in ("iter_max", "penalty_update", "penalty_iter_max", "qp_maxiter", "lp_maxiter")] +
                [(k, C.c_double) for k in ("eta_c", "eta_s", "eta_e", "gamma_c", "gamma_e", "delta", "delta_min", "delta_max", "tol",
                                           "penalty_update_tol", "rho", "rho_max", "increase_parm", "eps1", "eps1_change_parm", "eps2",
                                           "opt_prim_fea_tol", "opt_dual_fea_tol", "opt_compl_tol", "opt_stat_tol")] +
                [("second_order_correction", C.c_int)])


_GEN = None


def _gen_dir():
    """Where SqpOracle compiles model evaluators: one temporary directory per process, removed at exit."""
    global _GEN
    if _GEN is None:
        import atexit
        import shutil
        import tempfile
        _GEN = tempfile.mkdtemp(prefix="sqpb200_oracle_gen_")
        atexit.register(shutil.rmtree, _GEN, True)
    return _GEN


class SqpOracle:
    """CPU restatement of Algorithm::Optimize (oracle_sqp.c) for one model: `nlp` is a restartsqp_b200.nl_reader.AmplNLP (or
    anything with c_source(), the triplet patterns, bounds and start); its evaluator is generated as C and compiled with gcc
    (-ffp-contract=off) into a temporary directory of this process, so that a read-only checkout can run it."""

    def __init__(self, nlp, options):
        import hashlib
        src = nlp.c_source()
        gen = _gen_dir()
        tag = hashlib.sha1(src.encode()).hexdigest()[:16]
        so = os.path.join(gen, "nlp_%s_%s.so" % (getattr(nlp, "name", "model"), tag))
        if not os.path.exists(so):
            cfile = so[:-3] + ".c"
            with open(cfile, "w") as f:
                f.write(src)
            subprocess.run(["gcc", "-O1", "-fPIC", "-shared", "-ffp-contract=off", "-o", so, cfile, "-lm"], check=True, capture_output=True)
        self._nlp_lib = C.CDLL(so)
        self.evaluator = so  # the compiled evaluator (nlp_fc, nlp_all), for programs that load it themselves
        self.L = lib()
        info = nlp.Get_nlp_info()
        xl, xu, cl, cu = nlp.Get_bounds_info()
        self.n, self.m = info.nVar, info.nCon
        self._keep = [_i32(nlp.J_row1), _i32(nlp.J_col1), _i32(nlp.H_row1), _i32(nlp.H_col1), _f64(xl), _f64(xu), _f64(cl), _f64(cu)]
        P = self.P = _SqpProblem()
        P.n, P.m, P.zJ, P.zH = self.n, self.m, len(nlp.J_row1), len(nlp.H_row1)
        for k, a in zip(("J_row1", "J_col1", "H_row1", "H_col1", "x_l", "x_u", "c_l", "c_u"), self._keep):
            setattr(P, k, a.ctypes.data)
        P.fc = C.cast(self._nlp_lib.nlp_fc, C.c_void_p).value
        P.all = C.cast(self._nlp_lib.nlp_all, C.c_void_p).value
        o = options
        P.iter_max, P.penalty_update, P.penalty_iter_max, P.qp_maxiter, P.lp_maxiter = o.iter_max, int(o.penalty_update), o.penalty_iter_max, o.qp_maxiter, o.lp_maxiter
        for k in ("eta_c", "eta_s", "eta_e", "gamma_c", "gamma_e", "delta", "delta_min", "delta_max", "tol", "penalty_update_tol", "rho", "rho_max",
                  "increase_parm", "eps1", "eps1_change_parm", "eps2", "opt_prim_fea_tol", "opt_dual_fea_tol", "opt_compl_tol", "opt_stat_tol"):
            setattr(P, k, float(getattr(o, k)))
        P.second_order_correction = int(bool(getattr(o, "second_order_correction", False)))
        self.lam0 = _f64(nlp.Get_starting_point()[1])

    def solve_batch(self, x0, nthreads=0):
        x0 = _f64(np.atleast_2d(x0))
        B = x0.shape[0]
        x, f, kkt = np.empty((B, self.n)), np.empty(B), np.empty(B)
        ex, it, qi = np.empty(B, np.int32), np.empty(B, np.int32), np.empty(B, np.int64)
        used = self.L.orc_sqp_solve_batch(C.byref(self.P), B, _dp(x0), _dp(self.lam0), _dp(x), _dp(f), _ip(ex), _ip(it),
                                          qi.ctypes.data_as(C.c_void_p), _dp(kkt), int(nthreads))
        return dict(x=x, obj=f, exitflag=ex, iters=it.astype(np.int64), qp_iter=qi, KKT_error=kkt, threads=used)

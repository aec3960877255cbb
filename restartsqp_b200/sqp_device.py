"""Device-resident batched Sl1QP driver (SURVEY.md section 8f-1).

Same algorithm and same arithmetic as `sqp_driver.BatchedSQP` (the host mirror of src/Algorithm.cpp), but the iterates, the
trust-region radius, the penalty parameter, the flags and every intermediate stay on the GPU: the per-instance steps are phases
of one CUDA kernel (csrc/sqp_outer.cu, one thread per instance), the NLP is evaluated by the NVRTC-compiled kernels of
`DeviceNLP`, QP data is built by the qphandler kernels and the QP/LP solves take their instance mask from device memory.  The
host sequences launches and reads eight counters per outer iteration.  torch is used for device memory only.

optimize_async / solve_stream_async queue the same solves without any read-back: the loop is recorded once as a CUDA graph whose
branches are decided on the device (sqpb200_sqp_graph_*), so objects on different streams solve concurrently from one thread.

By default the backend's init / hotstart decision (src/qpOASESInterface.cpp:141-211, 817-833) is made per instance inside the solve
kernel, so every instance of the batch follows the reference's single-instance semantics: tests/test_gpu_sqp.py compares it bitwise
with the C oracle of the loop (oracle/oracle_sqp.c), and, with per_instance_modes=False, with BatchedSQP.
"""
import ctypes as C

import numpy as np

from . import _capi as capi
from .qp_handler import QPhandler
from .sqp_driver import SQPResult, classify_single_constraint
from .sqp_types import Exitflag, Options, QPType, SpTripletMat

PH_INIT = 13  # SQPB200_PH_INIT of include/sqpb200.h: initialization (src/Algorithm.cpp:438-472) after the evaluation at the start

_P, _D, _I = C.c_void_p, C.c_double, C.c_int


class SqpState(C.Structure):
    """sqpb200_sqp_state of include/sqpb200.h"""
    _fields_ = ([(k, _I) for k in ("B", "n", "m", "zJ", "zH", "iter_max", "penalty_update", "penalty_iter_max", "clear_flags")] +
                [(k, _D) for k in ("eta_c", "eta_s", "eta_e", "gamma_c", "gamma_e", "delta_min", "delta_max", "tol", "penalty_update_tol",
                                   "rho_max", "increase_parm", "eps1_change_parm", "eps2", "opt_prim_fea_tol", "opt_dual_fea_tol",
                                   "opt_compl_tol", "opt_stat_tol")] +
                [(k, _P) for k in ("J_row1", "J_col1", "x_l", "x_u", "c_l", "c_u", "bound_type", "cons_type",
                                   "x_k", "c_k", "f_k", "grad", "jac", "hess", "lam_c", "lam_x", "neg_lam",
                                   "delta", "rho", "eps1", "infea", "p_k", "x_trial", "c_trial", "f_trial", "infea_trial", "infea_model",
                                   "infea_model_tmp", "rho_trial", "infea_infty", "actual_red", "pred_red", "kkt_err",
                                   "g_new", "j_new", "h_new", "scratch", "exitflag", "iter", "pen_trial", "qp_iter",
                                   "active", "need", "go", "acc", "upd", "feasible_lp",
                                   "qp_x", "qp_y", "qp_obj", "qp_kkt", "lp_x", "qp_status", "qp_iters", "lp_status", "lp_iters", "counters",
                                   "H_row1", "H_col1", "soc_g", "soc_x", "soc_c", "p_tmp", "qp_obj_tmp", "qp_obj_soc", "norm_p", "rej",
                                   "qp_inst", "lp_inst")] +
                [(k, _D) for k in ("delta0", "rho0", "eps10")])


class SqpStream(C.Structure):
    """sqpb200_sqp_stream of include/sqpb200.h"""
    _fields_ = ([("N", C.c_longlong), ("refill_min", _I)] +
                [(k, _P) for k in ("x0_all", "lam_start", "x", "obj", "kkt_err", "rho", "delta", "exitflag", "iter", "qp_iter",
                                   "slot_id", "head", "refill")] +
                [("rounds", C.c_longlong)])


#: default refill_min of solve_stream as a fraction of the slot count (see solve_stream)
REFILL_MIN_FRACTION = 16


class PendingSQP:
    """A solve queued by optimize_async / solve_stream_async.  Its results are copied on the object's stream into tensors this object
    owns, so later calls on the object (reset, further solves) do not change them.  `event` is recorded behind the copies."""

    def __init__(self, out, event, keep=None):
        self._out, self.event, self._keep = out, event, keep

    def done(self):
        return self.event.query()

    def wait(self):
        self.event.synchronize()
        return self

    def result(self):
        self.wait()
        h = lambda k: self._out[k].cpu().numpy()
        return SQPResult(x=h("x"), obj=h("obj"), exitflag=h("exitflag"), iters=h("iter").astype(np.int64), qp_iter=h("qp_iter"),
                         KKT_error=h("kkt_err"), rho=h("rho"), delta=h("delta"))


class DeviceBatchedSQP:
    def __init__(self, nlp, x0=None, options: Options = None, device=0, per_instance_modes=True, stream=None):
        """per_instance_modes: the backend's init/hotstart decision is made per instance, as the reference does for its single
        instance (and as oracle/oracle_sqp.c does); False: per handle, which is what the numpy mirror BatchedSQP does.
        stream: a torch.cuda.Stream on which everything this object does runs (both handles, the NLP evaluations, the phases and its
        torch work); None: the default stream."""
        import torch
        if not hasattr(nlp, "eval_device"):
            raise TypeError("DeviceBatchedSQP needs a DeviceNLP (device-side evaluation)")
        self.torch, self.nlp_, self.L = torch, nlp, capi.lib()
        self.dev = torch.device("cuda", device)
        torch.cuda.set_device(self.dev)
        self.stream = stream
        self._sp = None if stream is None else C.c_void_p(stream.cuda_stream)
        self._graph = None
        with torch.cuda.stream(stream):
            self._init(nlp, x0, options, device, per_instance_modes)

    def _init(self, nlp, x0, options, device, per_instance_modes):
        torch = self.torch
        o = self.options_ = options if options is not None else Options()
        info = self.info = nlp.Get_nlp_info()
        n, m = self.nVar_, self.nCon_ = info.nVar, info.nCon
        x_start, lam_start = nlp.Get_starting_point()
        x0 = np.atleast_2d(np.asarray(x_start if x0 is None else x0, dtype=np.float64))
        B = self.batch = x0.shape[0]
        zJ, zH = len(nlp.J_row1), len(nlp.H_row1)
        self.myQP_ = QPhandler(info, QPType.QP, o, batch=B, device=device, refresh_ubA=True)  # src/Algorithm.cpp:561-562
        self.myLP_ = QPhandler(info, QPType.LP, o, batch=B, device=device, refresh_ubA=True)
        if self.stream is not None:
            for hd in (self.myQP_, self.myLP_):
                hd.solverInterface_.set_stream(self.stream.cuda_stream)
        f64 = lambda *shape: torch.zeros(shape, dtype=torch.float64, device=self.dev)
        u8 = lambda: torch.zeros(B, dtype=torch.uint8, device=self.dev)
        up = lambda a, dt=torch.float64: torch.as_tensor(np.ascontiguousarray(a), dtype=dt).to(self.dev)
        xl, xu, cl, cu = nlp.Get_bounds_info()
        # bounds, constraint classes and multipliers are the same for every instance: upload one row, replicate on the device
        rep = lambda a, dt=torch.float64: up(np.asarray(a).reshape(1, -1), dt).repeat(B, 1).contiguous()
        T = self.T = {}
        T["x_l"], T["x_u"], T["c_l"], T["c_u"] = rep(xl), rep(xu), rep(cl), rep(cu)
        T["bound_type"] = rep(classify_single_constraint(np.atleast_2d(xl), np.atleast_2d(xu)), torch.int32)
        T["cons_type"] = rep(classify_single_constraint(np.atleast_2d(cl).reshape(1, m), np.atleast_2d(cu).reshape(1, m)), torch.int32)
        T["J_row1"], T["J_col1"] = up(nlp.J_row1, torch.int32), up(nlp.J_col1, torch.int32)
        T["H_row1"], T["H_col1"] = up(nlp.H_row1, torch.int32), up(nlp.H_col1, torch.int32)
        T["x_k"] = torch.minimum(torch.maximum(up(x0), T["x_l"]), T["x_u"])  # shift_starting_point, src/SQPTNLP.cpp:140-153
        T["lam_c"] = rep(np.asarray(lam_start, dtype=np.float64).reshape(1, m))
        T["neg_lam"] = -T["lam_c"]
        for k, shp in (("c_k", (B, m)), ("f_k", (B,)), ("grad", (B, n)), ("jac", (B, zJ)), ("hess", (B, zH)), ("lam_x", (B, n)),
                       ("infea", (B,)), ("p_k", (B, n)), ("x_trial", (B, n)), ("c_trial", (B, m)), ("f_trial", (B,)), ("infea_trial", (B,)),
                       ("infea_model", (B,)), ("infea_model_tmp", (B,)), ("rho_trial", (B,)), ("infea_infty", (B,)), ("actual_red", (B,)),
                       ("pred_red", (B,)), ("g_new", (B, n)), ("j_new", (B, zJ)), ("h_new", (B, zH)), ("scratch", (B, max(n, 1))),
                       ("f_tmp", (B,)), ("c_tmp", (B, m)), ("soc_g", (B, n)), ("soc_x", (B, n)), ("soc_c", (B, m)), ("p_tmp", (B, n)),
                       ("qp_obj_tmp", (B,)), ("qp_obj_soc", (B,)), ("norm_p", (B,))):
            T[k] = f64(*shp)
        T["delta"] = torch.full((B,), float(o.delta), dtype=torch.float64, device=self.dev)
        T["rho"] = torch.full((B,), float(o.rho), dtype=torch.float64, device=self.dev)
        T["eps1"] = torch.full((B,), float(o.eps1), dtype=torch.float64, device=self.dev)
        T["kkt_err"] = torch.full((B,), float("inf"), dtype=torch.float64, device=self.dev)
        T["exitflag"] = torch.full((B,), int(Exitflag.UNKNOWN), dtype=torch.int32, device=self.dev)
        T["iter"] = torch.zeros(B, dtype=torch.int32, device=self.dev)
        T["pen_trial"] = torch.zeros(B, dtype=torch.int32, device=self.dev)
        T["qp_iter"] = torch.zeros(B, dtype=torch.int64, device=self.dev)
        for k in ("active", "need", "go", "acc", "upd", "feasible_lp", "rej"):
            T[k] = u8()
        T["counters"] = torch.zeros(8, dtype=torch.int32, device=self.dev)
        self.per_instance_modes = bool(per_instance_modes)
        if self.per_instance_modes:
            for k in ("qp_inst", "lp_inst"):
                T[k] = torch.zeros((B, 8), dtype=torch.int8, device=self.dev)
                T[k][:, 2:4] = -1  # matrix status undefined (get_Matrix_change_status, src/qpOASESInterface.cpp:817-833)
        # initialization(), src/Algorithm.cpp:438-472: f, c, grad, Jacobian, Hessian at the (shifted) start in one launch
        nlp.eval_device(1, B, T["x_k"], T["neg_lam"], T["f_k"], T["c_k"], T["grad"], T["jac"], T["hess"], stream=self.stream)
        S = self.S = SqpState()
        S.B, S.n, S.m, S.zJ, S.zH = B, n, m, zJ, zH
        S.iter_max, S.penalty_update, S.penalty_iter_max, S.clear_flags = o.iter_max, int(o.penalty_update), o.penalty_iter_max, 0
        for k in ("eta_c", "eta_s", "eta_e", "gamma_c", "gamma_e", "delta_min", "delta_max", "tol", "penalty_update_tol", "rho_max",
                  "increase_parm", "eps1_change_parm", "eps2", "opt_prim_fea_tol", "opt_dual_fea_tol", "opt_compl_tol", "opt_stat_tol"):
            setattr(S, k, float(getattr(o, k)))
        for k, _ in SqpState._fields_:
            if k in T:
                setattr(S, k, T[k].data_ptr())
        bq, bl = (C.c_void_p * 6)(), (C.c_void_p * 6)()
        self.L.sqpb200_device_buffers(self.myQP_.solverInterface_.h, bq)
        self.L.sqpb200_device_buffers(self.myLP_.solverInterface_.h, bl)
        S.qp_x, S.qp_y, S.qp_obj, S.qp_status, S.qp_iters, S.qp_kkt = bq[0], bq[1], bq[2], bq[3], bq[4], bq[5]
        S.lp_x, S.lp_status, S.lp_iters = bl[0], bl[3], bl[4]
        self._counters = (C.c_int * 8)()
        self.first_ = True
        self.launches = 0
        S.delta0, S.rho0, S.eps10 = float(o.delta), float(o.rho), float(o.eps1)
        self._lam_start = np.asarray(lam_start, dtype=np.float64).reshape(1, m)
        # infea_measure_ of the starting point (:472) and the per-instance algorithm state
        self._phase(PH_INIT)

    def reset(self, x0):
        """Algorithm::initialization (src/Algorithm.cpp:438-472) for a new batch of `batch` starting points on the same object:
        handles, device buffers and the compiled NLP are kept, so the per-batch cost is one upload, one evaluation and one
        state-reset launch."""
        B = self.batch
        x0 = np.ascontiguousarray(np.atleast_2d(np.asarray(x0, dtype=np.float64)))
        if x0.shape != (B, self.nVar_):
            raise ValueError("reset() needs %d starting points of dimension %d" % (B, self.nVar_))
        with self.torch.cuda.stream(self.stream):
            self._reset(x0)

    def _reset(self, x0):
        torch, T, B = self.torch, self.T, self.batch
        T["x_k"].copy_(torch.from_numpy(x0), non_blocking=False)
        torch.minimum(torch.maximum(T["x_k"], T["x_l"]), T["x_u"], out=T["x_k"])  # shift_starting_point
        T["lam_c"].copy_(torch.from_numpy(self._lam_start).to(self.dev).expand(B, -1))
        torch.neg(T["lam_c"], out=T["neg_lam"])
        self.nlp_.eval_device(1, B, T["x_k"], T["neg_lam"], T["f_k"], T["c_k"], T["grad"], T["jac"], T["hess"], stream=self.stream)
        self.S.clear_flags = 0
        self._phase(PH_INIT)
        for hd in (self.myQP_, self.myLP_):
            self.L.sqpb200_reset(hd.solverInterface_.h)
        self.first_ = True

    # ---- helpers
    def _phase(self, phase, read=False):
        rc = self.L.sqpb200_sqp_phase(C.byref(self.S), phase, self._counters if read else None, self._sp)
        if rc != 0:
            raise capi.SqpB200Error("sqpb200_sqp_phase(%d) failed: %d" % (phase, rc))
        self.launches += 1
        return list(self._counters) if read else None

    # ---- src/Algorithm.cpp:55-168
    def Optimize(self):
        """The whole loop runs behind one C call (sqpb200_sqp_optimize: no interpreter between the launches)."""
        T = self.T
        self._structures()
        first, nl = C.c_int(1 if self.first_ else 0), C.c_longlong(0)
        rc = self.L.sqpb200_sqp_optimize(C.byref(self.S), self.myQP_.solverInterface_.h, self.myLP_.solverInterface_.h, self.nlp_.h,
                                         int(bool(self.options_.second_order_correction)), 1, C.byref(first),
                                         C.c_void_p(T["f_tmp"].data_ptr()), C.c_void_p(T["c_tmp"].data_ptr()), C.byref(nl), self._sp)
        self._check(rc, "sqpb200_sqp_optimize")
        self.first_ = bool(first.value)
        self.launches += int(nl.value)
        return self._result()

    def solve_stream(self, x0_all, refill_min=None):
        """Algorithm::Optimize for N starting points x0_all[N][n] through the `batch` instances of this object used as slots: a slot
        whose instance has stopped takes the next starting point on the device, so no batch waits for its slowest instance and
        device memory stays that of `batch` instances (plus the N-row inputs and results).  Returns an SQPResult with N rows in input
        order; each row is bit for bit what one batch over all N gives.  Needs per-instance backend state machines.

        refill_min: a refill round (retire the stopped instances, refill their slots, one evaluation of the whole batch at the new
        starts) runs once at least this many occupied slots have stopped, or when no slot is active.  Default batch // 16 (at least 1):
        on the B200 (profiles/r3_sqp_stream.md) batch // 64, // 16 and // 4 were within 1 % of each other, while 1 (a refill round in
        nearly every iteration) was up to 30 % slower.  self.stream_rounds holds the number of
        refill rounds of the last call, the initial fill included.  The object serves reset() / Optimize() afterwards as before."""
        torch, T = self.torch, self.T
        O, D = self._stream_buffers("solve_stream", x0_all, refill_min)
        self._structures()
        first, nl = C.c_int(1 if self.first_ else 0), C.c_longlong(0)
        rc = self.L.sqpb200_sqp_optimize_stream(C.byref(self.S), self.myQP_.solverInterface_.h, self.myLP_.solverInterface_.h, self.nlp_.h,
                                                int(bool(self.options_.second_order_correction)), 1, C.byref(first),
                                                C.c_void_p(T["f_tmp"].data_ptr()), C.c_void_p(T["c_tmp"].data_ptr()), C.byref(D),
                                                C.byref(nl), self._sp)
        self._check(rc, "sqpb200_sqp_optimize_stream")
        self.first_ = bool(first.value)
        self.launches += int(nl.value)
        self.stream_rounds = int(D.rounds)
        torch.cuda.synchronize()
        h = lambda k: O[k].cpu().numpy()
        return SQPResult(x=h("x"), obj=h("obj"), exitflag=h("exitflag"), iters=h("iter").astype(np.int64), qp_iter=h("qp_iter"),
                         KKT_error=h("kkt_err"), rho=h("rho"), delta=h("delta"))

    def _need_per_instance_modes(self, what):
        if not self.per_instance_modes:
            raise ValueError("%s needs per_instance_modes=True: with handle-level modes the instances of a handle share its init / "
                             "hotstart decision (a refilled slot would inherit a hot start; the host reads the Update_* bits back)"
                             % what)

    def _stream_buffers(self, what, x0_all, refill_min):
        """inputs, results and slot bookkeeping of a streamed solve (device tensors, queued on the object's stream) and their
        sqpb200_sqp_stream descriptor"""
        torch, B, n = self.torch, self.batch, self.nVar_
        self._need_per_instance_modes(what)
        x0 = np.asarray(x0_all, dtype=np.float64)
        if x0.ndim != 2 or x0.shape[1] != n:
            raise ValueError("%s needs starting points of shape (N, %d), got %s" % (what, n, x0.shape))
        refill_min = max(1, B // REFILL_MIN_FRACTION) if refill_min is None else int(refill_min)
        if refill_min < 1:
            raise ValueError("refill_min must be at least 1")
        N = x0.shape[0]
        dev, f64, i32 = self.dev, torch.float64, torch.int32
        # pinned host copies: the upload is queued on the stream instead of waiting for it
        up = lambda a: torch.as_tensor(np.ascontiguousarray(a)).pin_memory().to(dev, non_blocking=True)
        with torch.cuda.stream(self.stream):
            O = dict(x0_all=up(x0), lam_start=up(self._lam_start.reshape(-1)), x=torch.empty((N, n), dtype=f64, device=dev),
                 obj=torch.empty(N, dtype=f64, device=dev), kkt_err=torch.empty(N, dtype=f64, device=dev),
                 rho=torch.empty(N, dtype=f64, device=dev), delta=torch.empty(N, dtype=f64, device=dev),
                 exitflag=torch.empty(N, dtype=i32, device=dev), iter=torch.empty(N, dtype=i32, device=dev),
                 qp_iter=torch.empty(N, dtype=torch.int64, device=dev), slot_id=torch.empty(B, dtype=torch.int64, device=dev),
                     head=torch.empty(1, dtype=torch.int64, device=dev), refill=torch.empty(B, dtype=torch.uint8, device=dev))
        D = SqpStream()
        D.N, D.refill_min = N, refill_min
        for k, t in O.items():
            setattr(D, k, t.data_ptr() if t.numel() else None)
        return O, D

    # ---- asynchronous solves (sqpb200_sqp_graph_*)
    def optimize_async(self):
        """Optimize() queued on the object's stream; returns a PendingSQP at once.  Bit for bit what Optimize() gives for the same
        sequence of calls on the object.  Needs per-instance backend state machines."""
        self._need_per_instance_modes("optimize_async")
        T = self.T
        self._launch_graph(None)
        with self.torch.cuda.stream(self.stream):
            out = {k: T[s].clone() for k, s in (("x", "x_k"), ("obj", "f_k"), ("exitflag", "exitflag"), ("iter", "iter"),
                                                 ("qp_iter", "qp_iter"), ("kkt_err", "kkt_err"), ("rho", "rho"), ("delta", "delta"))}
        return self._pending(out)

    def solve_stream_async(self, x0_all, refill_min=None):
        """solve_stream() queued on the object's stream; returns a PendingSQP at once (stream_rounds is not set).  Each call records
        its loop again: the descriptor of the call is part of the graph."""
        O, D = self._stream_buffers("solve_stream_async", x0_all, refill_min)
        self._launch_graph(D)
        return self._pending(O, keep=D)

    def _create_graph(self):
        """records the loop of Optimize (once per object; close() releases it)"""
        T = self.T
        self._structures()
        g = C.c_void_p()
        rc = self.L.sqpb200_sqp_graph_create(C.byref(self.S), self.myQP_.solverInterface_.h, self.myLP_.solverInterface_.h, self.nlp_.h,
                                             int(bool(self.options_.second_order_correction)), 1, C.c_void_p(T["f_tmp"].data_ptr()),
                                             C.c_void_p(T["c_tmp"].data_ptr()), self._sp, C.byref(g))
        self._check(rc, "sqpb200_sqp_graph_create")
        self._graph = g

    def _launch_graph(self, D):
        if self._graph is None:
            self._create_graph()
        first = C.c_int(1 if self.first_ else 0)
        rc = self.L.sqpb200_sqp_graph_launch(self._graph, C.byref(first), None if D is None else C.byref(D))
        self._check(rc, "sqpb200_sqp_graph_launch")
        self.first_ = bool(first.value)

    def _pending(self, out, keep=None):
        ev = self.torch.cuda.Event()
        ev.record(self.stream if self.stream is not None else self.torch.cuda.current_stream(self.dev))
        return PendingSQP(out, ev, keep)

    def _structures(self):
        """structures of both backends (first set_A / set_H call of setupQP / setupLP, values follow in the loop)"""
        if self.first_:
            self.myQP_.solverInterface_.set_A(SpTripletMat(self.nlp_.J_row1, self.nlp_.J_col1, None, self.nCon_, self.nVar_, False), self.myQP_.I_info_A_)
            self.myQP_.solverInterface_.set_H(SpTripletMat(self.nlp_.H_row1, self.nlp_.H_col1, None, self.nVar_, self.nVar_, True))
        if not self.myLP_.solverInterface_._A_set:
            self.myLP_.solverInterface_.set_A(SpTripletMat(self.nlp_.J_row1, self.nlp_.J_col1, None, self.nCon_, self.nVar_, False), self.myLP_.I_info_A_)

    def _check(self, rc, what):
        if rc != 0:
            raise capi.SqpB200Error("%s failed (%d): %s / %s" % (
                what, rc, self.L.sqpb200_last_error(self.myQP_.solverInterface_.h).decode(), self.L.sqpb200_last_error(self.myLP_.solverInterface_.h).decode()))

    def _result(self):
        T = self.T
        self.torch.cuda.synchronize()
        h = lambda k: T[k].cpu().numpy()
        return SQPResult(x=h("x_k"), obj=h("f_k"), exitflag=h("exitflag"), iters=h("iter").astype(np.int64), qp_iter=h("qp_iter"),
                         KKT_error=h("kkt_err"), rho=h("rho"), delta=h("delta"))

    def close(self):
        if self._graph is not None:
            self.L.sqpb200_sqp_graph_destroy(self._graph)
            self._graph = None
        self.myQP_.solverInterface_.close()
        self.myLP_.solverInterface_.close()

"""BASELINE.json config 1 / 3 on the GPU: HS071 through the batched SQP loop (mirror of src/Algorithm.cpp) with the
CUDA backend behind QPhandler, compared iterate-for-iterate with the same loop driven by the CPU oracle twin."""
import numpy as np
import pytest

import restartsqp_b200 as r
from restartsqp_b200.sqp_driver import BatchedSQP, HS071
from oracle_backend import OracleQPInterface

pytestmark = pytest.mark.gpu
X_STAR = np.array([1.0, 4.74299963, 3.82114998, 1.37940829])


def starts(B, seed=71000):
    rng = np.random.default_rng(seed)
    x0 = np.array([1.0, 5.0, 5.0, 1.0])
    s = np.clip(x0 * (1 + 0.1 * rng.standard_normal((B, 4))) + 0.1 * rng.standard_normal((B, 4)), 1.0, 5.0)
    s[0] = x0
    return s


def test_hs071_gpu_equals_oracle_driven_loop(gpu_lib):
    B = 16
    s = starts(B)
    opt_g, opt_o = r.Options(), r.Options()
    res_g = BatchedSQP(HS071(), x0=s, options=opt_g).Optimize()
    mk = lambda info, qt: r.QPhandler(info, qt, opt_o, batch=B, backend=OracleQPInterface(info, qt, opt_o, batch=B), refresh_ubA=True)
    res_o = BatchedSQP(HS071(), x0=s, options=opt_o, make_handler=mk).Optimize()
    assert (res_g.exitflag == res_o.exitflag).all() and (res_g.exitflag == int(r.Exitflag.OPTIMAL)).all()
    assert (res_g.iters == res_o.iters).all() and (res_g.qp_iter == res_o.qp_iter).all()
    assert np.abs(res_g.x - res_o.x).max() <= 1e-10  # the QP solutions are bit-identical, so are the iterates
    assert (res_g.rho == res_o.rho).all() and (res_g.delta == res_o.delta).all()
    assert np.abs(res_g.x - X_STAR).max() < 1e-4


def test_hs071_many_perturbed_starts(gpu_lib):
    B = 2000
    res = BatchedSQP(HS071(), x0=starts(B, seed=71001)).Optimize()
    ok = res.exitflag == int(r.Exitflag.OPTIMAL)
    assert ok.mean() > 0.99, np.unique(res.exitflag, return_counts=True)
    assert np.abs(res.x[ok] - X_STAR).max() < 1e-3
    assert np.abs(res.obj[ok] - 17.0140173).max() < 1e-3


HS_SAMPLE = ["hs001", "hs015", "hs035", "hs043", "hs056", "hs071", "hs076", "hs087", "hs100", "hs104", "hs113", "hs118", "hs119"]


@pytest.mark.parametrize("name", HS_SAMPLE)
def test_hs_suite_gpu_equals_oracle_driven_loop(gpu_lib, name):
    """BASELINE.json configs[2] (HS suite via the .nl reader, perturbed starts): the SQP loop on the CUDA backend takes
    the same path, iteration for iteration, as the same loop on the CPU oracle twin."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP
    from test_hs_suite import HS_DIR, perturbed_starts
    nlp = AmplNLP(os.path.join(HS_DIR, name + ".nl"))
    B = 6
    X = perturbed_starts(nlp, B, HS_SAMPLE.index(name))
    opt_g, opt_o = r.Options(iter_max=200), r.Options(iter_max=200)
    res_g = BatchedSQP(nlp, x0=X, options=opt_g).Optimize()
    mk = lambda info, qt: r.QPhandler(info, qt, opt_o, batch=B, backend=OracleQPInterface(info, qt, opt_o, batch=B), refresh_ubA=True)
    res_o = BatchedSQP(nlp, x0=X, options=opt_o, make_handler=mk).Optimize()
    assert (res_g.exitflag == res_o.exitflag).all(), (res_g.exitflag, res_o.exitflag)
    assert (res_g.iters == res_o.iters).all() and (res_g.qp_iter == res_o.qp_iter).all()
    assert np.abs(res_g.x - res_o.x).max() <= 1e-8 * max(1.0, np.abs(res_o.x).max())
    assert (res_g.exitflag[0] == int(r.Exitflag.OPTIMAL))


def test_failed_qp_is_dumped_and_replays(gpu_lib, tmp_path):
    """src/Algorithm.cpp:64-72: the QP that could not be solved is written as `<problem>qpdata.log` (QORE layout); the dump
    reads back (qp_dump) and replays through the data constructor of the backend to the same failure / to the oracle's answer."""
    import glob
    from restartsqp_b200 import qp_dump
    from oracle import oracle_py as orc
    import helpers as H
    opt = r.Options(qp_maxiter=1)  # every non-trivial QP stops in PERFORMINGHOMOTOPY
    alg = BatchedSQP(HS071(), x0=starts(5), options=opt, dump_dir=str(tmp_path), dump_max=2)
    res = alg.Optimize()
    assert (res.exitflag == int(r.Exitflag.QPERROR_PERFORMINGHOMOTOPY)).all()
    files = sorted(glob.glob(str(tmp_path / "QORE_*qpdata.log")))
    assert len(files) == 2
    q = qp_dump.read_qore_log(files[0])
    assert (q["nV"], q["nC"]) == (8, 2)
    s = qp_dump.replay(q, batch=3, options=opt)
    s.optimizeQP()
    assert (s.get_status() == int(r.Exitflag.QPERROR_PERFORMINGHOMOTOPY)).all()
    s.close()
    s = qp_dump.replay(files[0], batch=3)
    s.optimizeQP()
    p = dict(nV=8, nC=2, g=np.array(q["g"]), lb=np.array(q["lb"]), ub=np.array(q["ub"]), lbA=np.array(q["lbA"]), ubA=np.array(q["ubA"]))
    o = H.oracle_solve(orc, p, Acsc=(q["A_colptr"], q["A_rowidx"], np.array(q["A_val"])), Hcsc=(q["H_colptr"], q["H_rowidx"], np.array(q["H_val"])))
    assert (s.get_status() == o["status"]).all() and np.abs(s.get_optimal_solution()[1] - o["x"]).max() <= 1e-8 * max(1.0, np.abs(o["x"]).max())
    s.close()


@pytest.mark.parametrize("name", ["hs071", "hs043", "hs099", "hs100", "hs113", "hs085"])
def test_device_nlp_evaluator_matches_host_evaluator(gpu_lib, name):
    """The NVRTC-compiled evaluator (one thread per instance) against the numpy evaluator generated from the same DAG:
    + - * / are identical (--fmad=false); exp/log/sin/cos/pow differ by libm vs CUDA rounding only."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from test_hs_suite import HS_DIR, perturbed_starts
    host = AmplNLP(os.path.join(HS_DIR, name + ".nl"))
    dev = DeviceNLP(host)
    B = 257
    X = perturbed_starts(host, B, 3)
    lam = np.random.default_rng(5).standard_normal((B, host.m))
    f, c, g, J, Hh = dev.Eval_all(X, lam)
    f2, c2 = dev.Eval_f_c(X)
    rel = lambda a, b: float(np.abs(a - b).max() / max(1.0, np.abs(b).max())) if a.size else 0.0
    assert rel(f, host.Eval_f(X)) < 1e-12 and rel(c, host.Eval_constraints(X)) < 1e-12
    assert rel(g, host.Eval_gradient(X)) < 1e-12 and rel(J, host.Eval_Jacobian(X)) < 1e-12
    assert rel(Hh, host.Eval_Hessian(X, lam)) < 1e-11
    assert np.array_equal(f, f2) and np.array_equal(c, c2)
    assert dev.launch_count() == 2
    dev.close()


def test_sqp_with_device_evaluator(gpu_lib):
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from test_hs_suite import HS_DIR, perturbed_starts
    host = AmplNLP(os.path.join(HS_DIR, "hs071.nl"))
    dev = DeviceNLP(host)
    X = perturbed_starts(host, 512, 0)
    res_d = BatchedSQP(dev, x0=X).Optimize()
    res_h = BatchedSQP(host, x0=X).Optimize()
    assert (res_d.exitflag == int(r.Exitflag.OPTIMAL)).all() and (res_h.exitflag == res_d.exitflag).all()
    assert np.abs(res_d.x - res_h.x).max() < 1e-6 and np.abs(res_d.x - X_STAR).max() < 1e-4
    dev.close()


@pytest.mark.parametrize("name", ["hs071", "hs015", "hs043", "hs100", "hs113", "hs104", "hs099", "hs106"])
def test_device_resident_loop_equals_host_loop(gpu_lib, name):
    """csrc/sqp_outer.cu + DeviceBatchedSQP (iterates never leave the GPU) against BatchedSQP (numpy mirror of
    src/Algorithm.cpp) on the same NVRTC evaluator and the same QP backend: identical exit flags, outer and QP iteration
    counts, penalty parameters, radii and iterates."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    from test_hs_suite import HS_DIR, perturbed_starts
    host = AmplNLP(os.path.join(HS_DIR, name + ".nl"))
    dev = DeviceNLP(host)
    X = perturbed_starts(host, 200, 1)
    opt_h, opt_d = r.Options(iter_max=120), r.Options(iter_max=120)
    res_h = BatchedSQP(dev, x0=X, options=opt_h).Optimize()
    alg = DeviceBatchedSQP(dev, x0=X, options=opt_d, per_instance_modes=False)  # the numpy mirror decides per handle
    res_d = alg.Optimize()
    assert (res_d.exitflag == res_h.exitflag).all(), (np.unique(res_d.exitflag, return_counts=True), np.unique(res_h.exitflag, return_counts=True))
    assert (res_d.iters == res_h.iters).all() and (res_d.qp_iter == res_h.qp_iter).all()
    assert (res_d.rho == res_h.rho).all() and (res_d.delta == res_h.delta).all()
    fin = np.isfinite(res_h.x).all(axis=1)
    assert np.array_equal(res_d.x[fin], res_h.x[fin]) and np.array_equal(res_d.obj[fin], res_h.obj[fin])
    assert (res_d.exitflag[0] == int(r.Exitflag.OPTIMAL)) or name == "hs106"
    alg.close(); dev.close()


@pytest.mark.parametrize("name", ["hs006", "hs043", "hs100", "hs038"])
def test_device_loop_second_order_correction_equals_host_loop(gpu_lib, name):
    """The opt-in second-order correction (src/Algorithm.cpp:1140-1211) in the device-resident loop (PH_SOC_* phases) against the
    numpy mirror: identical exit flags, iteration counts and iterates on problems that reject steps."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    from test_hs_suite import HS_DIR, perturbed_starts
    dev = DeviceNLP(AmplNLP(os.path.join(HS_DIR, name + ".nl")))
    X = perturbed_starts(dev.host, 100, 2)
    res_h = BatchedSQP(dev, x0=X, options=r.Options(iter_max=120, second_order_correction=True)).Optimize()
    alg = DeviceBatchedSQP(dev, x0=X, options=r.Options(iter_max=120, second_order_correction=True), per_instance_modes=False)
    res_d = alg.Optimize()
    res_off = BatchedSQP(dev, x0=X, options=r.Options(iter_max=120)).Optimize()
    assert (res_d.exitflag == res_h.exitflag).all() and (res_d.iters == res_h.iters).all() and (res_d.qp_iter == res_h.qp_iter).all()
    assert (res_d.rho == res_h.rho).all() and (res_d.delta == res_h.delta).all()
    fin = np.isfinite(res_h.x).all(axis=1)
    assert np.array_equal(res_d.x[fin], res_h.x[fin])
    assert (res_h.qp_iter != res_off.qp_iter).any()  # the correction was actually taken somewhere
    alg.close(); dev.close()


@pytest.mark.parametrize("name", ["hs006", "hs043", "hs100"])
def test_device_loop_second_order_correction_equals_mirror_on_cpu_oracle(gpu_lib, name):
    """Second-order correction against a CPU path that shares no QP arithmetic with the kernels: the numpy mirror of
    Algorithm::Optimize with every QP / LP solved by the C oracle (tests/oracle_backend.py: the backend's state machine around
    oracle_qp.c), the NLP evaluated by the same NVRTC evaluator.  Handle-level init / hotstart decisions on both sides
    (per_instance_modes=False).  Identical exit flags, outer and QP iteration counts, penalty parameters, radii and iterates."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    from oracle_backend import OracleQPInterface
    from test_hs_suite import HS_DIR, perturbed_starts
    dev = DeviceNLP(AmplNLP(os.path.join(HS_DIR, name + ".nl")))
    B = 24
    X = perturbed_starts(dev.host, B, 2)
    opt = r.Options(iter_max=120, second_order_correction=True)
    mk = lambda info, qptype: r.QPhandler(info, qptype, opt, batch=B, backend=OracleQPInterface(info, qptype, opt, batch=B), refresh_ubA=True)
    res_h = BatchedSQP(dev, x0=X, options=opt, make_handler=mk).Optimize()
    alg = DeviceBatchedSQP(dev, x0=X, options=r.Options(iter_max=120, second_order_correction=True), per_instance_modes=False)
    res_d = alg.Optimize()
    res_off = DeviceBatchedSQP(dev, x0=X, options=r.Options(iter_max=120), per_instance_modes=False).Optimize()
    assert (res_d.exitflag == res_h.exitflag).all() and (res_d.iters == res_h.iters).all() and (res_d.qp_iter == res_h.qp_iter).all()
    assert (res_d.rho == res_h.rho).all() and (res_d.delta == res_h.delta).all()
    fin = np.isfinite(res_h.x).all(axis=1)
    assert np.array_equal(res_d.x[fin], res_h.x[fin])
    assert (res_d.qp_iter != res_off.qp_iter).any()  # the correction was actually taken somewhere
    alg.close(); dev.close()


@pytest.mark.parametrize("name", ["hs015", "hs043", "hs071", "hs083", "hs093", "hs106", "hs108", "hs113", "hs116", "hs118"])
def test_device_loop_per_instance_modes_equal_the_c_oracle(gpu_lib, name):
    """Default mode of DeviceBatchedSQP: the backend's init/hotstart state machine runs per instance inside the solve kernel, i.e.
    the reference's semantics for every instance of the batch.  Against oracle/oracle_sqp.c (one independent solve per instance)
    on problems evaluated with + - * and squares only, where the NVRTC and the gcc evaluators agree bitwise: identical exit flags, outer and QP iteration
    counts and iterates, although the instances of the batch accept and reject steps at different iterations."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    from oracle import oracle_py as orc
    from test_hs_suite import HS_DIR, perturbed_starts
    host = AmplNLP(os.path.join(HS_DIR, name + ".nl"))
    dev = DeviceNLP(host)
    X = perturbed_starts(host, 96, 4)
    alg = DeviceBatchedSQP(dev, x0=X, options=r.Options(iter_max=150))
    res_d = alg.Optimize()
    res_c = orc.SqpOracle(host, r.Options(iter_max=150)).solve_batch(X)
    assert (res_d.exitflag == res_c["exitflag"]).all(), (res_d.exitflag, res_c["exitflag"])
    assert (res_d.iters == res_c["iters"]).all() and (res_d.qp_iter == res_c["qp_iter"]).all()
    fin = np.isfinite(res_c["x"]).all(axis=1)
    assert np.array_equal(res_d.x[fin], res_c["x"][fin]) and np.array_equal(res_d.obj[fin], res_c["obj"][fin])
    alg.close(); dev.close()


@pytest.mark.parametrize("name", ["hs015", "hs043", "hs113"])
def test_device_loop_second_order_correction_equals_the_c_oracle(gpu_lib, name):
    """The same with the opt-in second-order correction (src/Algorithm.cpp:1140-1211) on both sides: per-instance state machines
    in the solve kernels against one independent solve per instance in oracle/oracle_sqp.c."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    from oracle import oracle_py as orc
    from test_hs_suite import HS_DIR, perturbed_starts
    host = AmplNLP(os.path.join(HS_DIR, name + ".nl"))
    dev = DeviceNLP(host)
    X = perturbed_starts(host, 96, 4)
    alg = DeviceBatchedSQP(dev, x0=X, options=r.Options(iter_max=150, second_order_correction=True))
    res_d = alg.Optimize()
    res_c = orc.SqpOracle(host, r.Options(iter_max=150, second_order_correction=True)).solve_batch(X)
    res_off = orc.SqpOracle(host, r.Options(iter_max=150)).solve_batch(X)
    assert (res_d.exitflag == res_c["exitflag"]).all(), (res_d.exitflag, res_c["exitflag"])
    assert (res_d.iters == res_c["iters"]).all() and (res_d.qp_iter == res_c["qp_iter"]).all()
    fin = np.isfinite(res_c["x"]).all(axis=1)
    assert np.array_equal(res_d.x[fin], res_c["x"][fin]) and np.array_equal(res_d.obj[fin], res_c["obj"][fin])
    assert (res_c["qp_iter"] != res_off["qp_iter"]).any()  # the correction was taken somewhere
    alg.close(); dev.close()


def test_device_loop_qp_unchanged_guard(gpu_lib):
    """setupQP's QP_UNCHANGED guard (src/Algorithm.cpp:651-670) in the device loop (PH_FLAGS): an instance whose QP data did not
    change since its last solve ends with Exitflag.QP_UNCHANGED instead of re-solving the same QP until iter_max.  hs105 gets
    there after one iteration from most perturbed starts; against the C oracle instance by instance (exp / log are evaluated by
    NVRTC and by libm: agreement on nearly all starts, not bit for bit)."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    from oracle import oracle_py as orc
    from test_hs_suite import HS_DIR, perturbed_starts
    host = AmplNLP(os.path.join(HS_DIR, "hs105.nl"))
    dev = DeviceNLP(host)
    X = perturbed_starts(host, 64, 1)
    U = int(r.Exitflag.QP_UNCHANGED)
    for pim in (True, False):
        alg = DeviceBatchedSQP(dev, x0=X, options=r.Options(iter_max=50), per_instance_modes=pim)
        res_d = alg.Optimize()
        alg.close()
        assert (res_d.exitflag == U).sum() >= 32 and (res_d.iters[res_d.exitflag == U] < 50).all()
        if pim:
            res_c = orc.SqpOracle(host, r.Options(iter_max=50)).solve_batch(X)
            same = (res_d.exitflag == res_c["exitflag"]) & (res_d.iters == res_c["iters"])
            assert same.mean() >= 0.9, same.mean()
    dev.close()


def test_reset_serves_batch_after_batch(gpu_lib):
    """DeviceBatchedSQP.reset(x0): the same object (handles, buffers, compiled NLP) re-initialised for a new batch gives bit for bit
    what a freshly constructed object gives, with and without per-instance backend state machines."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    from test_hs_suite import HS_DIR, perturbed_starts
    dev = DeviceNLP(AmplNLP(os.path.join(HS_DIR, "hs100.nl")))
    X1, X2 = perturbed_starts(dev.host, 96, 11), perturbed_starts(dev.host, 96, 12)
    for pim in (True, False):
        a = DeviceBatchedSQP(dev, x0=X1, options=r.Options(iter_max=120), per_instance_modes=pim)
        a.Optimize()
        a.reset(X2)
        r_reused = a.Optimize()
        b = DeviceBatchedSQP(dev, x0=X2, options=r.Options(iter_max=120), per_instance_modes=pim)
        r_fresh = b.Optimize()
        assert (r_reused.exitflag == r_fresh.exitflag).all() and (r_reused.iters == r_fresh.iters).all() and (r_reused.qp_iter == r_fresh.qp_iter).all()
        assert np.array_equal(r_reused.x, r_fresh.x, equal_nan=True) and np.array_equal(r_reused.obj, r_fresh.obj, equal_nan=True)
        a.close(); b.close()
    dev.close()


def test_device_evaluator_large_dag_and_imported_function(gpu_lib):
    """hs025 (9.8 k-node DAG: compiled in pieces, math functions through __noinline__ wrappers) and hs068 (imported function
    `myerf` = the normal distribution function) on the NVRTC evaluator against the numpy evaluator of the same DAG; hs068 through the
    device-resident SQP loop to the tabulated optimum f* = -0.920425."""
    import os
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    from test_hs_suite import HS_DIR, perturbed_starts
    rel = lambda a, b: float(np.abs(a - b).max() / max(1.0, np.abs(b).max())) if a.size else 0.0
    for name in ("hs025", "hs068"):
        host = AmplNLP(os.path.join(HS_DIR, name + ".nl"))
        dev = DeviceNLP(host)
        X = perturbed_starts(host, 64, 3)
        lam = np.random.default_rng(5).standard_normal((64, host.m))
        f, c, g, J, Hh = dev.Eval_all(X, lam)
        fin = np.isfinite(host.Eval_Hessian(X, lam)).all(axis=1) & np.isfinite(Hh).all(axis=1)
        assert fin.sum() > 32
        assert rel(f[fin], host.Eval_f(X)[fin]) < 1e-11 and rel(c[fin], host.Eval_constraints(X)[fin]) < 1e-11
        assert rel(g[fin], host.Eval_gradient(X)[fin]) < 1e-10 and rel(J[fin], host.Eval_Jacobian(X)[fin]) < 1e-10
        assert rel(Hh[fin], host.Eval_Hessian(X, lam)[fin]) < 1e-9
        if name == "hs068":
            alg = DeviceBatchedSQP(dev, x0=X[:16], options=r.Options(iter_max=300))
            res = alg.Optimize()
            ok = res.exitflag == int(r.Exitflag.OPTIMAL)
            # the reference's optimality test stops at a stationarity residual of 1e-4 and the objective is flat near the optimum
            assert ok.sum() >= 8 and np.abs(res.obj[ok] + 0.920425).max() < 5e-3 and np.abs(res.obj[ok] + 0.920425).min() < 1e-4
            alg.close()
        dev.close()

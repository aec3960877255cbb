"""Streamed solves (sqpb200_sqp_optimize_stream, DeviceBatchedSQP.solve_stream, BatchedAlgorithm::OptimizeStream): N starting
points through B < N device slots, a stopped slot refilled with the next starting point on the device.  Every instance must follow
the trajectory it follows in one batch over all N, bit for bit, whichever slot it lands in and whenever."""
import functools
import os
import subprocess

import numpy as np
import pytest

import restartsqp_b200 as r
from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP, write_model_file
from restartsqp_b200.sqp_device import DeviceBatchedSQP
from test_hs_suite import HS_DIR, perturbed_starts

pytestmark = pytest.mark.gpu
FIELDS = ("exitflag", "iters", "qp_iter", "x", "obj", "rho", "delta", "KKT_error")


def assert_same(a, b):
    for k in FIELDS:
        u, v = getattr(a, k), getattr(b, k)
        assert np.array_equal(u, v, equal_nan=True), (k, u.shape, v.shape)


def device_nlp(name):
    return DeviceNLP(AmplNLP(os.path.join(HS_DIR, name + ".nl")))


def streamed(dev, X, slots, options, refill_min=None):
    """solve_stream on an object of `slots` instances (its own starting points are irrelevant: every slot is refilled)"""
    alg = DeviceBatchedSQP(dev, x0=perturbed_starts(dev.host, slots, 99), options=options)
    res = alg.solve_stream(X, refill_min=refill_min)
    rounds = alg.stream_rounds
    alg.close()
    return res, rounds


def one_batch(dev, X, options):
    alg = DeviceBatchedSQP(dev, x0=X, options=options)
    res = alg.Optimize()
    alg.close()
    return res


@pytest.mark.parametrize("name,soc", [("hs071", False), ("hs100", False), ("hs116", False), ("hs036", False), ("hs043", True)])
def test_stream_equals_one_batch(gpu_lib, name, soc):
    dev = device_nlp(name)
    X = perturbed_starts(dev.host, 1000, 21)
    opt = lambda: r.Options(iter_max=120, second_order_correction=soc)
    ref = one_batch(dev, X, opt())
    for slots in (64, 128):
        for refill_min in (1, slots // 4):
            res, rounds = streamed(dev, X, slots, opt(), refill_min)
            assert_same(res, ref)
            assert rounds >= -(-1000 // slots)  # at least enough rounds to hand out every starting point
    dev.close()


@pytest.mark.parametrize("N,slots", [(40, 64), (64, 64), (257, 64)])
def test_stream_sizes(gpu_lib, N, slots):
    """fewer starting points than slots (some slots never hold an instance), exactly one batch, and N not a multiple of the slots"""
    dev = device_nlp("hs071")
    X = perturbed_starts(dev.host, N, 22)
    ref = one_batch(dev, X, r.Options(iter_max=120))
    res, rounds = streamed(dev, X, slots, r.Options(iter_max=120))
    assert_same(res, ref)
    assert res.x.shape == (N, 4) and (rounds == 1) == (N <= slots)
    dev.close()


def test_stream_is_repeatable(gpu_lib):
    """slot assignment is not deterministic (atomicAdd), results are: two runs of the same stream, on one object and on another"""
    dev = device_nlp("hs100")
    X = perturbed_starts(dev.host, 500, 23)
    alg = DeviceBatchedSQP(dev, x0=X[:48], options=r.Options(iter_max=120))
    a = alg.solve_stream(X, refill_min=1)
    b = alg.solve_stream(X, refill_min=1)
    alg.close()
    c, _ = streamed(dev, X, 48, r.Options(iter_max=120), 1)
    assert_same(a, b)
    assert_same(a, c)
    dev.close()


@pytest.mark.parametrize("name", ["hs015", "hs043", "hs113", "hs118"])
def test_stream_equals_the_c_oracle(gpu_lib, name):
    """polynomial models, where the NVRTC and the gcc evaluators agree bitwise: against oracle/oracle_sqp.c (one independent solve
    per instance) with fewer slots than instances"""
    from oracle import oracle_py as orc
    dev = device_nlp(name)
    X = perturbed_starts(dev.host, 96, 4)
    res, _ = streamed(dev, X, 32, r.Options(iter_max=150), 4)
    res_c = orc.SqpOracle(dev.host, r.Options(iter_max=150)).solve_batch(X)
    assert (res.exitflag == res_c["exitflag"]).all(), (res.exitflag, res_c["exitflag"])
    assert (res.iters == res_c["iters"]).all() and (res.qp_iter == res_c["qp_iter"]).all()
    fin = np.isfinite(res_c["x"]).all(axis=1)
    assert np.array_equal(res.x[fin], res_c["x"][fin]) and np.array_equal(res.obj[fin], res_c["obj"][fin])
    dev.close()


def test_stream_retires_exceed_max_iter(gpu_lib):
    """iter_max = 5: instances that reach it leave their slot labelled EXCEED_MAX_ITER, as PH_FINAL labels them in one batch"""
    dev = device_nlp("hs100")
    X = perturbed_starts(dev.host, 300, 24)
    ref = one_batch(dev, X, r.Options(iter_max=5))
    res, _ = streamed(dev, X, 32, r.Options(iter_max=5), 1)
    assert_same(res, ref)
    assert (res.exitflag == int(r.Exitflag.EXCEED_MAX_ITER)).any()
    dev.close()


def test_stream_retires_qp_unchanged(gpu_lib):
    """hs105: instances that PH_FLAGS ends with QP_UNCHANGED are retired with that flag"""
    dev = device_nlp("hs105")
    X = perturbed_starts(dev.host, 200, 1)
    ref = one_batch(dev, X, r.Options(iter_max=50))
    res, _ = streamed(dev, X, 32, r.Options(iter_max=50), 1)
    assert_same(res, ref)
    assert (res.exitflag == int(r.Exitflag.QP_UNCHANGED)).any()
    dev.close()


def test_object_serves_batches_after_a_stream(gpu_lib):
    """after solve_stream, reset(X) + Optimize() on the same object gives what a fresh object gives"""
    dev = device_nlp("hs100")
    X1, X2 = perturbed_starts(dev.host, 300, 25), perturbed_starts(dev.host, 64, 26)
    a = DeviceBatchedSQP(dev, x0=X2, options=r.Options(iter_max=120))
    a.solve_stream(X1)
    a.reset(X2)
    reused = a.Optimize()
    assert_same(reused, one_batch(dev, X2, r.Options(iter_max=120)))
    a.close()
    dev.close()


def test_stream_rejects_what_it_cannot_do(gpu_lib):
    dev = device_nlp("hs071")
    X = perturbed_starts(dev.host, 16, 27)
    a = DeviceBatchedSQP(dev, x0=X[:8], per_instance_modes=False)
    with pytest.raises(ValueError):
        a.solve_stream(X)
    a.close()
    a = DeviceBatchedSQP(dev, x0=X[:8])
    for bad in (X[:, :3], X[0], X.reshape(1, 16, 4)):
        with pytest.raises(ValueError):
            a.solve_stream(bad)
    with pytest.raises(ValueError):
        a.solve_stream(X, refill_min=0)
    a.close()
    dev.close()


def test_stream_on_the_cluster_kernel(gpu_lib, monkeypatch):
    """both handles forced onto the one-QP-per-cluster kernel (team_size 1024), whose hot-start data stays in a global slice per
    slot: a refilled slot starts cold there too"""
    import restartsqp_b200.sqp_device as sd
    monkeypatch.setattr(sd, "QPhandler", functools.partial(sd.QPhandler, team_size=1024))
    dev = device_nlp("hs071")
    X = perturbed_starts(dev.host, 48, 28)
    alg = DeviceBatchedSQP(dev, x0=X, options=r.Options(iter_max=60))
    ref = alg.Optimize()
    assert alg.myQP_.solverInterface_.solve_config()["team_size"] == 1024
    alg.close()
    res, rounds = streamed(dev, X, 16, r.Options(iter_max=60), 1)
    assert_same(res, ref)
    assert rounds >= 3  # 48 starts through 16 slots: every slot is refilled at least twice
    dev.close()


BIN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "restartsqp_b200", "lib", "batched_sqp")


@pytest.mark.parametrize("name,soc", [("hs071", False), ("hs043", True)])
def test_cpp_driver_slots_output_identical(gpu_lib, tmp_path, name, soc):
    """batched_sqp --slots 64 (BatchedAlgorithm::OptimizeStream): the instance lines are byte-identical to the one-batch run"""
    host = AmplNLP(os.path.join(HS_DIR, name + ".nl"))
    path = str(tmp_path / (name + ".model"))
    write_model_file(host, path, perturbed_starts(host, 300, 29))
    flags = ["--iter-max", "120"] + (["--soc"] if soc else [])
    run = lambda *extra: subprocess.run([BIN, path, *flags, *extra], capture_output=True, text=True, timeout=300)
    a, b = run(), run("--slots", "64")
    assert a.returncode == 0 and b.returncode == 0, a.stderr[-2000:] + b.stderr[-2000:]
    la, lb = a.stdout.splitlines(), b.stdout.splitlines()
    assert len(la) == 301 and la[:-1] == lb[:-1]
    summary = lb[-1].split()
    assert summary[summary.index("slots") + 1] == "64" and int(summary[summary.index("refill_rounds") + 1]) >= 5

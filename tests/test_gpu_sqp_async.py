"""Asynchronous device SQP solves (sqpb200_sqp_graph_*, DeviceBatchedSQP.optimize_async / solve_stream_async): the outer loop recorded
as a CUDA graph with device-side branching.  Every result must equal, bit for bit, what the synchronous call gives for the same
sequence of calls on an object."""
import ctypes as C
import functools

import numpy as np
import pytest

import restartsqp_b200 as r
from restartsqp_b200.sqp_device import DeviceBatchedSQP
from test_gpu_sqp_stream import assert_same, device_nlp, one_batch, streamed
from test_hs_suite import perturbed_starts

pytestmark = pytest.mark.gpu


def async_batch(dev, X, options, **kw):
    alg = DeviceBatchedSQP(dev, x0=X, options=options, **kw)
    res = alg.optimize_async().result()
    alg.close()
    return res


@pytest.mark.parametrize("name,soc", [("hs071", False), ("hs100", False), ("hs116", False), ("hs036", False), ("hs043", True),
                                      ("hs038", False), ("hs108", False), ("hs105", False)])
def test_optimize_async_equals_optimize(gpu_lib, name, soc):
    """hs038: m = 0; hs108: QP failures; hs105: QP_UNCHANGED"""
    dev = device_nlp(name)
    X = perturbed_starts(dev.host, 500, 31)
    opt = lambda: r.Options(iter_max=120, second_order_correction=soc)
    assert_same(async_batch(dev, X, opt()), one_batch(dev, X, opt()))
    dev.close()


def test_optimize_async_exceed_max_iter(gpu_lib):
    dev = device_nlp("hs100")
    X = perturbed_starts(dev.host, 300, 32)
    res = async_batch(dev, X, r.Options(iter_max=5))
    assert_same(res, one_batch(dev, X, r.Options(iter_max=5)))
    assert (res.exitflag == int(r.Exitflag.EXCEED_MAX_ITER)).any()
    dev.close()


def test_optimize_async_on_the_cluster_kernel(gpu_lib, monkeypatch):
    import restartsqp_b200.sqp_device as sd
    monkeypatch.setattr(sd, "QPhandler", functools.partial(sd.QPhandler, team_size=1024))
    dev = device_nlp("hs071")
    X = perturbed_starts(dev.host, 48, 33)
    alg = DeviceBatchedSQP(dev, x0=X, options=r.Options(iter_max=60))
    res = alg.optimize_async().result()
    assert alg.myQP_.solverInterface_.solve_config()["team_size"] == 1024
    alg.close()
    assert_same(res, one_batch(dev, X, r.Options(iter_max=60)))
    dev.close()


def test_call_sequence_equals_synchronous(gpu_lib):
    """construct -> solve -> reset -> solve -> solve (no reset: first = 0), asynchronous against synchronous"""
    dev = device_nlp("hs100")
    X1, X2 = perturbed_starts(dev.host, 256, 34), perturbed_starts(dev.host, 256, 35)
    out = {}
    for mode in ("sync", "async"):
        alg = DeviceBatchedSQP(dev, x0=X1, options=r.Options(iter_max=60))
        run = alg.Optimize if mode == "sync" else (lambda: alg.optimize_async().result())
        a = run()
        alg.reset(X2)
        b = run()
        c = run()
        alg.close()
        out[mode] = (a, b, c)
    for u, v in zip(out["sync"], out["async"]):
        assert_same(u, v)
    dev.close()


@pytest.mark.parametrize("N", [40, 64, 300])
def test_solve_stream_async_equals_solve_stream(gpu_lib, N):
    """below, at and above the slot count, refill_min 1 and slots / 4, on one object (the streamed graph is recorded per call)"""
    dev = device_nlp("hs071")
    X = perturbed_starts(dev.host, N, 36)
    alg = DeviceBatchedSQP(dev, x0=perturbed_starts(dev.host, 64, 99), options=r.Options(iter_max=120))
    for refill_min in (1, 16):
        ref, _ = streamed(dev, X, 64, r.Options(iter_max=120), refill_min)
        assert_same(alg.solve_stream_async(X, refill_min=refill_min).result(), ref)
    alg.close()
    dev.close()


def test_solve_stream_async_with_soc(gpu_lib):
    dev = device_nlp("hs043")
    X = perturbed_starts(dev.host, 300, 37)
    opt = lambda: r.Options(iter_max=120, second_order_correction=True)
    ref, _ = streamed(dev, X, 64, opt(), 16)
    alg = DeviceBatchedSQP(dev, x0=X[:64], options=opt())
    assert_same(alg.solve_stream_async(X, refill_min=16).result(), ref)
    alg.close()
    dev.close()


def test_models_run_concurrently_from_one_thread(gpu_lib):
    """six models, each object on its own stream, all queued before any wait; each equals its solo synchronous run"""
    import torch
    names = ["hs071", "hs100", "hs036", "hs043", "hs108", "hs113"]
    devs = {k: device_nlp(k) for k in names}
    X = {k: perturbed_starts(devs[k].host, 400, 38) for k in names}
    algs = [DeviceBatchedSQP(devs[k], x0=X[k], options=r.Options(iter_max=100), stream=torch.cuda.Stream()) for k in names]
    pending = [a.optimize_async() for a in algs]
    results = [p.result() for p in pending]
    for a in algs:
        a.close()
    for k, res in zip(names, results):
        assert_same(res, one_batch(devs[k], X[k], r.Options(iter_max=100)))
        devs[k].close()


def test_launch_does_not_block(gpu_lib):
    """the call returns while the stream is still busy with earlier work; the result is right once it is waited for"""
    import torch
    dev = device_nlp("hs071")
    X1, X2 = perturbed_starts(dev.host, 256, 39), perturbed_starts(dev.host, 256, 40)
    s = torch.cuda.Stream()
    alg = DeviceBatchedSQP(dev, x0=X1, options=r.Options(iter_max=100), stream=s)
    alg.optimize_async().wait()  # records the graph
    alg.reset(X2)
    with torch.cuda.stream(s):
        torch.cuda._sleep(2_000_000_000)  # about a second
    p = alg.optimize_async()
    busy = not s.query()
    res = p.result()
    alg.close()
    assert busy and p.done()
    assert_same(res, one_batch(dev, X2, r.Options(iter_max=100)))
    dev.close()


def test_pending_result_survives_reset(gpu_lib):
    dev = device_nlp("hs100")
    X1, X2 = perturbed_starts(dev.host, 256, 41), perturbed_starts(dev.host, 256, 42)
    alg = DeviceBatchedSQP(dev, x0=X1, options=r.Options(iter_max=60))
    p = alg.optimize_async()
    alg.reset(X2)
    q = alg.optimize_async()
    a, b = p.result(), q.result()
    alg.close()
    assert_same(a, one_batch(dev, X1, r.Options(iter_max=60)))
    assert_same(b, one_batch(dev, X2, r.Options(iter_max=60)))
    dev.close()


def test_async_rejects_handle_level_modes(gpu_lib):
    dev = device_nlp("hs071")
    X = perturbed_starts(dev.host, 16, 43)
    a = DeviceBatchedSQP(dev, x0=X[:8], per_instance_modes=False)
    with pytest.raises(ValueError):
        a.optimize_async()
    with pytest.raises(ValueError):
        a.solve_stream_async(X)
    a._structures()
    g = C.c_void_p()
    T = a.T
    rc = gpu_lib.sqpb200_sqp_graph_create(C.byref(a.S), a.myQP_.solverInterface_.h, a.myLP_.solverInterface_.h, dev.h, 0, 1,
                                          C.c_void_p(T["f_tmp"].data_ptr()), C.c_void_p(T["c_tmp"].data_ptr()), None, C.byref(g))
    assert rc == -1 and not g.value  # SQPB200_ERR_INVALID: st->qp_inst == NULL
    a.close()
    dev.close()

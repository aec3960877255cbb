"""One HS problem x B perturbed starts through the device-resident SQP loop on one reused object: time per batch, SQP / QP iteration
statistics (mean, max) and launch count."""
import sys, os, time, numpy as np
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, R); sys.path.insert(0, R + "/tests")
from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
from restartsqp_b200.sqp_device import DeviceBatchedSQP
Bs = int(sys.argv[2]) if len(sys.argv) > 2 else 10000
for name in sys.argv[1].split(","):
    host = AmplNLP(os.path.join(R, "tests", "golden", "hs_nl", name + ".nl")); dev = DeviceNLP(host)
    x0, _ = host.Get_starting_point(); xl, xu, _, _ = host.Get_bounds_info()
    rng = np.random.default_rng(71000)
    X = np.clip(x0 * (1 + 0.1 * rng.standard_normal((Bs, host.n))) + 0.1 * rng.standard_normal((Bs, host.n)), xl, xu)
    alg = DeviceBatchedSQP(dev, x0=X); alg.Optimize()
    for rep in range(3):
        l0 = alg.launches
        t0 = time.perf_counter(); alg.reset(X); res = alg.Optimize(); t1 = time.perf_counter()
        print("%s x %d: %.2f ms -> %.2f M solves/s  optimal %d  SQP iters mean %.2f max %d  QP iters mean %.1f max %d  launches %d" % (
            name, Bs, 1e3 * (t1 - t0), Bs / (t1 - t0) / 1e6, (res.exitflag == 0).sum(), res.iters.mean(), res.iters.max(),
            res.qp_iter.mean(), res.qp_iter.max(), alg.launches - l0), flush=True)
    alg.close(); dev.close()

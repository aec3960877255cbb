"""Synchronous against asynchronous device SQP solves (DeviceBatchedSQP.Optimize / solve_stream against optimize_async /
solve_stream_async, the loop recorded as a CUDA graph with device-side branching), in one session, alternating the two:

  1. HS071 x 10^4 and x 10^6: wall time of one call, host to host (Optimize() against optimize_async().result()), after reset();
  2. the 24 models of bench.py's HS slice x 10^4: one after another (synchronous) against all 24 queued at once, one stream per
     object, then waited for (solves/s over the whole slice);
  3. recording costs: sqpb200_sqp_graph_create (capture + instantiation of the Optimize loop, once per object) and the enqueue time of
     solve_stream_async (which records its loop per call) against that of optimize_async.

Every asynchronous result is checked bit for bit against the synchronous one.

    python tools/sqp_async.py [--out profiles/r3_sqp_async.md] [--reps 5]
"""
import argparse
import os
import sys
import time

import numpy as np

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
sys.path.insert(0, os.path.join(R, "tools"))
import restartsqp_b200 as r  # noqa: E402
from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP  # noqa: E402
from restartsqp_b200.sqp_device import DeviceBatchedSQP  # noqa: E402
from sqp_stream import FIELDS, card, starts  # noqa: E402

HS_SLICE = ["hs003", "hs004", "hs005", "hs012", "hs014", "hs016", "hs019", "hs022", "hs023", "hs024", "hs028", "hs029", "hs030", "hs031",
            "hs033", "hs035", "hs036", "hs043", "hs051", "hs052", "hs071", "hs076", "hs100", "hs113"]  # bench.py's HS_SLICE


def same(a, b):
    return all(np.array_equal(getattr(a, k), getattr(b, k), equal_nan=True) for k in FIELDS)


def model(name):
    host = AmplNLP(os.path.join(R, "tests", "golden", "hs_nl", name + ".nl"))
    return host, DeviceNLP(host)


def stats(ts):
    ts = np.asarray(ts) * 1e3
    return "%.2f | %.2f-%.2f" % (np.median(ts), ts.min(), ts.max())


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="10000,1000000")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rows = ["# Synchronous against asynchronous device SQP solves (`tools/sqp_async.py`)", "",
            "Card: %s (name, power limit, max SM clock, read in the same run).  Default options (`iter_max` = 1000).  Times are host "
            "wall times of whole calls including the results' copy to the host, after one warm-up call of each mode; the two modes "
            "alternate, %d repetitions each.  `bitwise`: every field of every instance equals the synchronous result." % (card(), a.reps), ""]

    # 1. one model, one object, per-call wall time
    rows += ["## HS071, one object, one call", "", "| B | mode | median ms | min-max ms | bitwise |", "|---:|---|---:|---:|---|"]
    host, dev = model("hs071")
    for B in (int(v) for v in a.sizes.split(",")):
        X = starts(host, B, 81000)
        alg = DeviceBatchedSQP(dev, x0=X, options=r.Options())
        ref = alg.Optimize()
        t = {"Optimize()": [], "optimize_async().result()": []}
        ok = True
        for rep in range(a.reps + 1):
            for mode in t:
                alg.reset(X)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = alg.Optimize() if mode == "Optimize()" else alg.optimize_async().result()
                dt = time.perf_counter() - t0
                if rep:
                    t[mode].append(dt)
                ok &= same(res, ref)
        for mode, ts in t.items():
            rows.append("| %d | %s | %s | %s |" % (B, mode, stats(ts), "yes" if ok else "**NO**"))
        print("\n".join(rows[-2:]), flush=True)
        # 3. recording costs on this object
        tc = []
        for _ in range(a.reps):
            r.capi.lib().sqpb200_sqp_graph_destroy(alg._graph)
            alg._graph = None
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            alg._create_graph()
            tc.append(time.perf_counter() - t0)
        te, ts_ = [], []
        Xs = starts(host, 2 * B, 81001)
        ref_s = alg.solve_stream(Xs)
        for _ in range(a.reps):
            alg.reset(X)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            p = alg.optimize_async()
            te.append(time.perf_counter() - t0)
            p.wait()
            t0 = time.perf_counter()
            p = alg.solve_stream_async(Xs)
            ts_.append(time.perf_counter() - t0)
            ok_s = same(p.result(), ref_s)
        rows.append("| %d | (recording) sqpb200_sqp_graph_create | %s | - |" % (B, stats(tc)))
        rows.append("| %d | (enqueue) optimize_async() | %s | - |" % (B, stats(te)))
        rows.append("| %d | (enqueue, records per call) solve_stream_async(N = %d) | %s | %s |" % (B, 2 * B, stats(ts_), "yes" if ok_s else "**NO**"))
        print("\n".join(rows[-3:]), flush=True)
        alg.close()
    dev.close()

    # 2. the HS slice: 24 models one after another against all concurrently
    rows += ["", "## bench.py's HS slice, 24 models x 10^4, one object (and stream) per model", "",
             "| mode | median ms | min-max ms | solves/s (median) | bitwise |", "|---|---:|---:|---:|---|"]
    objs, Xs, refs = [], [], []
    for k, name in enumerate(HS_SLICE):
        host, dev = model(name)
        X = starts(host, 10000, 82000 + k)
        objs.append((dev, DeviceBatchedSQP(dev, x0=X, options=r.Options(), stream=torch.cuda.Stream())))
        Xs.append(X)
    refs = [alg.Optimize() for _, alg in objs]
    t = {"synchronous, one after another": [], "asynchronous, 24 streams": []}
    ok = True
    for rep in range(a.reps + 1):
        for mode in t:
            for (_, alg), X in zip(objs, Xs):
                alg.reset(X)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if mode.startswith("sync"):
                res = [alg.Optimize() for _, alg in objs]
            else:
                res = [p.result() for p in [alg.optimize_async() for _, alg in objs]]
            dt = time.perf_counter() - t0
            if rep:
                t[mode].append(dt)
            ok &= all(same(u, v) for u, v in zip(res, refs))
    for mode, ts in t.items():
        rows.append("| %s | %s | %.3g | %s |" % (mode, stats(ts), len(objs) * 10000 / np.median(ts), "yes" if ok else "**NO**"))
    print("\n".join(rows[-2:]), flush=True)
    for dev, alg in objs:
        alg.close()
        dev.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    main()

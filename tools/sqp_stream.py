"""Chunked against streamed multistart: N starting points of one HS model through B device instances, either as N / B batches
(DeviceBatchedSQP.reset + Optimize per chunk, each chunk waiting for its slowest instance) or as one solve_stream call (a stopped
slot takes the next starting point on the device), for several refill_min.  Wall times are synchronised (both paths end with their
results on the host), taken after one warm-up run of each configuration; the median of `--reps` runs is reported.  Every streamed
result is checked bit for bit against the chunked one.

    python tools/sqp_stream.py [--out profiles/r3_sqp_stream.md] [--reps 3] [--cases hs036:100000,hs071:1000000] [--slots 10000,100000]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
import restartsqp_b200 as r  # noqa: E402
from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP  # noqa: E402
from restartsqp_b200.sqp_device import DeviceBatchedSQP, REFILL_MIN_FRACTION  # noqa: E402
from restartsqp_b200.sqp_driver import SQPResult  # noqa: E402

FIELDS = ("exitflag", "iters", "qp_iter", "x", "obj", "rho", "delta", "KKT_error")


def starts(nlp, N, seed):
    """perturbed starts as tests/test_hs_suite.py draws them (SURVEY.md 8d config 3)"""
    x0, _ = nlp.Get_starting_point()
    xl, xu, _, _ = nlp.Get_bounds_info()
    rng = np.random.default_rng(seed)
    return np.clip(x0 * (1 + 0.1 * rng.standard_normal((N, nlp.n))) + 0.1 * rng.standard_normal((N, nlp.n)), xl, xu)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        return q.stdout.strip().splitlines()[0]
    except (OSError, subprocess.SubprocessError, IndexError):
        import torch
        return torch.cuda.get_device_name(0) + ", power limit not readable"


def chunked(alg, X):
    B, out = alg.batch, []
    for k in range(0, len(X), B):
        c = X[k:k + B]
        if len(c) < B:  # last chunk: pad with its own first start, drop the padding afterwards
            c = np.concatenate([c, np.repeat(c[:1], B - len(c), axis=0)])
        alg.reset(c)
        out.append(alg.Optimize())
    return SQPResult(**{k: np.concatenate([getattr(o, k) for o in out])[:len(X)] for k in FIELDS})


def timed(fn, reps):
    fn()  # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        res = fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="hs036:100000,hs071:1000000")
    ap.add_argument("--slots", default="10000,100000")
    ap.add_argument("--refill", default="1,64,16,4", help="refill_min values: 1, then slot-count divisors")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--iter-max", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rows = ["# Streamed against chunked multistart (`tools/sqp_stream.py`)", "",
            "Card: %s (name, power limit, max SM clock, read in the same run).  Median of %d synchronised wall times after one warm-up "
            "run per configuration; host-to-host (starting points in, results out).  `iter_max` = %d, default options otherwise.  "
            "`rounds`: refill rounds of the streamed run, the initial fill included (chunked: the number of chunks).  `bitwise`: every "
            "field of every instance equals the chunked run's." % (card(), a.reps, a.iter_max), "",
            "| model | N | slots B | mode | refill_min | rounds | time (s) | solves/s | vs chunked | bitwise |",
            "|---|---:|---:|---|---:|---:|---:|---:|---:|---|"]
    print("\n".join(rows), flush=True)
    for case in a.cases.split(","):
        name, N = case.split(":")
        N = int(N)
        host = AmplNLP(os.path.join(R, "tests", "golden", "hs_nl", name + ".nl"))
        dev = DeviceNLP(host)
        X = starts(host, N, 71000)
        for B in (int(s) for s in a.slots.split(",")):
            if B > N:
                continue
            opt = r.Options(iter_max=a.iter_max)
            alg = DeviceBatchedSQP(dev, x0=X[:B], options=opt)
            t_c, ref = timed(lambda: chunked(alg, X), a.reps)
            line = "| %s | %d | %d | chunked | - | %d | %.4f | %.3g | 1.00 | - |" % (name, N, B, -(-N // B), t_c, N / t_c)
            rows.append(line)
            print(line, flush=True)
            for d in (int(v) for v in a.refill.split(",")):
                rm = 1 if d == 1 else max(1, B // d)
                t_s, res = timed(lambda: alg.solve_stream(X, refill_min=rm), a.reps)
                same = all(np.array_equal(getattr(res, k), getattr(ref, k), equal_nan=True) for k in FIELDS)
                tag = "B/%d" % d if d != 1 else "1"
                if d == REFILL_MIN_FRACTION:
                    tag += " (default)"
                line = "| %s | %d | %d | streamed | %s = %d | %d | %.4f | %.3g | %.2f | %s |" % (
                    name, N, B, tag, rm, alg.stream_rounds, t_s, N / t_s, t_c / t_s, "yes" if same else "**NO**")
                rows.append(line)
                print(line, flush=True)
            alg.close()
        dev.close()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(rows) + "\n")


if __name__ == "__main__":
    main()

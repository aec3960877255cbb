#!/usr/bin/env python
"""The reference's real SQP loop against the oracle of the loop over every fixture model (dev container only: needs the
oracle/_ref/algorithm_nl_twin* programs that `make -C oracle ref` builds from /root/reference).

    python tools/reference_loop_pin.py [starts per model] > profiles/r2_reference_loop_pin.md

For every `.nl` fixture (124 HS, 25 CUTE) and every perturbed start: src/Algorithm.cpp + SQPTNLP.cpp + QPhandler.cpp on the
QORE-layout plugin over the CPU twin of the C ABI (clipping of infinite bounds off: `_noclip`, and as shipped) against
oracle/oracle_sqp.c on the same C evaluator.  See tests/test_reference_algorithm.py for what may differ and why."""
import glob
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def main():
    import numpy as np
    import restartsqp_b200 as r
    from restartsqp_b200.nl_reader import AmplNLP, write_model_file
    from oracle import oracle_py as orc
    from test_hs_suite import perturbed_starts
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 6
    files = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "hs_nl", "*.nl"))) + sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "cute_nl", "*.nl")))
    rows, tot = [], dict(noclip=[0, 0, 0], shipped=[0, 0, 0])
    with tempfile.TemporaryDirectory() as td:
        for path in files:
            name = os.path.basename(path)[:-3]
            try:
                h = AmplNLP(path)
                X = perturbed_starts(h, B, 4)
                so = orc.SqpOracle(h, r.Options())
                res = so.solve_batch(X)
                model = os.path.join(td, name + ".model")
                write_model_file(h, model, X)
                ev = so.evaluator
            except Exception as e:  # noqa: BLE001
                rows.append((name, "-", "-", "skipped: %s" % repr(e)[:60]))
                continue
            cell = {}
            for kind in ("noclip", "shipped"):
                exe = os.path.join(ROOT, "oracle", "_ref", "algorithm_nl_twin" + ("_noclip" if kind == "noclip" else ""))
                same = labels = other = 0
                notes = []
                for k in range(B):
                    p = subprocess.run([exe, model, ev, str(k), "qore"], cwd=td, capture_output=True, text=True, timeout=600)
                    t = p.stdout.split()
                    if p.returncode != 0:
                        other += 1
                        notes.append("#%d %s" % (k, p.stdout.strip()[:30]))
                        continue
                    ex, it, qi = int(t[0]), int(t[1]), int(t[2])
                    x = np.array([float.fromhex(v) for v in t[4:]])
                    path_same = it == int(res["iters"][k]) and qi == int(res["qp_iter"][k]) and np.array_equal(x, res["x"][k], equal_nan=True)
                    if path_same and ex == int(res["exitflag"][k]):
                        same += 1
                    elif path_same:
                        labels += 1
                        notes.append("#%d flag %d/%d" % (k, ex, int(res["exitflag"][k])))
                    else:
                        other += 1
                        notes.append("#%d (%d,%d,%d)/(%d,%d,%d)" % (k, ex, it, qi, int(res["exitflag"][k]), int(res["iters"][k]), int(res["qp_iter"][k])))
                tot[kind][0] += same; tot[kind][1] += labels; tot[kind][2] += other
                cell[kind] = ("%d/%d" % (same, B)) + ((" " + "; ".join(notes[:3])) if notes else "")
            rows.append((name, "%d x %d" % (h.n, h.m), cell["noclip"], cell["shipped"]))
    n = sum(tot["noclip"])
    print("# r2 — the reference's real SQP loop against the oracle of the loop, every fixture model x %d perturbed starts\n" % B)
    print("`python tools/reference_loop_pin.py %d` (dev container).  Left: `oracle/_ref/algorithm_nl_twin_noclip` (the reference's `Algorithm.cpp` +\n"
          "`SQPTNLP.cpp` + `QPhandler.cpp` on the QORE-layout plugin over the CPU twin of the C ABI, QORE setters' clipping of infinite bounds off);\n"
          "right: the plugin as shipped.  A run counts as identical when exit flag, outer iterations, QP iterations and the final iterate\n"
          "agree bit for bit with `oracle/oracle_sqp.c`; `flag a/b` = same path, other failure label (reference / oracle); `(flag, iterations,\n"
          "QP iterations)` pairs = other path.\n" % B)
    for kind, label in (("noclip", "bounds as the oracle takes them"), ("shipped", "plugin as shipped (bounds clipped to +-1e18)")):
        t = tot[kind]
        print("* %s: **%d of %d runs identical**, %d with another failure label only, %d other (exceptions, other paths)." % (label, t[0], n, t[1], t[2]))
    print("\n| model | n x m | identical (no clipping) | identical (as shipped) |\n|---|---|---|---|")
    for row in rows:
        print("| %s | %s | %s | %s |" % row)


if __name__ == "__main__":
    main()

"""A/B timing of two builds of libsqpb200.so in one session on one GPU.

    python tools/qp_ab.py LIB_A LIB_B [--rounds 3] [--replicas 4096] [--steps 5] [--warmup 3] [--json FILE]

Each run is one subprocess with SQPB200_LIB pointing at one library, and the runs alternate A, B, A, B, ... so that
clock and co-tenant drift hit both builds alike.  A run is (1) tools/per_fixture.py: the launch time of every dumped QP x
replicas, cold start, and (2) bench.py --extras 0 --strong 0: the headline QPs/s.  The report gives, per build, the
median and the max-min spread over its rounds, and the GPU's name, power limit and clocks read in the same session (a
time is only worth something with what it was measured on).
"""
import argparse
import json
import os
import re
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIXTURE_LINE = re.compile(r"^(\S+)\s+nV=\s*(\d+)\s+nC=\s*(\d+).*?solve=([0-9.]+)ms.*?status=(\{[^}]*\})")


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem,temperature.gpu"
    r = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]],
                       capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "nvidia-smi unavailable: " + r.stderr.strip()


def run(lib, cmd):
    env = dict(os.environ, SQPB200_LIB=os.path.abspath(lib))
    r = subprocess.run([sys.executable] + cmd, cwd=ROOT, env=env, capture_output=True, text=True)
    if r.returncode != 0:
        raise SystemExit("run failed (%s, %s):\n%s\n%s" % (lib, " ".join(cmd), r.stdout[-4000:], r.stderr[-4000:]))
    return r.stdout


def one_round(lib, args):
    fx = {}
    for line in run(lib, ["tools/per_fixture.py", str(args.replicas)]).splitlines():
        m = FIXTURE_LINE.match(line.strip())
        if m:
            fx[m.group(1)] = dict(nV=int(m.group(2)), nC=int(m.group(3)), ms=float(m.group(4)), status=m.group(5))
    out = run(lib, ["bench.py", "--gpus", "1", "--steps", str(args.steps), "--warmup", str(args.warmup),
                    "--replicas", str(args.replicas), "--extras", "0", "--strong", "0"])
    res = json.loads([l for l in out.splitlines() if l.startswith("{")][-1])
    return fx, dict(value=res["value"], ms_per_step=res["ms_per_step"], solved_optimal=res["config"]["solved_optimal"])


def spread(v):
    return max(v) - min(v)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("lib_a")
    ap.add_argument("lib_b")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--replicas", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--json", default=None, help="also write every raw number to this file")
    args = ap.parse_args()
    libs = {"A": args.lib_a, "B": args.lib_b}
    info = [gpu_info()]
    runs = {"A": [], "B": []}
    for k in range(args.rounds):
        for tag in ("A", "B"):
            runs[tag].append(one_round(libs[tag], args))
            print("round %d %s: %.4g QPs/s, %.3f ms/step" % (k, tag, runs[tag][-1][1]["value"], runs[tag][-1][1]["ms_per_step"]), flush=True)
    info.append(gpu_info())
    print("\nGPU (start / end): " + " | ".join(info))
    print("A = %s\nB = %s\n%d alternating rounds, %d replicas per dumped QP, cold start\n" % (libs["A"], libs["B"], args.rounds, args.replicas))
    print("| QP | nV | nC | A median ms | A spread | B median ms | B spread | B/A |")
    print("|---|---|---|---|---|---|---|---|")
    for name in runs["A"][0][0]:
        a = [r[0][name]["ms"] for r in runs["A"]]
        b = [r[0][name]["ms"] for r in runs["B"]]
        q = runs["A"][0][0][name]
        print("| %s | %d | %d | %.3f | %.3f | %.3f | %.3f | %.3f |" % (name, q["nV"], q["nC"], statistics.median(a), spread(a),
                                                                 statistics.median(b), spread(b), statistics.median(b) / statistics.median(a)))
    va = [r[1]["value"] for r in runs["A"]]
    vb = [r[1]["value"] for r in runs["B"]]
    print("\nbench value (QPs/s): A median %.4g (spread %.3g), B median %.4g (spread %.3g), B/A %.3f"
          % (statistics.median(va), spread(va), statistics.median(vb), spread(vb), statistics.median(vb) / statistics.median(va)))
    print("solved_optimal: A %s, B %s" % (sorted({r[1]["solved_optimal"] for r in runs["A"]}), sorted({r[1]["solved_optimal"] for r in runs["B"]})))
    if args.json:
        with open(args.json, "w") as f:
            json.dump(dict(gpu=info, libs=libs, runs=runs), f, indent=1)


if __name__ == "__main__":
    main()

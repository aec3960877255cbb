#!/usr/bin/env python
"""bench.py -- QP subproblems/sec of the batched QP-subproblem hot path on B200.

Workload (BASELINE.json configs[1], SURVEY.md 8d config 2): replay of the dumped QP subproblems of
test/unsolved_QP_data + test/unsolved_QPs as a batch.  Every dumped QP with a symmetric Hessian array that is solvable
(20 of the 27: six hold a non-symmetric "H", i.e. are not QPs, and QORE_hs107 is the reference's own non-convex failure
case; all seven stay robustness tests) is replicated B = 4096 times with g *= 1 + 1e-3*U(-1,1) (seed 1234, replica 0
exact).  One step = one cold-start solve (init) of every replica of every dumped QP = 20*B QPs per GPU.  With N GPUs every
rank solves its own 20*B replicas (rank-seeded perturbations): weak scaling, no collective on the path.

  value  QPs/s with all inputs resident in HBM: K steps of 20 solve launches, CUDA events, max over ranks.
  e2e    the same through the public plugin API with HOST (pinned) buffers: every step uploads H, A values,
         g, lb, ub, lbA, ubA of every instance (sqpb200_solve_host: one copy per block), solves, and reads x, y,
         objective, KKT residuals, status and iteration counts back.
  roofline  qp_solve_kernel, dominant launch (hs116 x B): the binding resource of SURVEY.md 8d for nV <~ 100 is the
         on-chip one, so `achieved` is the shared-memory rate (wavefronts of the committed ncu capture of exactly this
         launch x 128 B over the launch's CUDA-event time of this run) against the shared-memory peak measured in this
         run; the HBM figure (algorithmic compulsory bytes, DRAM traffic of the capture) and the FP64 rate are beside it.
  cpu_baseline  the CPU oracle (oracle/, a port: qpOASES itself is not available) on all host cores over the same
         replicas per dumped QP.
  extras (1 GPU)  the other BASELINE.json configs, each with its own CPU figure: full SQP solves/s (HS071 x 1e4 / 1e6,
         a 24-problem slice of the HS suite x 1e4), the synthetic large QPs n = 256 / 512 / 1024 on the DMMA + TMA
         cluster kernel, and the HBM-bound L0 kernels (GB/s against the measured copy peak).
  strong  BASELINE.json configs[4]: a FIXED 10^6 HS071 instances sharded by instance index over the N ranks
         (device-resident SQP loop, no collective on the path), so that the driver's 1/2/4/8 runs show strong scaling too.
  weak_sqp  the weak-scaling leg of the same config: 1.25 x 10^5 HS071 instances per GPU.

`--impl reference` times the CPU path alone and prints the same JSON line with "impl": "reference".
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
METRIC = "QP subproblems/sec"
UNIT = "QPs/s"
WORKLOAD = "replay_dumped_qps (test/unsolved_QP_data + test/unsolved_QPs, the 20 symmetric-H dumps that are solvable x B replicas, cold start)"
# QORE_hs107 is the reference's own failure case (non-convex: the projected Hessian of the working set the homotopy reaches is
# indefinite); GPU kernel, CPU oracle and the reference's qpOASES run all end it with an error status, so it is a robustness
# test (tests/test_gpu_qp.py), not a throughput workload: the headline counts only solves that end QP_OPTIMAL (VERDICT r1).
EXCLUDED = ("QORE_hs107",)
HS_SLICE = ["hs003", "hs004", "hs005", "hs012", "hs014", "hs016", "hs019", "hs022", "hs023", "hs024", "hs028", "hs029", "hs030", "hs031",
            "hs033", "hs035", "hs036", "hs043", "hs051", "hs052", "hs071", "hs076", "hs100", "hs113"]


# ------------------------------------------------------------------------------------------ workload
def load_fixtures():
    import scipy.sparse as sp
    with open(os.path.join(ROOT, "tests", "golden", "qp_fixtures.json")) as f:
        qps = json.load(f)["qps"]
    out = []
    for q in qps:
        nV = q["nV"]
        Hd = sp.csc_matrix((q["H_val"], q["H_rowidx"], q["H_colptr"]), shape=(nV, nV)).toarray()
        if np.abs(Hd - Hd.T).max() == 0.0 and q["name"] not in EXCLUDED:
            out.append(q)
    return out


def make_batch(q, B, seed):
    nV, nC = q["nV"], q["nC"]
    rng = np.random.default_rng(seed)
    g = np.tile(np.array(q["g"], dtype=np.float64), (B, 1))
    g[1:] *= 1.0 + 1e-3 * rng.uniform(-1.0, 1.0, size=g[1:].shape)
    tile = lambda k, n: np.ascontiguousarray(np.tile(np.array(q[k], dtype=np.float64).reshape(1, n), (B, 1)))
    return dict(nV=nV, nC=nC, g=g, lb=tile("lb", nV), ub=tile("ub", nV), lbA=tile("lbA", nC), ubA=tile("ubA", nC),
                Av=tile("A_val", len(q["A_val"])), Hv=tile("H_val", len(q["H_val"])))


def algorithmic_bytes(q):
    """Compulsory HBM bytes of one solve (SURVEY.md 8d, row 'QP/LP solve'): data in, x/y/working set/obj/status out."""
    nV, nC, zA, zH = q["nV"], q["nC"], len(q["A_val"]), len(q["H_val"])
    return 8 * (zH + zA + 3 * nV + 2 * nC) + 8 * (2 * nV + nC) + 4 * (nV + nC) + 16


DUMP_BYTES = 60 * 1000 * 1000  # array data of --dump-outputs: the files, headers included, stay under 64 MB


def dump_outputs(path, groups, B):
    """What a caller of the timed path holds after its last step, per dumped QP: x [B, nV], the multipliers of the bounds
    [B, nV] and of the constraints [B, nC] (not written when nC = 0), the objective, status and iteration count [B], written as
    float64 `path/<dump>_<array>.npy`.  Above DUMP_BYTES in all, the same seeded sample of replicas (rows) is kept for every dumped QP."""
    os.makedirs(path, exist_ok=True)
    total = sum(8 * B * (2 * gr["nV"] + gr["nC"] + 3) for gr in groups)
    rows = np.arange(B)
    if total > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(B, B * DUMP_BYTES // total, replace=False))
    for gr in sorted(groups, key=lambda gr: gr["q"]["name"]):
        s = gr["s"]
        arrays = {"x": s.get_optimal_solution(), "y_bounds": s.get_multipliers_bounds(), "y_constr": s.get_multipliers_constr(),
                  "obj": s.get_obj_value(), "status": s.get_status(), "iters": s.get_iterations()}
        for k, a in arrays.items():
            if a.size == 0:  # y_constr of a dump without constraints (nC = 0): nothing to compare
                continue
            np.save(os.path.join(path, "%s_%s.npy" % (gr["q"]["name"], k)), np.ascontiguousarray(a[rows], dtype=np.float64))


def perturbed_starts(nlp, B, k):
    """SURVEY.md 8d config 3: x0_i = clip(x0*(1 + 0.1 N) + 0.1 N), default_rng(71000 + problem index)."""
    x0, _ = nlp.Get_starting_point()
    xl, xu, _, _ = nlp.Get_bounds_info()
    rng = np.random.default_rng(71000 + k)
    return np.clip(x0 * (1 + 0.1 * rng.standard_normal((B, nlp.n))) + 0.1 * rng.standard_normal((B, nlp.n)), xl, xu)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([t.strip() for t in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_rate(fixtures, sample_B, seed, max_seconds=25.0, min_seconds=0.0):
    """QPs/s of the CPU oracle on all host cores over `sample_B` replicas of every dumped QP (whole passes over the
    dumps are repeated until `min_seconds` of CPU work have been timed; data generation is outside the timed region)."""
    from oracle import oracle_py as orc
    cores = orc.lib().orc_max_threads()
    total, t_total = 0, 0.0
    batches = [make_batch(q, sample_B, seed + k) for k, q in enumerate(fixtures)]
    while True:
        for q, d in zip(fixtures, batches):
            A = (q["A_colptr"], q["A_rowidx"], q["A_val"])
            H = (q["H_colptr"], q["H_rowidx"], q["H_val"])
            t0 = time.perf_counter()
            r = orc.solve_batch(d["nV"], d["nC"], A, H, d["g"], d["lb"], d["ub"], d["lbA"], d["ubA"], Avals=d["Av"], Hvals=d["Hv"])
            t_total += time.perf_counter() - t0
            total += sample_B
            cores = r["threads"]
        if t_total >= min_seconds or t_total > max_seconds:
            break
    return total / t_total, cores, total, t_total


def run_reference(args, rank, world):
    if rank != 0:
        return
    fixtures = load_fixtures()
    sample_B = args.replicas  # the same replicas per dumped QP as the GPU arm
    cores = 1
    for _ in range(args.warmup):
        cpu_rate(fixtures, min(sample_B, 64), 1234)
    tot, tt = 0, 0.0
    for _ in range(args.steps):
        r, cores, n, t = cpu_rate(fixtures, sample_B, 1234, max_seconds=30.0, min_seconds=4.0)
        tot += n; tt += t
    value = tot / tt
    sample = "per step: passes over %d replicas of each of the %d dumped QPs for >= 4 s (%d QPs/step on average)" % (
        sample_B, len(fixtures), tot // max(1, args.steps))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * tt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic (dumped QP fixtures of the reference, perturbed replicas)",
        "config": {"workload": WORKLOAD, "replicas_per_qp": sample_B, "qps_per_step_per_gpu": len(fixtures) * sample_B},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "CPU oracle (restatement of the qpOASES path; qpOASES 3.2.1 is not available offline), "
                                 "one solver object per thread, pthreads over instances"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------ GPU arm
def run_gpu(args, rank, world, local_rank):
    import torch
    import restartsqp_b200 as r
    from restartsqp_b200 import capi
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    fixtures = load_fixtures()
    B = args.replicas
    groups = []
    h2d = d2h = 0
    for k, q in enumerate(fixtures):
        d = make_batch(q, B, 1234 + 1000 * rank + k)
        s = r.CudaQPInterface(nV=d["nV"], nC=d["nC"], qptype=r.QPType.QP, batch=B, device=local_rank, keep_state=False,
                              team_size=args.team)
        s.set_csc(capi.MAT_A, q["A_colptr"], q["A_rowidx"], d["Av"])
        s.set_csc(capi.MAT_H, q["H_colptr"], q["H_rowidx"], d["Hv"])
        s.set_g(d["g"]); s.set_lb(d["lb"]); s.set_ub(d["ub"])
        if d["nC"]:
            s.set_lbA(d["lbA"]); s.set_ubA(d["ubA"])
        # pinned host mirror of the handle's two contiguous blocks (sqpb200_io_layout) + the matrix values
        lay = s.io_layout()
        inb = torch.zeros(lay["in_bytes"], dtype=torch.uint8).pin_memory()
        for kk, off in lay["in_off"].items():
            v = np.ascontiguousarray(d[kk])
            if v.size:
                inb[off:off + v.nbytes] = torch.from_numpy(v.view(np.uint8).reshape(-1))
        outb = torch.zeros(lay["out_bytes"], dtype=torch.uint8).pin_memory()
        Av, Hv = torch.from_numpy(d["Av"]).pin_memory(), torch.from_numpy(d["Hv"]).pin_memory()
        h2d += lay["in_bytes"] + Av.numel() * 8 + Hv.numel() * 8
        d2h += lay["out_bytes"]
        groups.append(dict(q=q, s=s, inb=inb, outb=outb, Av=Av, Hv=Hv, lay=lay, nV=d["nV"], nC=d["nC"]))
    # End-to-end path, double-buffered: a second handle per dumped QP (own device arena, own stream, own pinned result block,
    # the same pinned inputs), so that the uploads of step k+1 run while step k is being solved, as a host that replays a stream
    # of batches would arrange it.  Every step still uploads all its inputs and downloads all its results.
    groups_b = []
    if args.e2e_overlap:
        for gr in groups:
            q = gr["q"]
            s2 = r.CudaQPInterface(nV=gr["nV"], nC=gr["nC"], qptype=r.QPType.QP, batch=B, device=local_rank, keep_state=False, team_size=args.team)
            s2.set_csc(capi.MAT_A, q["A_colptr"], q["A_rowidx"], gr["Av"].numpy())
            s2.set_csc(capi.MAT_H, q["H_colptr"], q["H_rowidx"], gr["Hv"].numpy())
            groups_b.append(dict(gr, s=s2, outb=torch.zeros(gr["lay"]["out_bytes"], dtype=torch.uint8).pin_memory()))
    torch.cuda.synchronize()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    # one CUDA stream per dumped QP: the independent solve launches of a step overlap, so small groups fill the
    # SMs that the tail of the long one (hs116) leaves idle
    streams = [torch.cuda.Stream() for _ in groups] if args.streams else None

    def use_streams(on):
        for k, gr in enumerate(groups):
            gr["s"].set_stream(streams[k].cuda_stream if (on and streams) else 0)

    def fork():
        flush.zero_()
        if streams:
            ev = torch.cuda.Event()
            ev.record()
            for st in streams:
                st.wait_event(ev)

    def join():
        if streams:
            cur = torch.cuda.current_stream()
            for st in streams:
                cur.wait_stream(st)

    def step_resident():
        fork()
        for gr in groups:
            gr["s"]._solve(r.QPType.QP, None, None, 0)
        join()

    def step_e2e():
        fork()
        for gr in groups:  # one call per group: 3 uploads, the solve, 1 download, all queued on the group's stream
            gr["s"].solve_host(r.QPType.QP, gr["inb"].data_ptr(), gr["Av"].data_ptr(), gr["Hv"].data_ptr(), gr["outb"].data_ptr())
        join()

    streams_b = [torch.cuda.Stream() for _ in groups_b]
    for gr, st in zip(groups_b, streams_b):
        gr["s"].set_stream(st.cuda_stream)

    def run_e2e_overlapped(n):
        """n steps; step k goes to handle set k % 2.  All streams start after the current stream and are joined at the end."""
        ev = torch.cuda.Event()
        ev.record()
        for st in (streams or []) + streams_b:
            st.wait_event(ev)
        for k in range(n):
            for gr in (groups if k % 2 == 0 else groups_b):
                gr["s"].solve_host(r.QPType.QP, gr["inb"].data_ptr(), gr["Av"].data_ptr(), gr["Hv"].data_ptr(), gr["outb"].data_ptr())
        cur = torch.cuda.current_stream()
        for st in (streams or []) + streams_b:
            cur.wait_stream(st)

    def timed_e2e_overlapped(steps, warmup):
        run_e2e_overlapped(warmup)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run_e2e_overlapped(steps)
        e1.record()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn, steps, warmup, collect_kernel_ms=False):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = sum(gr["s"].launch_count() for gr in groups)
        kms = 0.0
        e0.record()
        for _ in range(steps):
            fn()
            if collect_kernel_ms:  # per-launch CUDA-event time recorded by the library around qp_solve_kernel
                kms += sum(gr["s"].last_solve_ms() for gr in groups)
        e1.record()
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        ms = e0.elapsed_time(e1)
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        launches = sum(gr["s"].launch_count() for gr in groups) - launches0
        return float(t.item()), launches, kms

    # Launch order: longest solve first (the step is bounded by its longest kernel, so that kernel must start first and
    # the short ones fill the SMs its tail leaves idle).  The order comes from untimed calibration passes on the default
    # stream (two: the handles learn their factor capacity in the first).
    for _ in range(2):
        step_resident()
        torch.cuda.synchronize()
    cal = [gr["s"].last_solve_ms() for gr in groups]
    order = sorted(range(len(groups)), key=lambda i: -cal[i])
    groups[:] = [groups[i] for i in order]
    if groups_b:
        groups_b[:] = [groups_b[i] for i in order]
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    use_streams(True)
    ms_res, launches, _ = timed(step_resident, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, groups, B)
    ms_e2e_serial, _, _ = timed(step_e2e, args.steps, max(3, args.warmup // 2))  # one step at a time (L2 flush + join between steps)
    ms_e2e = timed_e2e_overlapped(args.steps, max(4, args.warmup)) if (groups_b and streams) else ms_e2e_serial
    clocks = sampler.stop() if rank == 0 else None  # sampled every 20 ms across both timed regions (and their warm-ups)
    # serial pass on the default stream, only to attribute device time to the solve kernel (per-launch CUDA events)
    torch.cuda.synchronize()
    use_streams(False)
    ms_serial, _, kernel_ms = timed(step_resident, args.steps, 1, collect_kernel_ms=True)
    qps_step = len(fixtures) * B * world
    value = qps_step * args.steps / (ms_res * 1e-3)
    e2e = qps_step * args.steps / (ms_e2e * 1e-3)

    strong = run_strong(args, rank, world, local_rank, dist) if args.strong else None
    # the weak-scaling leg of configs[4] (SURVEY.md 8d config 5): 1.25 x 10^5 instances per GPU
    weak_sqp = run_strong(args, rank, world, local_rank, dist, N=125000 * world, scaling="weak") if args.strong else None

    if rank == 0:
        status_ok, per_dump, e2e_ok = 0, {}, 0
        for gr in groups:
            ok = int((gr["s"].get_status() == 20).sum())
            status_ok += ok
            per_dump[gr["q"]["name"]] = ok
            o0 = gr["lay"]["out_off"]["status"]
            st = gr["outb"][o0:o0 + 4 * B].numpy().view(np.int32)
            e2e_ok += int((st == 20).sum())  # the statuses the end-to-end path brought back to the host
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        bytes_step = sum(algorithmic_bytes(gr["q"]) for gr in groups) * B
        kernel_s_per_step = kernel_ms * 1e-3 / args.steps
        fp64 = smem = None
        try:
            P = C.CDLL(os.path.join(ROOT, "restartsqp_b200", "lib", "libsqpb200_peaks.so"))
            a, b = C.c_double(0), C.c_double(0)
            if P.peaks_measure(C.byref(a), C.byref(b)) == 0:
                fp64, smem = a.value, b.value
        except Exception:
            pass
        flops_step = dom_flops = None
        try:
            from oracle import oracle_py as orc
            fl = 0.0
            for gr in groups:
                q = gr["q"]
                o = orc.OracleQP(q["nV"], q["nC"])
                o.init((q["H_colptr"], q["H_rowidx"], q["H_val"]), q["g"], (q["A_colptr"], q["A_rowidx"], q["A_val"]), q["lb"], q["ub"], q["lbA"], q["ubA"])
                fl += o.flops()
                if q["name"] == "QORE_hs116":
                    dom_flops = o.flops() * B
            flops_step = fl * B
        except Exception:
            pass
        # the dominant single launch: hs116, the largest dumped QP (nV=69, nC=28).  Counters that only ncu can see (DRAM bytes,
        # shared-memory wavefronts) come from the committed capture of exactly this launch shape (profiles/r2_qp_solve_hs116.json);
        # the time they are divided by is this run's CUDA-event time of the same launch.
        prof = {}
        try:
            with open(os.path.join(ROOT, "profiles", "r2_qp_solve_hs116.json")) as f:
                prof = json.load(f)
        except Exception:
            pass
        same_shape = prof.get("batch") == B
        dom = [gr for gr in groups if gr["q"]["name"] == "QORE_hs116"]
        roofline = {"kernel": "qp_solve_kernel", "peak_source_hbm": peak_src}
        if dom:
            dom_ms = dom[0]["s"].last_solve_ms()
            dom_bytes = algorithmic_bytes(dom[0]["q"]) * B
            smem_bytes = prof.get("smem_wavefronts", 0) * 128 if same_shape else None
            smem_gbs = smem_bytes / (dom_ms * 1e-3) / 1e9 if smem_bytes else None
            roofline.update({
                "launch": "QORE_hs116 x %d" % B, "launch_ms": dom_ms,
                "bound": "smem", "achieved": smem_gbs, "peak": smem, "unit": "GB/s",
                "frac": (smem_gbs / smem) if (smem_gbs and smem) else None,
                "traffic": prof.get("dram_bytes") if same_shape else None,
                "peak_source": "shared-memory read microbenchmark tools/peaks.cu, this run",
                "counter_source": prof.get("source"),
                "hbm": {"algorithmic_bytes": dom_bytes, "achieved_gbs": dom_bytes / (dom_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                        "frac": dom_bytes / (dom_ms * 1e-3) / 1e9 / hbm_peak, "traffic_bytes_ncu": prof.get("dram_bytes") if same_shape else None},
                "fp64": {"achieved_gflops": (dom_flops / (dom_ms * 1e-3) / 1e9) if dom_flops else None, "peak_gflops": fp64,
                         "frac": (dom_flops / (dom_ms * 1e-3) / 1e9 / fp64) if (dom_flops and fp64) else None,
                         "flop_model": "SURVEY.md 8d, counted by the oracle on replica 0",
                         "pipe_fp64_pct_ncu": prof.get("pipe_fp64_pct")},
                "ncu": {k: prof.get(k) for k in ("issue_active_pct", "warps_active_pct", "inst_executed", "registers", "smem_per_cta_kb")},
                "note": "active-set iterations run out of shared memory (every input byte is read from DRAM once); none of the three "
                        "rooflines binds: the kernel is latency / issue bound (ncu block, DESIGN.md 4)"})
        roofline["all_launches"] = {"algorithmic_bytes_per_step": bytes_step, "hbm_gbs": bytes_step / kernel_s_per_step / 1e9,
                                    "fp64_gflops": (flops_step / kernel_s_per_step / 1e9) if flops_step else None,
                                    "kernel_ms_per_step": 1e3 * kernel_s_per_step, "serial_ms_per_step": ms_serial / args.steps,
                                    "kernel_share_of_step": kernel_s_per_step / (ms_serial * 1e-3 / args.steps)}
        try:  # FP64 tensor-pipe peak (SURVEY.md 8d): cuBLAS DGEMM 8192^3 through torch, best of 3
            a_ = torch.randn(8192, 8192, dtype=torch.float64, device="cuda"); b_ = torch.randn(8192, 8192, dtype=torch.float64, device="cuda")
            torch.matmul(a_, b_); torch.cuda.synchronize()
            best = 1e9
            for _ in range(3):
                t0_, t1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                t0_.record(); torch.matmul(a_, b_); t1_.record(); torch.cuda.synchronize()
                best = min(best, t0_.elapsed_time(t1_))
            roofline["dgemm_peak_gflops"] = 2.0 * 8192 ** 3 / (best * 1e-3) / 1e9
            del a_, b_
        except Exception:
            pass
        rate, cores, n, t = cpu_rate(fixtures, B, 1234, max_seconds=60.0, min_seconds=12.0)  # >= 12 s of CPU work, same replicas
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic (dumped QP fixtures of the reference, perturbed replicas)",
            "config": {"workload": WORKLOAD, "replicas_per_qp": B, "qps_per_step_per_gpu": len(fixtures) * B,
                       "l2": "256 MiB buffer written between steps (inside the timed region)",
                       "solved_optimal": status_ok, "solved_optimal_e2e": e2e_ok, "solved_optimal_per_dump": per_dump,
                       "team_size": args.team or "auto", "streams": len(streams) if streams else 1},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps,
                    "api": "sqpb200_solve_host (CudaQPInterface.solve_host): per dumped QP one upload of the vector block, one each of the A and H "
                           "values, the solve, one download of the result block",
                    "overlap": ("two handles per dumped QP alternate, so the copies of step k+1 overlap the solves of step k; every step uploads all "
                                "inputs and downloads all results") if (groups_b and streams) else "none",
                    "serial": {"value": qps_step * args.steps / (ms_e2e_serial * 1e-3), "ms_per_step": ms_e2e_serial / args.steps,
                               "note": "one step at a time: L2 flush and a join of all streams between steps"}},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline,
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d QPs (passes over %d replicas of each of the %d dumped QPs) in %.1f s" % (n, B, len(fixtures), t)},
        }
        if strong is not None:
            out["strong"] = strong
        if weak_sqp is not None:
            out["weak_sqp"] = weak_sqp
        if args.extras and (world == 1 or args.extras > 1):
            out["extras"] = run_extras(local_rank, hbm_peak)
        print(json.dumps(out))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def run_strong(args, rank, world, local_rank, dist, N=None, scaling="strong"):
    """BASELINE.json configs[4], strong scaling: a fixed N = args.strong HS071 instances (perturbed starts, SURVEY 8d config 5)
    sharded contiguously by instance index over the ranks; each rank runs the device-resident SQP loop on its shard (no collective
    on the path).  Timed with CUDA events around reset (upload of the shard's starts + evaluation + state) and Optimize, after two
    warm-up batches on the same object; max over ranks, median of three repetitions."""
    import torch
    try:
        from restartsqp_b200 import sharding
        from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
        from restartsqp_b200.sqp_device import DeviceBatchedSQP
        N = int(args.strong) if N is None else int(N)
        host = AmplNLP(os.path.join(ROOT, "tests", "golden", "hs_nl", "hs071.nl"))
        dev = DeviceNLP(host, device=local_rank)
        lo, hi = sharding.shard_range(N, rank, world)
        X = perturbed_starts(host, N, 0)[lo:hi]
        alg = DeviceBatchedSQP(dev, x0=X, device=local_rank)
        # two warm-up batches: the handles learn their factor capacity in the first, and the kernel configuration chosen from it
        # is first used (and its module loaded) in the second
        alg.Optimize()
        alg.reset(X)
        alg.Optimize()
        reps, times = 3, []
        for _ in range(reps):
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            alg.reset(X)
            res = alg.Optimize()
            e1.record()
            torch.cuda.synchronize()
            tm = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
            if dist is not None:
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            times.append(float(tm.item()))
        t = torch.tensor([0.0, float((res.exitflag == 0).sum()), float(res.iters.sum())], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(t[1:], op=dist.ReduceOp.SUM)
        alg.close(); dev.close()
        ms = sorted(times)[reps // 2]
        return {"metric": "SQP solves/sec", "config": "10^6-scale HS071 instances sharded by instance index (BASELINE.json configs[4])",
                "scaling": scaling, "instances": N, "per_rank": hi - lo, "n_gpus": world, "ms": ms, "value": N / (ms * 1e-3), "unit": "solves/s",
                "optimal": int(t[1].item()), "sqp_iters_mean": float(t[2].item()) / N,
                "ms_all": times,
                "timing": "CUDA events around reset(x0) + Optimize on every rank, max over ranks, median of 3 repetitions (all in ms_all); handles and the "
                          "compiled NLP are created once before, two warm-up batches"}
    except Exception as e:  # never takes the headline down
        return {"error": repr(e)[:300]}


def run_extras(device, hbm_peak):
    """Side measurements on rank 0 (outside the timed region of the headline metric): the other BASELINE.json configurations
    that fit one GPU, each through the public API, each with its own CPU-oracle figure."""
    import restartsqp_b200 as r
    from restartsqp_b200 import capi
    from restartsqp_b200.nl_reader import AmplNLP, DeviceNLP
    from restartsqp_b200.sqp_device import DeviceBatchedSQP
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as H
    ex = {}

    def sqp_case(name, k, Bs, cpu_B=None, reps=3):
        """Full SQP solves/s on `name` x Bs perturbed starts: (a) construction + Optimize of a fresh object, like the reference times
        itself (initialization + Optimize, src/Algorithm.cpp:57); (b) the same object serving further batches (reset + Optimize)."""
        host = AmplNLP(os.path.join(ROOT, "tests", "golden", "hs_nl", name + ".nl"))
        dev = DeviceNLP(host, device=device)
        X = perturbed_starts(host, Bs, k)
        w = DeviceBatchedSQP(dev, x0=X[:min(Bs, 256)], device=device); w.Optimize(); w.close()
        t0 = time.perf_counter()
        alg = DeviceBatchedSQP(dev, x0=X, device=device)
        res = alg.Optimize()
        t_fresh = time.perf_counter() - t0
        reuse = []
        for _ in range(reps):
            t0 = time.perf_counter()
            alg.reset(X)
            res = alg.Optimize()
            reuse.append(time.perf_counter() - t0)
        alg.close(); dev.close()
        t_re = float(np.median(reuse))
        out = {"metric": "SQP solves/sec", "n": host.n, "m": host.m, "instances": Bs, "value": Bs / t_re, "unit": "solves/s",
               "seconds": t_re, "seconds_fresh_object": t_fresh, "value_fresh_object": Bs / t_fresh,
               "optimal": int((res.exitflag == 0).sum()), "sqp_iters_mean": float(res.iters.mean()), "qp_iters_mean": float(res.qp_iter.mean())}
        if cpu_B:
            try:  # the same solves by the CPU oracle's C restatement of the outer loop on all host cores
                from oracle import oracle_py as orc
                so = orc.SqpOracle(host, r.Options())
                Xc = np.tile(X, ((cpu_B + Bs - 1) // Bs, 1))[:cpu_B]
                so.solve_batch(Xc[:min(cpu_B, 2000)])
                t0 = time.perf_counter()
                rc_ = so.solve_batch(Xc)
                tc = time.perf_counter() - t0
                out["cpu_baseline"] = {"value": cpu_B / tc, "unit": "solves/s", "cores": int(rc_["threads"]), "kind": "port",
                                       "sample": "%d solves in %.2f s (oracle/oracle_sqp.c)" % (cpu_B, tc), "optimal": int((rc_["exitflag"] == 0).sum())}
            except Exception as e:
                out["cpu_baseline"] = {"error": repr(e)[:200]}
        return out

    try:  # configs[0]/[2]: HS071 x 10^4 and (configs[4] at one GPU) x 10^6
        ex["sqp_hs071"] = sqp_case("hs071", 0, 10000, cpu_B=100000)
        ex["sqp_hs071"]["note"] = ("device-resident outer loop (sqpb200_sqp_optimize: csrc/sqp_outer.cu), NVRTC NLP evaluation and every QP/LP on the GPU; "
                                   "starts uploaded from the host, results read back; wall clock; value = one object serving batch after batch")
        ex["sqp_hs071_1e6"] = sqp_case("hs071", 0, 1000000, reps=2)
    except Exception as e:
        ex["sqp_hs071"] = {"error": repr(e)[:200]}
    try:  # the same 10^4 HS071 solves through the C++ host driver (csrc/driver/BatchedAlgorithm.cpp + batched_sqp), no Python in the loop
        import subprocess
        import tempfile
        from restartsqp_b200.nl_reader import write_model_file
        exe = os.path.join(ROOT, "restartsqp_b200", "lib", "batched_sqp")
        host = AmplNLP(os.path.join(ROOT, "tests", "golden", "hs_nl", "hs071.nl"))
        with tempfile.TemporaryDirectory() as td:
            mf = os.path.join(td, "hs071.model")
            write_model_file(host, mf, perturbed_starts(host, 10000, 0))
            p = subprocess.run([exe, mf, "--quiet", "--repeat", "3"], capture_output=True, text=True, timeout=120)
        if p.returncode != 0:
            raise RuntimeError((p.stdout + p.stderr)[-200:])
        t = p.stdout.strip().splitlines()[-1].split()
        kv = dict(zip(t[1::2], t[2::2]))
        ex["sqp_hs071_cpp_driver"] = {"metric": "SQP solves/sec", "instances": int(kv["instances"]), "optimal": int(kv["optimal"]),
                                      "value": float(kv["solves_per_s"]), "unit": "solves/s", "optimize_ms": float(kv["optimize_ms"]),
                                      "note": "restartsqp_b200/lib/batched_sqp: BatchedAlgorithm::Optimize of the third batch on one object, "
                                              "CUDA events around the call (starts already uploaded by reset)"}
    except Exception as e:
        ex["sqp_hs071_cpp_driver"] = {"error": repr(e)[:200]}
    try:  # configs[2]: a slice of the HS suite, 10^4 perturbed starts per problem, CPU figure per problem
        rows, tg, tc, ninst, nopt = {}, 0.0, 0.0, 0, 0
        for k, name in enumerate(HS_SLICE):
            try:
                c = sqp_case(name, k, 10000, cpu_B=10000, reps=1)
                rows[name] = {"n": c["n"], "m": c["m"], "solves_per_s": c["value"], "optimal": c["optimal"], "sqp_iters_mean": c["sqp_iters_mean"],
                              "cpu_solves_per_s": c.get("cpu_baseline", {}).get("value"), "cpu_optimal": c.get("cpu_baseline", {}).get("optimal")}
                tg += c["seconds"]; ninst += 10000; nopt += c["optimal"]
                if rows[name]["cpu_solves_per_s"]:
                    tc += 10000 / rows[name]["cpu_solves_per_s"]
            except Exception as e:
                rows[name] = {"error": repr(e)[:120]}
        ex["hs_suite_1e4"] = {"metric": "SQP solves/sec", "problems": len(rows), "instances": ninst, "optimal": nopt, "value": ninst / tg if tg else None,
                              "unit": "solves/s", "cpu_baseline": {"value": ninst / tc if tc else None, "unit": "solves/s", "kind": "port"}, "per_problem": rows}
    except Exception as e:
        ex["hs_suite_1e4"] = {"error": repr(e)[:200]}
    try:  # configs[3]: synthetic sparse QPs on the cluster kernel (TMA-staged FP64 DMMA refactorisation)
        lg = {}
        for n, Bq, cpu_n in ((256, 64, 16), (512, 16, 0), (1024, 16, 0)):
            d = H.synthetic_large_qp(n, batch=Bq)
            s = r.CudaQPInterface(nV=d["nV"], nC=d["nC"], qptype=r.QPType.QP, batch=Bq, device=device, keep_state=False,
                                  options=r.Options(qp_maxiter=max(1000, 6 * n)))
            s.set_csc(capi.MAT_A, *d["Ac"]); s.set_csc(capi.MAT_H, *d["Hc"])
            s.set_g(d["g"]); s.set_lb(d["lb"]); s.set_ub(d["ub"]); s.set_lbA(d["lbA"]); s.set_ubA(d["ubA"])
            for _ in range(2 if n <= 512 else 1):
                s._solve(r.QPType.QP, None, None, 0)
                ms = s.last_solve_ms()
            st, it = s.get_status(), s.get_iterations()
            kk = s.get_optimality_status()["KKT_error"]
            row = {"metric": "QP subproblems/sec", "value": Bq / (ms * 1e-3), "unit": "QPs/s", "batch": Bq, "nV": d["nV"], "nC": d["nC"], "ms": ms,
                   "optimal": int((st == 20).sum()), "iters_mean": float(it.mean()), "kkt_error_max": float(kk.max())}
            s.close()
            if cpu_n:
                from oracle import oracle_py as orc
                t0 = time.perf_counter()
                rr = orc.solve_batch(d["nV"], d["nC"], d["Ac"], d["Hc"], d["g"][:cpu_n], d["lb"][:cpu_n], d["ub"][:cpu_n], d["lbA"][:cpu_n], d["ubA"][:cpu_n])
                tcpu = time.perf_counter() - t0
                row["cpu_baseline"] = {"value": cpu_n / tcpu, "unit": "QPs/s", "cores": rr["threads"], "kind": "port", "sample": "%d instances in %.1f s" % (cpu_n, tcpu)}
            else:
                row["cpu_baseline"] = {"value": None, "note": "not run in the bench: the scalar oracle needs ~50 s per instance at n = 512 (tools/large_try.py checks instances against it)"}
            lg["n%d" % n] = row
        ex["large_qp"] = lg
    except Exception as e:
        ex["large_qp"] = {"error": repr(e)[:200]}
    try:
        ex["l0"] = run_l0(device, hbm_peak)
    except Exception as e:
        ex["l0"] = {"error": repr(e)[:200]}
    return ex


def run_l0(device, peak):
    """HBM roofline of the L0 kernels (SURVEY.md 8d): batched SpMV / SpMTV (A7), value scatter (A6), QP data construction (B2/B3),
    stand-alone KKT test (C8) and segmented triplet -> CSC assembly (A4/A5), on the hs116 shape.  Device-resident inputs and outputs,
    CUDA events around back-to-back launches, algorithmic bytes per unit as in SURVEY 8d; working sets far above the 126 MB L2."""
    import torch
    import restartsqp_b200 as r
    from restartsqp_b200 import capi
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as H
    L = capi.lib()
    dev = torch.device("cuda", device)
    out = {"peak_gbs": peak, "shape": "hs116 (nV=69, nC=28)"}

    def timed(fn, reps=5):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    def row(name, bytes_, ms):
        gbs = bytes_ / (ms * 1e-3) / 1e9
        out[name] = {"algorithmic_mb": bytes_ / 1e6, "ms": ms, "gbs": gbs, "frac": gbs / peak}

    q = [f for f in H.load_qp_fixtures() if f["name"] == "QORE_hs116"][0]
    nV, nC, n, m, B = q["nV"], q["nC"], 13, 28, 1 << 18
    Ac, Hc = (q["A_colptr"], q["A_rowidx"]), (q["H_colptr"], q["H_rowidx"])
    zA, zH = len(Ac[1]), len(Hc[1])
    s = r.CudaQPInterface(nV=nV, nC=nC, qptype=r.QPType.QP, batch=B, device=device, keep_state=False)
    g = torch.Generator(device=dev); g.manual_seed(1)
    rnd = lambda *sh: torch.randn(*sh, dtype=torch.float64, device=dev, generator=g)
    s.set_csc(capi.MAT_A, Ac[0], Ac[1], rnd(B, zA)); s.set_csc(capi.MAT_H, Hc[0], Hc[1], rnd(B, zH))
    x, yc = rnd(B, nV), rnd(B, nC)
    oC, oV = torch.empty(B, nC, dtype=torch.float64, device=dev), torch.empty(B, nV, dtype=torch.float64, device=dev)
    p = lambda t: C.c_void_p(t.data_ptr())
    row("spmv_A_x", 8 * (zA + nV + nC) * B, timed(lambda: L.sqpb200_spmv(s.h, capi.MAT_A, 0, p(x), p(oC), capi.LOC_DEVICE)))
    row("spmtv_At_y", 8 * (zA + nV + nC) * B, timed(lambda: L.sqpb200_spmv(s.h, capi.MAT_A, 1, p(yc), p(oV), capi.LOC_DEVICE)))
    row("spmv_H_x", 8 * (zH + 2 * nV) * B, timed(lambda: L.sqpb200_spmv(s.h, capi.MAT_H, 0, p(x), p(oV), capi.LOC_DEVICE)))
    delta = torch.ones(B, dtype=torch.float64, device=dev); rho = torch.ones(B, dtype=torch.float64, device=dev)
    xl, xu, xk, cl, cu, ck, gr = rnd(B, n), rnd(B, n), rnd(B, n), rnd(B, m), rnd(B, m), rnd(B, m), rnd(B, n)
    row("qphandler_bounds", 8 * (3 * n + 3 * m + 1 + 2 * nV + 2 * nC) * B,
        timed(lambda: L.sqpb200_qphandler_bounds(s.h, 0, n, m, p(delta), p(xl), p(xu), p(xk), p(cl), p(cu), p(ck), capi.LOC_DEVICE)))
    row("qphandler_g", 8 * (n + 1 + nV) * B, timed(lambda: L.sqpb200_qphandler_g(s.h, n, m, p(gr), p(rho), capi.LOC_DEVICE)))
    o5 = torch.empty(B, 5, dtype=torch.float64, device=dev)
    kkt_bytes = 8 * (zA + zH + 5 * nV + 2 * nC + (nV + nC)) + 2 * (nV + nC) + 4 * (nV + nC) + 40
    row("kkt_test", kkt_bytes * B, timed(lambda: L.sqpb200_kkt_residuals_recompute(s.h, p(o5), capi.LOC_DEVICE)))
    out["kkt_test"]["data"] = "random vectors, x = y = 0 (dense violation terms)"
    s.close()
    # the same kernel where test_optimality runs it: at the solutions of the dumped hs116 QP (replicated and perturbed)
    Bk = 1 << 16
    d = make_batch(q, Bk, 4242)
    sk = r.CudaQPInterface(nV=nV, nC=nC, qptype=r.QPType.QP, batch=Bk, device=device, keep_state=False)
    sk.set_csc(capi.MAT_A, q["A_colptr"], q["A_rowidx"], d["Av"]); sk.set_csc(capi.MAT_H, q["H_colptr"], q["H_rowidx"], d["Hv"])
    sk.set_g(d["g"]); sk.set_lb(d["lb"]); sk.set_ub(d["ub"]); sk.set_lbA(d["lbA"]); sk.set_ubA(d["ubA"])
    sk._solve(r.QPType.QP, None, None, 0)
    o5k = torch.empty(Bk, 5, dtype=torch.float64, device=dev)
    row("kkt_test_at_solution", kkt_bytes * Bk, timed(lambda: L.sqpb200_kkt_residuals_recompute(sk.h, p(o5k), capi.LOC_DEVICE)))
    out["kkt_test_at_solution"]["data"] = "2^16 perturbed replicas of the dumped hs116 QP, after the solve (the state test_optimality sees)"
    out["kkt_test_at_solution"]["kkt_error_max"] = float(o5k[:, 4].max().item())
    sk.close()
    # value scatter through `order` (A6) and segmented assembly (A4/A5) on the Jacobian triplets of the same shape
    jr, jc = [], []
    for c in range(n):
        for e in range(q["A_colptr"][c], q["A_colptr"][c + 1]):
            jr.append(q["A_rowidx"][e] + 1); jc.append(c + 1)
    info = r.NLPInfo(nCon=m, nVar=n, nnz_jac_g=len(jr), nnz_h_lag=0)
    s2 = r.CudaQPInterface(info, r.QPType.LP, batch=B, device=device, keep_state=False)
    I = r.IdentityInfo(irow=np.array([1, 1], np.int32), jcol=np.array([n + 1, n + m + 1], np.int32), size=np.array([m, m], np.int32), value=np.array([1.0, -1.0]))
    vals = torch.randn(B, len(jr), dtype=torch.float64, device=dev)
    s2.set_A(r.SpTripletMat(np.array(jr, np.int32), np.array(jc, np.int32), vals, m, n, False), I)
    row("scatter_values", 20 * len(jr) * B, timed(lambda: L.sqpb200_set_values_A(s2.h, p(vals), capi.LOC_DEVICE, 0)))
    s2.close()
    nmat, z = 1 << 15, len(jr) + 2 * m
    er = np.concatenate([jr, 1 + np.arange(m), 1 + np.arange(m)]).astype(np.int32); ec = np.concatenate([jc, n + 1 + np.arange(m), n + m + 1 + np.arange(m)]).astype(np.int32)
    row1, col1 = np.tile(er, nmat), np.tile(ec, nmat)
    seg = (np.arange(nmat + 1) * z).astype(np.int32); ncol = np.full(nmat, n + 2 * m, np.int32)
    colptr, rowidx, order = np.zeros(nmat * (n + 2 * m + 1), np.int32), np.zeros(nmat * z, np.int32), np.zeros(nmat * z, np.int32)
    ms = C.c_float(0)
    ip = lambda a: a.ctypes.data_as(C.c_void_p)
    for _ in range(2):
        rc = L.sqpb200_assemble_csc_batched(device, nmat, ip(seg), ip(ncol), ip(row1), ip(col1), ip(colptr), ip(rowidx), ip(order), C.byref(ms))
    if rc == 0:
        row("csc_assembly", (28 * z + 4 * (n + 2 * m + 1)) * nmat, ms.value)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--replicas", type=int, default=4096, help="replicas per dumped QP (B of SURVEY.md 8d config 2)")
    ap.add_argument("--team", type=int, default=0, help="threads per QP (0 = auto)")
    ap.add_argument("--extras", type=int, default=1, help="1: the other BASELINE configs on rank 0 when run on one GPU; 2: also under torchrun; 0: off")
    ap.add_argument("--strong", type=int, default=1000000, help="instances of the strong-scaling block (configs[4]); 0: off")
    ap.add_argument("--e2e-overlap", type=int, default=1, help="1: the end-to-end path alternates two handle sets (consecutive steps overlap); 0: one step at a time")
    ap.add_argument("--streams", type=int, default=1, help="1: one CUDA stream per dumped QP (overlapping launches), 0: default stream")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the solutions of the last one as DIR/<dump>_<array>.npy (rank 0; float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's solutions; --impl reference has none to write")
    rank =int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()

"""GPU parity for the active-set QP/LP kernel (row D) through the C ABI: the CUDA path against the CPU
oracle on the same inputs.  Gates (BASELINE.md section 4): identical final working sets (raw qpOASES
convention), identical status and iteration counts, x / y / objective within 1e-8 relative; KKT residuals
of the fused epilogue against the oracle's restatement of test_optimality."""
import numpy as np
import pytest

import restartsqp_b200 as r
from restartsqp_b200 import capi
from oracle import oracle_py as orc
import helpers as H

pytestmark = pytest.mark.gpu
RTOL = 1.0e-8
FIX = H.load_qp_fixtures()


def relerr(a, b):
    return float(np.abs(a - b).max() / max(1.0, np.abs(b).max())) if a.size else 0.0


def solve_batch_csc(nV, nC, Acsc, Hcsc, g, lb, ub, lbA, ubA, qptype=r.QPType.QP, team_size=0, Avals=None, Hvals=None, factor_cap=0):
    """g, lb, ... are [batch][len]; Acsc/Hcsc = (colptr,rowidx,val[z]) shared, Avals/Hvals optional [batch][z]."""
    B = g.shape[0]
    s = r.CudaQPInterface(nV=nV, nC=nC, qptype=qptype, batch=B, team_size=team_size, factor_cap=factor_cap)
    s.set_csc(capi.MAT_A, Acsc[0], Acsc[1], Acsc[2] if Avals is None else Avals)
    if qptype == r.QPType.QP:
        s.set_csc(capi.MAT_H, Hcsc[0], Hcsc[1], Hcsc[2] if Hvals is None else Hvals)
    s.set_g(g); s.set_lb(lb); s.set_ub(ub)
    if nC:
        s.set_lbA(lbA); s.set_ubA(ubA)
    if qptype == r.QPType.QP:
        s.optimizeQP() if B > 1 else s._solve(r.QPType.QP, None, None, 0)
    else:
        s.optimizeLP() if B > 1 else s._solve(r.QPType.LP, None, None, 0)
    return s


def check_against_oracle(s, b, o, nV, strict=True):
    x, y = s.get_optimal_solution()[b], np.concatenate([s.get_multipliers_bounds()[b], s.get_multipliers_constr()[b]])
    wc, wb = s.get_working_set(translated=False)
    assert int(s.get_status()[b]) == o["status"]
    assert int(s.get_iterations()[b]) == o["iters"]
    assert (wb[b] == o["wb"]).all() and (wc[b] == o["wc"]).all(), "working sets differ"
    if strict:
        assert relerr(x, o["x"]) <= RTOL and relerr(y, o["y"]) <= RTOL
        assert abs(s.get_obj_value()[b] - o["obj"]) <= RTOL * max(1.0, abs(o["obj"]))


# The library is built with -fmad=false and the kernel evaluates every sum in the oracle's order, so even the
# degenerate non-convex dumps (hs056, hs107: ~70 bound flips) follow the oracle's path bit for bit.
PATH_DEPENDENT = set()


@pytest.mark.parametrize("q", FIX, ids=[q["name"] for q in FIX])
def test_dumped_qp_replay_matches_oracle(gpu_lib, q):
    nV, nC = q["nV"], q["nC"]
    B = 4
    rng = np.random.default_rng(1234)
    g = np.tile(np.array(q["g"]), (B, 1))
    g[1:] *= 1.0 + 1e-3 * rng.uniform(-1, 1, size=g[1:].shape)  # SURVEY.md 8(d) config 2: replica 0 exact
    tile = lambda k, n_: np.tile(np.array(q[k], dtype=np.float64).reshape(1, n_), (B, 1))
    A = (q["A_colptr"], q["A_rowidx"], np.array(q["A_val"]))
    Hc = (q["H_colptr"], q["H_rowidx"], np.array(q["H_val"]))
    s = solve_batch_csc(nV, nC, A, Hc, g, tile("lb", nV), tile("ub", nV), tile("lbA", nC), tile("ubA", nC))
    st = s.get_status()
    assert ((st >= 20) & (st <= 30)).all()
    assert np.isfinite(s.get_optimal_solution()).all()
    if q["name"] in PATH_DEPENDENT:
        s.close()
        return
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=q["lb"], ub=q["ub"], lbA=q["lbA"], ubA=q["ubA"])
        o = H.oracle_solve(orc, p, Acsc=A, Hcsc=Hc)
        check_against_oracle(s, b, o, nV, strict=(o["status"] == 20))
    # fused KKT epilogue == stand-alone kernel == oracle restatement of test_optimality (replica 0)
    k_fused = s.get_optimality_status()["KKT_error"].copy()
    k_alone = s.get_optimality_status(recompute=True)
    p = dict(nV=nV, nC=nC, g=g[0], lb=q["lb"], ub=q["ub"], lbA=q["lbA"], ubA=q["ubA"])
    o = H.oracle_solve(orc, p, Acsc=A, Hcsc=Hc)
    if H.is_symmetric_fixture(q) and o["status"] == 20:
        x, y = s.get_optimal_solution()[0], np.concatenate([s.get_multipliers_bounds()[0], s.get_multipliers_constr()[0]])
        wc, wb = s.get_working_set(translated=False)
        Ax = orc.csc_times(nC, nV, *A, x)
        Wb, Wc = orc.translate_working_set(wb[0], wc[0], x, Ax, q["lb"], q["ub"], q["lbA"], q["ubA"])
        ok, res = orc.kkt_residuals(nV, nC, A, Hc, g[0], q["lb"], q["ub"], q["lbA"], q["ubA"], x, y, Wb, Wc)
        # stand-alone kernel: bit-exact with the restated reference formulas on the same (x, y, W)
        assert [k_alone[k][0] for k in ("primal_violation", "dual_violation", "stationarity_violation",
                                        "compl_violation", "KKT_error")] == res.tolist()
        WcT, WbT = s.get_working_set(translated=True)
        assert (WbT[0] == Wb).all() and (WcT[0] == Wc).all()
        scale = max(1.0, np.abs(y).max() * max(1.0, np.abs(x).max()))
        assert abs(k_fused[0] - res[4]) <= 1e-10 * scale
    s.close()


@pytest.mark.parametrize("team", [0, 32, 1024])
def test_random_convex_batch_all_team_sizes(gpu_lib, team):
    rng = np.random.default_rng(72 + team)
    n, m = 6, 4
    base = H.random_l1_qp(rng, n, m, convex=True, dens=0.7)
    nV, nC, B = base["nV"], base["nC"], 64
    Ac, Hc = H.csc(base["A"]), H.csc(base["H"])
    Avals = np.tile(Ac[2], (B, 1))
    Avals *= 1.0 + 0.1 * rng.standard_normal(Avals.shape) * (np.abs(np.abs(Avals) - 1.0) > 1e-12)  # keep the +-1 slack columns
    Hvals = np.tile(Hc[2], (B, 1))
    g = np.tile(base["g"], (B, 1)); g[:, :n] += rng.standard_normal((B, n))
    lbA = np.tile(base["lbA"], (B, 1)); ubA = np.tile(base["ubA"], (B, 1))
    shift = 0.5 * rng.standard_normal((B, m))
    lbA = np.where(lbA > -1e17, lbA + shift, lbA); ubA = np.where(ubA < 1e17, ubA + shift, ubA)
    lb, ub = np.tile(base["lb"], (B, 1)), np.tile(base["ub"], (B, 1))
    s = solve_batch_csc(nV, nC, Ac, Hc, g, lb, ub, lbA, ubA, team_size=team, Avals=Avals, Hvals=Hvals)
    # auto: nV = 14 runs on 16-lane sub-warp teams (two QPs per warp); 32 forces one warp per QP; 1024 one CTA (cluster) per QP
    assert s.solve_config()["team_size"] == {0: 16, 32: 32, 1024: 1024}[team]
    assert (s.get_status() == 20).all()
    assert s.test_optimality().all()
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b])
        o = H.oracle_solve(orc, p, Acsc=(Ac[0], Ac[1], Avals[b]), Hcsc=(Hc[0], Hc[1], Hvals[b]))
        check_against_oracle(s, b, o, nV)
    s.close()


@pytest.mark.parametrize("shape", [(1, 0), (2, 1), (4, 2), (10, 7), (23, 12), (30, 20)])
def test_random_shapes_incl_edge_cases(gpu_lib, shape):
    """n=1 / no constraints / nV above one warp's lane count; per-instance data, shared pattern."""
    n, m = shape
    rng = np.random.default_rng(1000 + 31 * n + m)
    base = H.random_l1_qp(rng, n, m, convex=True, dens=0.5)
    nV, nC, B = base["nV"], base["nC"], 8
    Ac, Hc = H.csc(base["A"]), H.csc(base["H"])
    g = np.tile(base["g"], (B, 1)); g[:, :n] += rng.standard_normal((B, n))
    lb, ub = np.tile(base["lb"], (B, 1)), np.tile(base["ub"], (B, 1))
    lbA, ubA = np.tile(base["lbA"], (B, 1)), np.tile(base["ubA"], (B, 1))
    s = solve_batch_csc(nV, nC, Ac, Hc, g, lb, ub, lbA, ubA)
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b])
        check_against_oracle(s, b, H.oracle_solve(orc, p, Acsc=Ac, Hcsc=Hc), nV)
    s.close()


@pytest.mark.parametrize("team", [0, 1024])
def test_lp_matches_oracle(gpu_lib, team):
    rng = np.random.default_rng(77)
    n, m, B = 5, 4, 16
    base = H.random_l1_qp(rng, n, m, rho=1.0)
    nV, nC = base["nV"], base["nC"]
    Ac = H.csc(base["A"])
    g = np.tile(base["g"], (B, 1)); g[:, :n] = 0.0
    lb, ub = np.tile(base["lb"], (B, 1)), np.tile(base["ub"], (B, 1))
    lbA, ubA = np.tile(base["lbA"], (B, 1)), np.tile(base["ubA"], (B, 1))
    shift = rng.standard_normal((B, m))
    lbA = np.where(lbA > -1e17, lbA + shift, lbA); ubA = np.where(ubA < 1e17, ubA + shift, ubA)
    s = solve_batch_csc(nV, nC, Ac, None, g, lb, ub, lbA, ubA, qptype=r.QPType.LP, team_size=team)
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b], A=base["A"])
        o = H.oracle_solve(orc, p, is_lp=True, max_iter=100, Acsc=Ac)
        check_against_oracle(s, b, o, nV)
    s.close()


@pytest.mark.parametrize("team", [0, 1024])
def test_hotstart_fixed_and_varied(gpu_lib, team):
    """hotstart(g,lb,ub,lbA,ubA) and hotstart(H,g,A,...) (src/qpOASESInterface.cpp:176-211) against the
    oracle's hot starts, and against cold starts on the new data (strictly convex => same point)."""
    rng = np.random.default_rng(9)
    n, m, B = 5, 3, 12
    base = H.random_l1_qp(rng, n, m, convex=True)
    nV, nC = base["nV"], base["nC"]
    Ac, Hc = H.csc(base["A"]), H.csc(base["H"])
    g = np.tile(base["g"], (B, 1)); g[:, :n] += rng.standard_normal((B, n))
    lb, ub = np.tile(base["lb"], (B, 1)), np.tile(base["ub"], (B, 1))
    lbA, ubA = np.tile(base["lbA"], (B, 1)), np.tile(base["ubA"], (B, 1))
    s = solve_batch_csc(nV, nC, Ac, Hc, g, lb, ub, lbA, ubA, team_size=team)
    oracles = []
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b])
        o = H.oracle_solve(orc, p, Acsc=Ac, Hcsc=Hc)
        check_against_oracle(s, b, o, nV)
        oracles.append(o["solver"])
    # 1) vectors only -> FIXED hot start
    g2 = g.copy(); g2[:, :n] += 0.3 * rng.standard_normal((B, n))
    lbA2 = np.where(lbA > -1e17, lbA - 0.2, lbA); ubA2 = np.where(ubA < 1e17, ubA + 0.1, ubA)
    s.set_g(g2); s.set_lbA(lbA2); s.set_ubA(ubA2)
    s.optimizeQP()
    for b in range(B):
        st = oracles[b].hotstart(g2[b], lb[b], ub[b], lbA2[b], ubA2[b])
        x, y, obj, it = oracles[b].solution(); wb, wc = oracles[b].working_set()
        check_against_oracle(s, b, dict(x=x, y=y, obj=obj, iters=it, status=st, wb=wb, wc=wc), nV)
    # 2) new matrix values: the FIXED -> VARIED flip is an init from the previous solution (:202-207), the solve after it a
    #    VARIED hot start, hotstart(H, g, A, ...) (:184-188)
    Hv2 = np.tile(Hc[2], (B, 1))
    Av2 = np.tile(Ac[2], (B, 1))
    for k, call in enumerate(("reinit", "hotstart_matrices", "hotstart_matrices")):
        Hv2 = Hv2 * 1.1
        g2 = g2.copy(); g2[:, :n] += 0.1 * rng.standard_normal((B, n))
        s.set_csc_values(capi.MAT_H, Hv2); s.set_csc_values(capi.MAT_A, Av2); s.set_g(g2)
        s.optimizeQP()
        for b in range(B):
            st = getattr(oracles[b], call)(Hv2[b], Av2[b], g2[b], lb[b], ub[b], lbA2[b], ubA2[b])
            x, y, obj, it = oracles[b].solution(); wb, wc = oracles[b].working_set()
            check_against_oracle(s, b, dict(x=x, y=y, obj=obj, iters=it, status=st, wb=wb, wc=wc), nV)
            p = dict(nV=nV, nC=nC, g=g2[b], lb=lb[b], ub=ub[b], lbA=lbA2[b], ubA=ubA2[b])
            cold = H.oracle_solve(orc, p, Acsc=Ac, Hcsc=(Hc[0], Hc[1], Hv2[b]))
            assert relerr(s.get_optimal_solution()[b], cold["x"]) <= RTOL
    s.close()


def test_qphandler_solveQP_and_reference_exceptions(gpu_lib):
    """QPhandler::solveQP (src/QPhandler.cpp:470-499) through triplets + IdentityInfo, batch == 1 semantics."""
    n, m = 4, 2  # HS071 shape: x0 = (1,5,5,1), 1<=x<=5, c1>=25, c2=40
    x_k = np.array([1.0, 5.0, 5.0, 1.0])
    hnd = r.QPhandler(r.NLPInfo(nCon=m, nVar=n, nnz_jac_g=8, nnz_h_lag=10), r.QPType.QP, batch=1)
    jr, jc = [1, 2] * 4, [1, 1, 2, 2, 3, 3, 4, 4]
    c1 = lambda x: x[0] * x[1] * x[2] * x[3]
    J = np.array([[x_k[1] * x_k[2] * x_k[3], x_k[0] * x_k[2] * x_k[3], x_k[0] * x_k[1] * x_k[3], x_k[0] * x_k[1] * x_k[2]],
                  2 * x_k])
    jv = np.array([J[r_ - 1, c_ - 1] for r_, c_ in zip(jr, jc)])
    hr, hc = [1, 1, 2, 1, 2, 3, 1, 2, 3, 4], [1, 2, 2, 3, 3, 3, 4, 4, 4, 4]
    Hd = np.array([[2 * x_k[3], x_k[3], x_k[3], 2 * x_k[0] + x_k[1] + x_k[2]], [0, 0, 0, x_k[0]], [0, 0, 0, x_k[0]], [0, 0, 0, 0]])
    Hd = np.triu(Hd) + np.triu(Hd, 1).T + 2.0 * np.eye(4)
    hv = np.array([Hd[r_ - 1, c_ - 1] for r_, c_ in zip(hr, hc)])
    grad = np.array([x_k[3] * (2 * x_k[0] + x_k[1] + x_k[2]), x_k[0] * x_k[3], x_k[0] * x_k[3] + 1, x_k[0] * (x_k[0] + x_k[1] + x_k[2])])
    c_k = np.array([c1(x_k), (x_k ** 2).sum()])
    hnd.set_bounds(1.0, np.ones(4), 5 * np.ones(4), x_k, np.array([25.0, 40.0]), np.array([1e18, 40.0]), c_k)
    hnd.set_g(grad, 1.0)
    hnd.set_A(r.SpTripletMat(np.array(jr), np.array(jc), jv, m, n))
    hnd.set_H(r.SpTripletMat(np.array(hr), np.array(hc), hv, n, n, True))
    stats = r.Stats()
    ok = hnd.solveQP(stats)
    assert ok.all() and int(hnd.get_status()[0]) == 20 and stats.qp_iter[0] > 0
    # same QP through the oracle
    I = orc.identity_info(n, m)
    A = orc.assemble_A(m, n + 2 * m, jr, jc, jv, I)
    Hh = orc.assemble_H(n + 2 * m, hr, hc, hv, True)
    si = hnd.solverInterface_
    p = dict(nV=n + 2 * m, nC=m, g=si.getG()[0], lb=si.getLb()[0], ub=si.getUb()[0], lbA=si.getLbA()[0], ubA=si.getUbA()[0])
    o = H.oracle_solve(orc, p, Acsc=A[:3], Hcsc=Hh[:3])
    check_against_oracle(si, 0, o, n + 2 * m)
    assert abs(hnd.get_infea_measure_model()[0] - orc.lib().orc_infea_measure_model(n, m, orc._dp(o["x"]))) < 1e-12
    assert abs(hnd.get_objective()[0] - o["obj"]) <= RTOL * max(1, abs(o["obj"]))
    # batch == 1 raises like the reference when the QP cannot be solved (max iterations exhausted)
    si2 = r.CudaQPInterface(r.NLPInfo(nCon=m, nVar=n), r.QPType.QP, r.Options(qp_maxiter=1), batch=1)
    si2.set_A(r.SpTripletMat(np.array(jr), np.array(jc), jv, m, n), hnd.I_info_A_)
    si2.set_H(r.SpTripletMat(np.array(hr), np.array(hc), hv, n, n, True))
    si2.set_g(p["g"]); si2.set_lb(p["lb"]); si2.set_ub(p["ub"]); si2.set_lbA(p["lbA"]); si2.set_ubA(p["ubA"])
    with pytest.raises(r.QP_NOT_OPTIMAL):
        si2.optimizeQP()
    assert int(si2.get_status()[0]) == int(r.Exitflag.QPERROR_PERFORMINGHOMOTOPY)
    si2.close(); si.close()


def test_active_mask_and_large_batch_properties(gpu_lib):
    """Size-independent properties at a large batch: every instance KKT-optimal by the reference's test;
    replicated inputs give bit-identical outputs; masked-out instances are untouched."""
    rng = np.random.default_rng(21)
    n, m, B = 8, 5, 20000
    base = H.random_l1_qp(rng, n, m, convex=True)
    nV, nC = base["nV"], base["nC"]
    Ac, Hc = H.csc(base["A"]), H.csc(base["H"])
    g = np.tile(base["g"], (B, 1)); g[: B // 2, :n] += rng.standard_normal((B // 2, n))
    g[B // 2:] = g[: B // 2]  # second half replicates the first
    lb, ub = np.tile(base["lb"], (B, 1)), np.tile(base["ub"], (B, 1))
    lbA, ubA = np.tile(base["lbA"], (B, 1)), np.tile(base["ubA"], (B, 1))
    s = r.CudaQPInterface(nV=nV, nC=nC, batch=B)
    s.set_csc(capi.MAT_A, *Ac); s.set_csc(capi.MAT_H, *Hc)
    s.set_g(g); s.set_lb(lb); s.set_ub(ub); s.set_lbA(lbA); s.set_ubA(ubA)
    mask = np.ones(B, np.uint8); mask[7] = 0
    s.optimizeQP(active_mask=mask)
    st, x = s.get_status(), s.get_optimal_solution()
    assert st[7] == int(r.Exitflag.QPERROR_NOTINITIALISED) and not x[7].any()
    keep = mask.astype(bool)
    assert (st[keep] == 20).all() and s.test_optimality()[keep].all()
    assert (x[: B // 2][keep[: B // 2]] == x[B // 2:][keep[: B // 2]]).all()
    for b in rng.integers(0, B // 2, 5):
        if b == 7:
            continue
        p = dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b])
        check_against_oracle(s, int(b), H.oracle_solve(orc, p, Acsc=Ac, Hcsc=Hc), nV)
    s.close()


@pytest.mark.parametrize("cap", [1, 3, -1])
def test_factor_capacity_rescue_path(gpu_lib, cap):
    """A factor capacity below the number of free variables the path needs must not change any result: the
    overflowing instances are re-solved by the rescue launch (cold and hot starts)."""
    rng = np.random.default_rng(123)
    n, m, B = 7, 4, 24
    base = H.random_l1_qp(rng, n, m, convex=True)
    nV, nC = base["nV"], base["nC"]
    Ac, Hc = H.csc(base["A"]), H.csc(base["H"])
    g = np.tile(base["g"], (B, 1)); g[:, :n] += rng.standard_normal((B, n))
    lb, ub = np.tile(base["lb"], (B, 1)), np.tile(base["ub"], (B, 1))
    lbA, ubA = np.tile(base["lbA"], (B, 1)), np.tile(base["ubA"], (B, 1))
    s = solve_batch_csc(nV, nC, Ac, Hc, g, lb, ub, lbA, ubA, factor_cap=cap)
    oracles, needs = [], 0
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b])
        o = H.oracle_solve(orc, p, Acsc=Ac, Hcsc=Hc)
        check_against_oracle(s, b, o, nV)
        oracles.append(o["solver"])
        needs = max(needs, orc.lib().orc_qp_get_max_free(o["solver"].h))
    if cap > 0:
        assert needs > cap, "test problem does not exercise the rescue path"
    g2 = g.copy(); g2[:, :n] += 0.5 * rng.standard_normal((B, n))
    s.set_g(g2)
    s.optimizeQP()
    for b in range(B):
        st = oracles[b].hotstart(g2[b], lb[b], ub[b], lbA[b], ubA[b])
        x, y, obj, it = oracles[b].solution(); wb, wc = oracles[b].working_set()
        check_against_oracle(s, b, dict(x=x, y=y, obj=obj, iters=it, status=st, wb=wb, wc=wc), nV)
    s.close()


@pytest.mark.parametrize("name", ["QORE_hs104", "QORE_hs107", "QORE_hs116"])
def test_dumped_qp_on_cta_per_qp_kernel(gpu_lib, name):
    """The one-QP-per-CTA kernel (slice in global memory) runs the same active-set code with the refactorisation on the
    FP64 tensor cores (DMMA accumulates in a different order than the oracle's scalar sums, and the factor is updated rather
    than recomputed after most additions).  Its gate is north_star's: same status, and where the oracle solves the QP the same objective to 1e-8 and
    a KKT point by the reference's own test.  On the rho = 1e8 scaled dump (hs104) the homotopy path is rounding-sensitive,
    so iteration counts may differ while the solution does not; the well-scaled hs116 must keep the oracle's working set."""
    q = [f for f in FIX if f["name"] == name][0]
    nV, nC, B = q["nV"], q["nC"], 3
    rng = np.random.default_rng(4321)
    g = np.tile(np.array(q["g"]), (B, 1)); g[1:] *= 1.0 + 1e-3 * rng.uniform(-1, 1, size=g[1:].shape)
    tile = lambda k, n_: np.tile(np.array(q[k], dtype=np.float64).reshape(1, n_), (B, 1))
    A = (q["A_colptr"], q["A_rowidx"], np.array(q["A_val"]))
    Hc = (q["H_colptr"], q["H_rowidx"], np.array(q["H_val"]))
    s = solve_batch_csc(nV, nC, A, Hc, g, tile("lb", nV), tile("ub", nV), tile("lbA", nC), tile("ubA", nC), team_size=1024)
    assert s.solve_config()["team_size"] == 1024
    st, obj = s.get_status(), s.get_obj_value()
    wc, wb = s.get_working_set(translated=False)
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=q["lb"], ub=q["ub"], lbA=q["lbA"], ubA=q["ubA"])
        o = H.oracle_solve(orc, p, Acsc=A, Hcsc=Hc)
        if o["status"] == 20:
            assert st[b] == 20
            assert abs(obj[b] - o["obj"]) <= RTOL * max(1.0, abs(o["obj"]))
            if name == "QORE_hs116":
                assert (wb[b] == o["wb"]).all() and (wc[b] == o["wc"]).all()
        else:
            assert 20 < st[b] <= 30
    s.close()


@pytest.mark.parametrize("n,B,checked", [(64, 8, 8), (128, 6, 3), (256, 4, 2)])
def test_synthetic_large_config4(gpu_lib, n, B, checked):
    """BASELINE.json configs[3] / SURVEY.md 8d config 4 (n variables, m = n/2, 1 % density, strictly convex): too large for
    the shared-memory kernel, solved by the one-QP-per-CTA kernel; identical working sets / iteration counts and x, y,
    objective within 1e-8 of the oracle; every instance passes the reference's own KKT test (1e-6)."""
    d = H.synthetic_large_qp(n, batch=B)
    nV, nC = d["nV"], d["nC"]
    s = solve_batch_csc(nV, nC, d["Ac"], d["Hc"], d["g"], d["lb"], d["ub"], d["lbA"], d["ubA"])
    assert s.solve_config()["team_size"] == 1024
    assert (s.get_status() == 20).all() and s.test_optimality().all()
    x = s.get_optimal_solution()
    assert (x[:, :n] >= -1.0 - 1e-12).all() and (x[:, :n] <= 1.0 + 1e-12).all() and (x[:, n:] >= -1e-12).all()
    for b in range(checked):
        p = dict(nV=nV, nC=nC, g=d["g"][b], lb=d["lb"][b], ub=d["ub"][b], lbA=d["lbA"][b], ubA=d["ubA"][b])
        o = H.oracle_solve(orc, p, Acsc=d["Ac"], Hcsc=d["Hc"], max_iter=100000)
        check_against_oracle(s, b, o, nV)
    s.close()


@pytest.mark.parametrize("n,B", [(96, 6), (200, 4)])
def test_cluster_kernel_factor_update_equals_recomputation(gpu_lib, n, B):
    """The one-QP-per-cluster kernel carries the projected Cholesky factor through additions (column rotations, row
    re-triangularisation, block inverses) and recomputes it every 64th addition; with refactorise_every = 1 it recomputes it
    after every addition, which is what qpOASES does under setToReliable and what the warp kernel and the oracle do.  Both are
    factors of the same matrix: same working sets and iteration counts, x and y to 1e-10, and both equal to the oracle."""
    d = H.synthetic_large_qp(n, batch=B)
    nV, nC = d["nV"], d["nC"]
    res = []
    for every in (0, 1):
        s = r.CudaQPInterface(nV=nV, nC=nC, qptype=r.QPType.QP, batch=B, team_size=1024, refactorise_every=every)
        s.set_csc(capi.MAT_A, *d["Ac"]); s.set_csc(capi.MAT_H, *d["Hc"])
        s.set_g(d["g"]); s.set_lb(d["lb"]); s.set_ub(d["ub"]); s.set_lbA(d["lbA"]); s.set_ubA(d["ubA"])
        s.optimizeQP()
        assert (s.get_status() == 20).all() and s.test_optimality().all()
        y = np.concatenate([s.get_multipliers_bounds(), s.get_multipliers_constr()], axis=1)
        res.append((s.get_optimal_solution().copy(), y, s.get_iterations().copy(), s.get_working_set(translated=False)))
        if every == 0:
            o = H.oracle_solve(orc, dict(nV=nV, nC=nC, g=d["g"][0], lb=d["lb"][0], ub=d["ub"][0], lbA=d["lbA"][0], ubA=d["ubA"][0]),
                               Acsc=d["Ac"], Hcsc=d["Hc"], max_iter=100000)
            check_against_oracle(s, 0, o, nV)
        s.close()
    (x0, y0, it0, ws0), (x1, y1, it1, ws1) = res
    assert (it0 == it1).all() and it0.min() > n // 2
    assert (ws0[0] == ws1[0]).all() and (ws0[1] == ws1[1]).all()
    assert relerr(x0, x1) <= 1e-10 and relerr(y0, y1) <= 1e-9


def _dense_case(nV, nC, Hd, A, g, lb, ub, lbA, ubA):
    return dict(nV=nV, nC=nC, H=np.asarray(Hd, float), A=np.asarray(A, float).reshape(nC, nV), g=np.asarray(g, float), lb=np.asarray(lb, float),
                ub=np.asarray(ub, float), lbA=np.asarray(lbA, float), ubA=np.asarray(ubA, float))


GENERIC_CASES = {
    # x0 + x1 >= 10 with 0 <= x <= 1
    "infeasible_bounds_vs_constraint": (_dense_case(2, 1, np.eye(2), [[1, 1]], [1, -1], [0, 0], [1, 1], [10], [1e18]), False, 22),
    # x0 >= 1 and x0 <= -1
    "infeasible_contradicting_rows": (_dense_case(2, 2, np.eye(2), [[1, 0], [1, 0]], [1, -1], [-5, -5], [5, 5], [1, -1e18], [1e18, -1]), False, 22),
    # indefinite H, "infinite" bounds of the reference (INF = 1e18 < qpOASES's 1e20: an ordinary finite bound, SURVEY 8a quirk 5)
    "indefinite_runs_to_the_1e18_bound": (_dense_case(2, 1, [[1, 0], [0, -1]], [[1, 1]], [0, 1], [-1e18] * 2, [1e18] * 2, [-1e18], [1e18]), False, 20),
    # LP without a finite minimiser: the eps-regularised problem has one
    "lp_unbounded_direction_regularised": (_dense_case(2, 1, np.zeros((2, 2)), [[1, 1]], [-1, 0], [0, 0], [1e18] * 2, [-1e18], [1e18]), True, 20),
}


@pytest.mark.parametrize("name", sorted(GENERIC_CASES))
@pytest.mark.parametrize("team", [0, 1024])
def test_infeasible_and_unbounded_qps_match_oracle(gpu_lib, name, team):
    """QPs outside the l1-penalty family: the Exitflag the backend must report (include/sqphot/Types.hpp:60-70, infeasible = 22)
    and the iterate it stops at, against the oracle, on both kernels."""
    p, is_lp, expect = GENERIC_CASES[name]
    nV, nC, B = p["nV"], p["nC"], 3
    Ac, Hc = H.csc(p["A"]), H.csc(p["H"] if not is_lp else np.zeros((nV, nV)))
    t = lambda v: np.ascontiguousarray(np.tile(v, (B, 1)))
    s = solve_batch_csc(nV, nC, Ac, None if is_lp else Hc, t(p["g"]), t(p["lb"]), t(p["ub"]), t(p["lbA"]), t(p["ubA"]),
                        qptype=r.QPType.LP if is_lp else r.QPType.QP, team_size=team)
    o = H.oracle_solve(orc, p, is_lp=is_lp, max_iter=100 if is_lp else 1000, Acsc=Ac, Hcsc=None if is_lp else Hc)
    assert o["status"] == expect
    for b in range(B):
        check_against_oracle(s, b, o, nV, strict=(expect == 20))
    s.close()


@pytest.mark.parametrize("team", [0, 1024])
def test_hotstart_state_is_bitwise_the_oracles(gpu_lib, team):
    """Regression: the KKT epilogue must not touch the solver's own Ax (part of the hot-start state).  A chain of
    hotstart(g, lb, ub, lbA, ubA) calls on fixed matrices has to stay bit-identical with the oracle, not just within 1e-8."""
    rng = np.random.default_rng(2024)
    n, m, B = 7, 6, 16
    base = H.random_l1_qp(rng, n, m, convex=True, dens=0.8)
    nV, nC = base["nV"], base["nC"]
    Ac, Hc = H.csc(base["A"]), H.csc(base["H"])
    g = np.tile(base["g"], (B, 1)); g[:, :n] += rng.standard_normal((B, n))
    t = lambda v: np.ascontiguousarray(np.tile(v, (B, 1)))
    lb, ub, lbA, ubA = t(base["lb"]), t(base["ub"]), t(base["lbA"]), t(base["ubA"])
    s = solve_batch_csc(nV, nC, Ac, Hc, g, lb, ub, lbA, ubA, team_size=team)
    solvers = []
    for b in range(B):
        o = H.oracle_solve(orc, dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b]), Acsc=Ac, Hcsc=Hc)
        solvers.append(o["solver"])
    for rnd in range(4):
        g = g.copy(); g[:, :n] += 0.4 * rng.standard_normal((B, n))
        lbA = np.where(lbA > -1e17, lbA + 0.1 * rng.standard_normal((B, m)), lbA)
        ubA = np.maximum(ubA, lbA)
        s.set_g(g); s.set_lbA(lbA); s.set_ubA(ubA)
        s.optimizeQP()
        x, it = s.get_optimal_solution(), s.get_iterations()
        yb, yc = s.get_multipliers_bounds(), s.get_multipliers_constr()
        for b in range(B):
            st = solvers[b].hotstart(g[b], lb[b], ub[b], lbA[b], ubA[b])
            xo, yo, _, ito = solvers[b].solution()
            assert st == int(s.get_status()[b])
            if team == 1024:  # CTA kernel: DMMA sums -> north_star's 1e-8 gate
                assert relerr(x[b], xo) <= RTOL and relerr(np.concatenate([yb[b], yc[b]]), yo) <= 10 * RTOL, (rnd, b)
            else:
                assert ito == int(it[b])
                assert np.array_equal(x[b], xo) and np.array_equal(np.concatenate([yb[b], yc[b]]), yo), (rnd, b)
    s.close()


def test_randomised_parity_stress(gpu_lib):
    """tools/qp_stress.py at a small size: random shapes, convex / non-convex / LP, cold + three hot starts, warp kernel with and
    without a tight factor capacity (rescue launch): bitwise against the oracle; the one-QP-per-CTA kernel at the 1e-8 gate."""
    import subprocess, sys, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "qp_stress.py"), "14", "7"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert " 0 mismatches" in out.stdout, out.stdout[-2000:]


@pytest.mark.parametrize("team", [0, 32, 1024])
def test_handle_error_infeasible_branch_forced(gpu_lib, team):
    """handle_error's infeasible branch (src/qpOASESInterface.cpp:716-729): re-init from the slack-feasible guess
    x0 = [0; max(0, lbA); -min(0, ubA)].  A feasible l1-penalty QP never reports INFEASIBLE, so the test hook
    debug_force_error_branch sends every instance through the branch after its first attempt.  The result must be (a) what the
    oracle's restatement of the same branch gives (bitwise on the warp kernels) and (b) the unique solution of the strictly convex
    QP, i.e. what the plain cold start found -- the branch is a different path to the same point."""
    rng = np.random.default_rng(515 + team)
    n, m, B = 6, 5, 24
    base = H.random_l1_qp(rng, n, m, convex=True, dens=0.8)
    nV, nC = base["nV"], base["nC"]
    Ac, Hc = H.csc(base["A"]), H.csc(base["H"])
    g = np.tile(base["g"], (B, 1)); g[:, :n] += rng.standard_normal((B, n))
    t = lambda v: np.ascontiguousarray(np.tile(v, (B, 1)))
    lb, ub, lbA, ubA = t(base["lb"]), t(base["ub"]), t(base["lbA"]), t(base["ubA"])
    shift = 0.5 * rng.standard_normal((B, m))
    lbA = np.where(lbA > -1e17, lbA + shift, lbA); ubA = np.where(ubA < 1e17, ubA + shift, ubA)
    s = r.CudaQPInterface(nV=nV, nC=nC, qptype=r.QPType.QP, batch=B, team_size=team, debug_force_error_branch=True)
    s.set_csc(capi.MAT_A, *Ac); s.set_csc(capi.MAT_H, *Hc)
    s.set_g(g); s.set_lb(lb); s.set_ub(ub); s.set_lbA(lbA); s.set_ubA(ubA)
    s.optimizeQP()
    assert (s.get_status() == 20).all() and s.test_optimality().all()
    x = s.get_optimal_solution()
    y = np.concatenate([s.get_multipliers_bounds(), s.get_multipliers_constr()], axis=1)
    it = s.get_iterations()
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b])
        o = H.oracle_solve(orc, p, Acsc=Ac, Hcsc=Hc, force_error_branch=True)
        plain = H.oracle_solve(orc, p, Acsc=Ac, Hcsc=Hc)
        assert o["status"] == 20
        if team != 1024:
            assert int(it[b]) == o["iters"] and np.array_equal(x[b], o["x"]) and np.array_equal(y[b], o["y"])
        assert relerr(x[b], plain["x"]) <= RTOL and relerr(y[b], plain["y"]) <= 10 * RTOL
        assert o["iters"] > plain["iters"]  # both attempts are counted (Stats::qp_iter, :752-753)
    s.close()


def test_failed_cold_start_counts_its_iterations_twice(gpu_lib):
    """src/qpOASESInterface.cpp:160-162, 746-754: a failed init is followed by handle_error's plain re-init -- the same
    deterministic solve again -- and the working-set changes of both runs are added to Stats::qp_iter."""
    q = [f for f in FIX if f["name"] == "QORE_hs107"][0]
    nV, nC = q["nV"], q["nC"]
    tile = lambda k, n_: np.array(q[k], dtype=np.float64).reshape(1, n_)
    A = (q["A_colptr"], q["A_rowidx"], np.array(q["A_val"]))
    Hc = (q["H_colptr"], q["H_rowidx"], np.array(q["H_val"]))
    s = solve_batch_csc(nV, nC, A, Hc, tile("g", nV), tile("lb", nV), tile("ub", nV), tile("lbA", nC), tile("ubA", nC), team_size=32)
    so = orc.OracleQP(nV, nC)
    st = so.init(Hc, q["g"], A, q["lb"], q["ub"], q["lbA"], q["ubA"])
    single = so.solution()[3]
    assert st != 20 and int(s.get_status()[0]) == st
    assert int(s.get_iterations()[0]) == 2 * single
    s.close()

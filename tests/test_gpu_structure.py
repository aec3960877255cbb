"""Structure calls of the C ABI (include/sqpb200.h: sqpb200_set_structure_A / _H / _csc and their compressed-row forms): the
kernel launches of every route and of the value calls that go with it, the rejection of malformed directly given patterns, and
the rule that a handle's structures are fixed once its solve buffers exist.  No solve here ever runs on a malformed pattern or
on a pattern set after a solve."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import restartsqp_b200 as r
from restartsqp_b200 import capi
import helpers as H

pytestmark = pytest.mark.gpu
ERR_INVALID, ERR_STATE = -1, -4
MATS = (capi.MAT_A, capi.MAT_H)


@pytest.fixture(scope="module")
def L():
    L = capi.lib()
    assert L.sqpb200_device_count() > 0, "no CUDA device"
    return L


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def csr(M):
    M = sp.csr_matrix(M)
    M.sort_indices()
    return i32(M.indptr), i32(M.indices)


def triplets(colptr, rowidx):
    """1-based (row, column) of every entry of a compressed-column pattern, in storage order."""
    return i32(np.asarray(rowidx) + 1), i32(np.repeat(np.arange(len(colptr) - 1), np.diff(colptr)) + 1)


def set_csc(L, s, which, colptr, rowidx):
    colptr, rowidx = i32(colptr), i32(rowidx)
    return L.sqpb200_set_structure_csc(s.h, which, len(rowidx), ptr(colptr), ptr(rowidx))


def set_csr(L, s, which, rowptr, colidx):
    rowptr, colidx = i32(rowptr), i32(colidx)
    return L.sqpb200_set_structure_csr(s.h, which, len(colidx), ptr(rowptr), ptr(colidx))


def set_triplets_A(L, s, row1, col1, ident=None, compressed_row=False):
    f = L.sqpb200_set_structure_A_csr if compressed_row else L.sqpb200_set_structure_A
    if ident is None:
        return f(s.h, len(row1), ptr(row1), ptr(col1), 0, None, None, None, None)
    ir, jc, sz, val = ident
    return f(s.h, len(row1), ptr(row1), ptr(col1), len(sz), ptr(ir), ptr(jc), ptr(sz), ptr(val))


def set_triplets_H(L, s, row1, col1, symmetric, compressed_row=False):
    f = L.sqpb200_set_structure_H_csr if compressed_row else L.sqpb200_set_structure_H
    return f(s.h, len(row1), ptr(row1), ptr(col1), int(symmetric))


def structure(L, s, which):
    nnz = L.sqpb200_get_nnz(s.h, which)
    cp, ri, od = np.zeros(s.nV_ + 1, np.int32), np.zeros(nnz, np.int32), np.zeros(nnz, np.int32)
    assert L.sqpb200_get_structure(s.h, which, ptr(cp), ptr(ri), ptr(od)) == 0
    vals = np.zeros((s.batch, nnz))
    assert L.sqpb200_get_values_csc(s.h, which, ptr(vals), capi.LOC_HOST) == 0
    return cp, ri, od, vals


def outputs(s):
    x, y, obj, st, it = s._get_solution(("x", "y", "obj", "status", "iters"))
    wc, wb = s.get_working_set(translated=False)
    return dict(x=x, y=y, obj=obj, status=st, iters=it, wc=wc, wb=wb)


def assert_same(a, b):
    for k in a:
        assert a[k].tobytes() == b[k].tobytes(), k


def qp(seed, dens=1.0):
    p = H.random_l1_qp(np.random.default_rng(seed), 5, 3, dens=dens)
    p["Ac"], p["Hc"] = H.csc(p["A"]), H.csc(p["H"])
    return p


def set_vectors(s, p, B):
    g = np.tile(p["g"], (B, 1))
    g[:, :p["n"]] += np.random.default_rng(7).standard_normal((B, p["n"]))
    s.set_g(g); s.set_lb(p["lb"]); s.set_ub(p["ub"]); s.set_lbA(p["lbA"]); s.set_ubA(p["ubA"])


# ---------------------------------------------------------------------------------------------------------- kernel launches
def launches(L, s, call):
    before = L.sqpb200_launch_count(s.h)
    rc = call()
    assert rc >= 0, (rc, L.sqpb200_last_error(s.h))
    return L.sqpb200_launch_count(s.h) - before


@pytest.mark.parametrize("route", ["triplet", "triplet_csr", "csc", "csr"])
def test_launches_per_route(L, route):
    """Structure: a triplet A is sorted and its identity entries broadcast (2), a triplet H is sorted (1), a pattern given
    directly launches nothing.  Values: triplet order and compressed-row order are scattered (1), compressed-column order is
    one copy (0) unless broadcast (1); reading values back in compressed-row order is one gather (1), in compressed-column
    order a copy (0)."""
    c = {c["name"]: c for c in H.load_l0_golden()}["rand1"]
    n, m, B = c["n"], c["m"], 4
    nV, nC = n + 2 * m, m
    rng = np.random.default_rng(3)
    s = r.CudaQPInterface(nV=nV, nC=nC, batch=B)
    if route in ("triplet", "triplet_csr"):
        ident = (i32([1, 1]), i32([n + 1, n + m + 1]), i32([m, m]), np.array([1.0, -1.0]))
        Jr, Jc, Hr, Hc = i32(c["J_row1"]), i32(c["J_col1"]), i32(c["H_row1"]), i32(c["H_col1"])
        row = route == "triplet_csr"
        assert launches(L, s, lambda: set_triplets_A(L, s, Jr, Jc, ident, row)) == 2
        assert launches(L, s, lambda: set_triplets_H(L, s, Hr, Hc, True, row)) == 1
        for bc, vJ, vH in ((0, rng.standard_normal((B, len(Jr))), rng.standard_normal((B, len(Hr)))),
                           (1, rng.standard_normal(len(Jr)), rng.standard_normal(len(Hr)))):
            assert launches(L, s, lambda: L.sqpb200_set_values_A(s.h, ptr(vJ), capi.LOC_HOST, bc)) == 1
            assert launches(L, s, lambda: L.sqpb200_set_values_H(s.h, ptr(vH), capi.LOC_HOST, bc)) == 1
    else:
        A = sp.csc_matrix((np.ones(len(c["A_rowidx"])), c["A_rowidx"], c["A_colptr"]), shape=(nC, nV))
        Hm = sp.csc_matrix((np.ones(len(c["H_rowidx"])), c["H_rowidx"], c["H_colptr"]), shape=(nV, nV))
        for which, M in ((capi.MAT_A, A), (capi.MAT_H, Hm)):
            if route == "csc":
                assert launches(L, s, lambda: set_csc(L, s, which, M.indptr, M.indices)) == 0
            else:
                assert launches(L, s, lambda: set_csr(L, s, which, *csr(M))) == 0
    for which in MATS:
        z = L.sqpb200_get_nnz(s.h, which)
        assert z > 0
        v, v1, out = rng.standard_normal((B, z)), rng.standard_normal(z), np.zeros((B, z))
        assert launches(L, s, lambda: L.sqpb200_set_values_csc(s.h, which, ptr(v), capi.LOC_HOST, 0)) == 0
        assert launches(L, s, lambda: L.sqpb200_set_values_csc(s.h, which, ptr(v1), capi.LOC_HOST, 1)) == 1
        assert launches(L, s, lambda: L.sqpb200_get_values_csc(s.h, which, ptr(out), capi.LOC_HOST)) == 0
        assert (out == v1).all()
        if route in ("triplet_csr", "csr"):
            assert launches(L, s, lambda: L.sqpb200_set_values_csr(s.h, which, ptr(v), capi.LOC_HOST, 0)) == 1
            assert launches(L, s, lambda: L.sqpb200_set_values_csr(s.h, which, ptr(v1), capi.LOC_HOST, 1)) == 1
            assert launches(L, s, lambda: L.sqpb200_get_values_csr(s.h, which, ptr(out), capi.LOC_HOST)) == 1
            assert (out == v1).all()
    s.close()


# ---------------------------------------------------------------------------------------------------------- malformed patterns
def malformed(p, layout, defect):
    """(ptr, idx) of A in the given layout with one defect."""
    nV, nC = p["nV"], p["nC"]
    P, I = (p["Ac"][0], p["Ac"][1]) if layout == "csc" else csr(p["A"])
    P, I = P.copy(), I.copy()
    bound = nC if layout == "csc" else nV
    if defect == "ptr0":
        P[0] = 1
    elif defect == "nonmonotone":
        assert P[2] > P[1]
        P[1], P[2] = P[2], P[1]
    elif defect == "index_at_bound":
        I[0] = bound
    elif defect == "index_negative":
        I[-1] = -1
    return P, I


@pytest.mark.parametrize("layout", ["csc", "csr"])
@pytest.mark.parametrize("defect", ["ptr0", "nonmonotone", "index_at_bound", "index_negative"])
def test_malformed_direct_pattern_is_rejected(L, layout, defect):
    """A malformed pattern returns SQPB200_ERR_INVALID and leaves the handle as it was; a valid pattern set afterwards solves
    bit for bit as on a fresh handle."""
    p, B = qp(11), 8
    nV, nC = p["nV"], p["nC"]
    s = r.CudaQPInterface(nV=nV, nC=nC, batch=B)
    assert set_csc(L, s, capi.MAT_A, *p["Ac"][:2]) == len(p["Ac"][1])
    before = structure(L, s, capi.MAT_A)
    f = set_csc if layout == "csc" else set_csr
    assert f(L, s, capi.MAT_A, *malformed(p, layout, defect)) == ERR_INVALID
    assert L.sqpb200_last_error(s.h)
    for a, b in zip(before, structure(L, s, capi.MAT_A)):
        assert a.tobytes() == b.tobytes()
    assert L.sqpb200_get_structure_csr(s.h, capi.MAT_A, None, None, None) == ERR_STATE
    res = []
    for h in (s, r.CudaQPInterface(nV=nV, nC=nC, batch=B)):
        h.set_csc(capi.MAT_A, *p["Ac"]); h.set_csc(capi.MAT_H, *p["Hc"])
        set_vectors(h, p, B)
        h.optimizeQP()
        res.append(outputs(h))
        h.close()
    assert (res[0]["status"] == capi.QP_OPTIMAL).all()
    assert_same(res[0], res[1])


# ---------------------------------------------------------------------------------------------------------- repeated calls
def test_second_structure_call_before_solve_wins(L):
    """Before the first solve a structure may be set again, through any route; the handle then holds exactly what a fresh
    handle given only the last structure holds."""
    p1, p2, B = qp(21, dens=0.4), qp(22), 4
    nV, nC, n = p1["nV"], p1["nC"], p1["n"]
    p1["H"][0, 1:n] = p1["H"][1:n, 0] = 0.0
    p1["Hc"] = H.csc(p1["H"])
    assert len(p1["Ac"][1]) != len(p2["Ac"][1]) and len(p1["Hc"][1]) != len(p2["Hc"][1])
    s, fresh = r.CudaQPInterface(nV=nV, nC=nC, batch=B), r.CudaQPInterface(nV=nV, nC=nC, batch=B)
    assert set_csr(L, s, capi.MAT_A, *csr(p1["A"])) == len(p1["Ac"][1])
    assert set_triplets_H(L, s, *triplets(*p1["Hc"][:2]), False) == len(p1["Hc"][1])
    assert set_csc(L, s, capi.MAT_A, *p2["Ac"][:2]) == len(p2["Ac"][1])
    assert set_triplets_H(L, s, *triplets(*p2["Hc"][:2]), False, compressed_row=True) == len(p2["Hc"][1])
    assert set_csc(L, fresh, capi.MAT_A, *p2["Ac"][:2]) == len(p2["Ac"][1])
    assert set_triplets_H(L, fresh, *triplets(*p2["Hc"][:2]), False, compressed_row=True) == len(p2["Hc"][1])
    assert L.sqpb200_get_structure_csr(s.h, capi.MAT_A, None, None, None) == ERR_STATE  # the compressed-row view went with A
    for which, v in ((capi.MAT_A, p2["Ac"][2]), (capi.MAT_H, p2["Hc"][2])):
        for h in (s, fresh):
            h.set_csc_values(which, v)
        for a, b in zip(structure(L, s, which), structure(L, fresh, which)):
            assert a.tobytes() == b.tobytes()
    rows = [(np.zeros(nV + 1, np.int32), np.zeros(len(p2["Hc"][1]), np.int32), np.zeros(len(p2["Hc"][1]), np.int32)) for _ in range(2)]
    for h, (rp, ci, od) in zip((s, fresh), rows):
        assert L.sqpb200_get_structure_csr(h.h, capi.MAT_H, ptr(rp), ptr(ci), ptr(od)) == 0
    for a, b in zip(*rows):
        assert a.tobytes() == b.tobytes()
    s.close(); fresh.close()


@pytest.mark.parametrize("team", [0, 1024])
def test_structure_call_after_solve_is_rejected(L, team):
    """Once a solve has allocated the solve buffers (sized by the structures) every structure call returns SQPB200_ERR_STATE,
    even with the same pattern, and changes nothing: the next solve is bit for bit the one of a handle that was never asked."""
    p, B = qp(31), 8
    nV, nC = p["nV"], p["nC"]
    (Ap, Ai, _), (Hp, Hi, _) = p["Ac"], p["Hc"]
    hs = [r.CudaQPInterface(nV=nV, nC=nC, batch=B, team_size=team) for _ in range(2)]
    first = []
    for h in hs:
        h.set_csc(capi.MAT_A, *p["Ac"]); h.set_csc(capi.MAT_H, *p["Hc"])
        set_vectors(h, p, B)
        h.optimizeQP()
        first.append(outputs(h))
    assert_same(first[0], first[1])
    s = hs[0]
    before = [structure(L, s, which) for which in MATS]
    calls = [lambda: set_csc(L, s, capi.MAT_A, Ap, Ai), lambda: set_csc(L, s, capi.MAT_H, Hp, Hi),
             lambda: set_csr(L, s, capi.MAT_A, *csr(p["A"])), lambda: set_csr(L, s, capi.MAT_H, *csr(p["H"]))]
    for row in (False, True):
        calls += [lambda row=row: set_triplets_A(L, s, *triplets(Ap, Ai), compressed_row=row),
                  lambda row=row: set_triplets_H(L, s, *triplets(Hp, Hi), False, compressed_row=row)]
    for call in calls:
        assert call() == ERR_STATE
        assert L.sqpb200_last_error(s.h)
    for which, b in zip(MATS, before):
        for x, y in zip(b, structure(L, s, which)):
            assert x.tobytes() == y.tobytes()
    second = []
    for h in hs:
        h.optimizeQP()
        second.append(outputs(h))
        h.close()
    assert (second[0]["status"] == capi.QP_OPTIMAL).all()
    assert_same(second[0], second[1])

"""The warp kernel with more active constraints than a warp has lanes.  Up to 32 active constraints the T solves keep the
right-hand side in registers and the removals of the exchange step run their Givens chains in registers, one row of T per lane;
above 32 both fall back to the barrier-per-step loops.  Equality-heavy rows end with more than 32 constraints in the oracle's
working set, so the T solves of these solves take their fallback; whether a removal happens while more than 32 constraints are
active depends on the path and is not asserted.  Every instance is checked bit for bit against the oracle like every other
warp-kernel shape."""
import numpy as np
import pytest

import restartsqp_b200 as r
from oracle import oracle_py as orc
import helpers as H
from test_gpu_qp import check_against_oracle, solve_batch_csc

pytestmark = pytest.mark.gpu


def equality_heavy_qp(n, m, seed):
    rng = np.random.default_rng(seed)
    base = H.random_l1_qp(rng, n, m, convex=True, dens=0.5)
    eq = rng.random(m) < 0.85  # most rows become equalities at their finite bound, the rest keep their one- or two-sided bounds
    at = np.where(base["lbA"] < -1e17, base["ubA"], base["lbA"])
    base["lbA"] = np.where(eq, at, base["lbA"])
    base["ubA"] = np.where(eq, at, base["ubA"])
    return rng, base


@pytest.mark.parametrize("shape", [(24, 40), (12, 44)])
def test_more_active_constraints_than_lanes(gpu_lib, shape):
    n, m = shape
    rng, base = equality_heavy_qp(n, m, 2000 + 31 * n + m)
    nV, nC, B = base["nV"], base["nC"], 8
    Ac, Hc = H.csc(base["A"]), H.csc(base["H"])
    g = np.tile(base["g"], (B, 1)); g[:, :n] += rng.standard_normal((B, n))
    lb, ub = np.tile(base["lb"], (B, 1)), np.tile(base["ub"], (B, 1))
    lbA, ubA = np.tile(base["lbA"], (B, 1)), np.tile(base["ubA"], (B, 1))
    s = solve_batch_csc(nV, nC, Ac, Hc, g, lb, ub, lbA, ubA, team_size=32)
    assert s.solve_config()["team_size"] == 32
    most_active = 0
    for b in range(B):
        p = dict(nV=nV, nC=nC, g=g[b], lb=lb[b], ub=ub[b], lbA=lbA[b], ubA=ubA[b])
        o = H.oracle_solve(orc, p, Acsc=Ac, Hcsc=Hc)
        check_against_oracle(s, b, o, nV)
        most_active = max(most_active, int(np.count_nonzero(o["wc"])))
    assert most_active > 32, "the shape no longer reaches the nAC > 32 T solves"
    s.close()

"""Batch independence of the bounded (TRF) branch.

The bounded branch runs every candidate of a batch in lock-step: its element-wise passes and reductions cover all
candidates in one launch, and candidates leave the outer and inner loops at different iterations.  A candidate's
arithmetic must not depend on which other candidates share its batch or are still running, so a candidate solved in a
batch must give the same bits as the same candidate solved alone: LSMR iterations, score, x, TRF iteration count and
the per-iteration TRF trace (inner iterations, step kind, p/r/ag values, predicted cost change).
"""
import numpy as np
import pytest

from tests.helpers import load

pytestmark = pytest.mark.gpu


def _make_batch(img, twist, rise_px, csym, L3, so, specs_extra=(), positive=False):
    from helicon_b200.engine import Batch, Problem
    from helicon_b200.planner import CandidateSpec, MAX_EQUATIONS

    N = img.shape[0]
    prob = Problem(img, 1.0, N, N, N, 0.0, N // 2 - 1)
    target = min(MAX_EQUATIONS, int(max(N * N, L3 * prob.ndisk) * so))
    specs = [CandidateSpec(twist, rise_px, csym, target, target, positive)]
    for tw, ri in specs_extra:
        specs.append(CandidateSpec(tw, ri, csym, target, target, positive))
    return prob, Batch(prob, L3, specs), target


def _bounded_solve(batch):
    # the options solver_linear_regression uses for positive_constraint (scipy lsq_linear defaults)
    m = batch.rows_padded(0)[1]
    res = batch.solve(atol=1e-12, btol=1e-12, max_iter=int(min(max(m, 1), batch.n)), trf_tol=1e-10, trf_max_iter=200)
    return res, [batch.trf_trace(c) for c in range(batch.nc)]


def test_bounded_batched_candidates_equal_single_candidate_solves():
    d = load("solve_nn_unb_48_t35")
    apix, twist, rise, csym, pc, so, L3 = d["args"]
    img = d["image"]
    extra = [(-3.1, 9.0 / apix), (-4.2, 10.1 / apix), (12.5, 9.5 / apix)]
    prob, batch, target = _make_batch(img, float(twist), float(rise / apix), int(csym), int(L3), int(so), extra, True)
    res, traces = _bounded_solve(batch)
    xs = [batch.x(c) for c in range(batch.nc)]
    batch.close()
    assert (res["trf_nit"] > 0).any(), "no candidate took the bounded branch: the case guards nothing"
    singles = [(float(twist), float(rise / apix))] + extra
    for c, (tw, ri) in enumerate(singles):
        p2, b2, _ = _make_batch(img, tw, ri, int(csym), int(L3), int(so), positive=True)
        r2, t2 = _bounded_solve(b2)
        assert r2[0]["itn"] == res[c]["itn"] and r2[0]["score"] == res[c]["score"]
        assert r2[0]["trf_nit"] == res[c]["trf_nit"] and r2[0]["flags"] == res[c]["flags"]
        tr_b, nit_b, status_b = traces[c]
        tr_s, nit_s, status_s = t2[0]
        assert (nit_s, status_s) == (nit_b, status_b)
        assert np.array_equal(tr_s, tr_b)  # identical bits, NaN-free by construction (inf compares equal)
        assert np.array_equal(b2.x(0), xs[c])
        b2.close(); p2.close()
    prob.close()

"""The batched ElasticNet / Lasso / Ridge solver (hb2_batch_solve_model, Batch.solve_model) and the grid search over it.

(a) the primitive everything rests on: MODE_PLAIN products over the whole batch equal the per-candidate products bit for
bit, on a batch with tie views; (b) the reference goldens with the assertions test_gpu_models.py applies to the host
path; (c) batch independence; (d) the device result against the host-driven one (regularized.py); (e) search_grid, the
CLI and a resumed search.
"""
import numpy as np
import pytest

from tests.helpers import load

pytestmark = pytest.mark.gpu


def _batch(img, L3, cands, so, pc):
    """One nearest-neighbour batch of (twist, rise_pixel, csym) candidates over the whole image (s = 1)."""
    from helicon_b200.engine import Batch, Problem
    from helicon_b200.planner import MAX_EQUATIONS, CandidateSpec, positive_rule

    N = img.shape[0]
    prob = Problem(img, 1.0, N, N, N, 0.0, N // 2 - 1)
    target = min(MAX_EQUATIONS, int(max(N * N, L3 * prob.ndisk) * so))
    specs = [CandidateSpec(tw, ri, cs, target, target, positive_rule(pc, ri, tw, L3)) for tw, ri, cs in cands]
    return prob, Batch(prob, L3, specs)


def test_batch_wide_plain_products_equal_per_candidate_products():
    d = load("solve_nn_unb_96_tie475")
    apix, twist, rise, csym, pc, so, L3 = d["args"]
    img = d["image"]
    cands = [(float(twist), float(rise / apix), int(csym)), (float(twist) + 1.3, float(rise / apix) * 1.04, int(csym)),
             (float(twist) - 2.1, float(rise / apix) * 0.97, int(csym))]
    prob, batch = _batch(img, int(L3), cands, int(so), 0)
    try:
        views = batch.plan.views
        print(f"tie views {int((views['tie'] >= 0).sum())}, Halton duplicates {int((views['dup_of'] >= 0).sum())}")
        assert (views["tie"] >= 0).any(), "no tie view: the case guards nothing"
        rng = np.random.default_rng(5)
        xs = rng.standard_normal((batch.nc, batch.n)).astype(np.float32)
        ys = [rng.standard_normal(batch.rows_padded(c)[1]).astype(np.float32) for c in range(batch.nc)]
        fw = batch.apply_all(xs=xs)
        ad = batch.apply_all(ys=ys)
        for c in range(batch.nc):
            assert np.array_equal(fw[c], batch.apply_forward(c, xs[c]))
            assert np.array_equal(ad[c], batch.apply_adjoint(c, ys[c]))
    finally:
        batch.close()
        prob.close()


def _objective(model, A, b, w, alpha, l1_ratio):
    r = b - A @ w
    r = r - r.mean()
    if model == "ridge":
        return float(r @ r + alpha * (w @ w))
    return float(r @ r / (2 * A.shape[0]) + alpha * l1_ratio * np.abs(w).sum() + 0.5 * alpha * (1 - l1_ratio) * (w @ w))


@pytest.mark.parametrize("name", ["model_enet_40", "model_enet_40_pos", "model_lasso_32", "model_ridge_32",
                                  "model_ridge_32_pos"])
def test_solve_model_vs_reference_goldens(name):
    from scipy.sparse import vstack

    from oracle import denovo3d_oracle as O

    d = load(name)
    apix, twist, rise, csym, L3, so, pc, alpha, l1r = (float(v) for v in d["args"])
    img, model = d["image"], str(d["model"])
    N, L3 = img.shape[0], int(L3)
    prob, batch = _batch(img, L3, [(twist, rise / apix, int(csym))], int(so), int(pc))
    try:
        res = batch.solve_model(dict(model=model, alpha=alpha, l1_ratio=l1r))
        rec, score, info = batch.rec3d(0), float(res[0]["score"]), batch.model_info(0)
    finally:
        batch.close()
        prob.close()
    mask = O.cylindrical_mask(L3, N, N, 0, N // 2 - 1)
    w, x_ref, x_tight = rec[mask].astype(np.float64), d["rec3d"][mask].astype(np.float64), d["x_tight"]
    target = int(max(N * N, int(mask.sum())) * so)
    A_d, b_d, _ = O.build_A_data_matrix(img, 1.0, twist, rise / apix, int(csym), 0, 0, 0, N, N, N, 0, L3, target, "nn")
    A_s, b_s = O.build_A_helical_sym_matrix(L3, N, N, twist, rise / apix, int(csym), 0.0, N // 2 - 1, target, "nn")
    A = vstack((A_d, A_s)).tocsr().astype(np.float64)
    b = np.concatenate((b_d, b_s)).astype(np.float64)
    f_gpu = _objective(model, A, b, w, alpha, l1r)
    f_ref, f_tight = float(d["f_ref"]), float(d["f_tight"])
    rel = lambda a, r: float(np.linalg.norm(a - r) / np.linalg.norm(r))  # noqa: E731
    print(f"{name}: score {score:.6f} (minimiser {float(d['score_tight']):.6f}); objective {f_gpu:.8e} (reference "
          f"{f_ref:.8e}, minimiser {f_tight:.8e}); rel-L2 vs minimiser {rel(w, x_tight):.2e}; {info}, flags {res[0]['flags']}")
    assert f_gpu <= f_ref
    assert f_gpu <= f_tight * (1 + 1e-3)
    assert rel(w, x_tight) <= 2e-2 and rel(w, x_tight) <= 0.25 * float(d["rel_ref_vs_tight"])
    assert abs(score - float(d["score_tight"])) <= 1e-4
    assert rel(w, x_ref) <= 1.5 * float(d["rel_ref_vs_tight"])


CASES_C = [("elasticnet", 1), ("lasso", 0), ("ridge", 0), ("ridge", 1)]


@pytest.mark.parametrize("model,pc", CASES_C)
def test_solve_model_batch_independence(model, pc):
    d = load("model_enet_40")
    apix, twist, rise, csym, L3, so = (float(v) for v in d["args"][:6])
    img = d["image"]
    cands = [(twist + dt, rise / apix * f, int(csym)) for dt, f in ((0, 1), (1.7, 1.03), (-2.4, 0.95), (3.1, 1.06))]
    alg = dict(model=model)

    def run(cs):
        prob, batch = _batch(img, int(L3), cs, int(so), pc)
        try:
            res = batch.solve_model(alg)
            return res, [batch.x(c) for c in range(batch.nc)], [batch.model_info(c) for c in range(batch.nc)]
        finally:
            batch.close()
            prob.close()

    res, xs, infos = run(cands)
    print(model, pc, res[["score", "itn", "flags"]], infos)
    for c in range(len(cands)):
        r1, x1, i1 = run([cands[c]])
        assert r1[0]["score"] == res[c]["score"] and r1[0]["itn"] == res[c]["itn"] and r1[0]["flags"] == res[c]["flags"]
        assert np.array_equal(x1[0], xs[c])
        assert i1[0] == infos[c]


@pytest.mark.parametrize("model,pc", [("elasticnet", 1), ("elasticnet", 0), ("lasso", 0)])
def test_solve_model_device_against_host(model, pc):
    from helicon_b200.engine import model_params
    from helicon_b200.regularized import _CenteredOperator, solve_model

    d = load("model_enet_40")
    apix, twist, rise, csym, L3, so = (float(v) for v in d["args"][:6])
    img = d["image"]
    cands = [(twist, rise / apix, int(csym)), (twist + 1.7, rise / apix * 1.03, int(csym))]
    alg = dict(model=model)
    _, alpha, l1 = model_params(alg)
    prob, batch = _batch(img, int(L3), cands, int(so), pc)
    try:
        batch.solve_model(alg)
        w_dev = [batch.x(c).astype(np.float64) for c in range(batch.nc)]
        for c in range(batch.nc):
            op = _CenteredOperator(batch, c)
            w_host = solve_model(batch, c, alg, bool(batch.plan.cands[c]["positive"])).astype(np.float64)
            a_s, b_s = alpha * l1 * op.m, alpha * (1 - l1) * op.m

            def f(w):
                r = op.yc - op.X(w)
                return 0.5 * float(r @ r) + a_s * float(np.abs(w).sum()) + 0.5 * b_s * float(w @ w)

            tol = 0.05 * 1e-2 * float(op.yc @ op.yc)
            print(f"{model} pc={pc} c={c}: device {f(w_dev[c]):.8e} host {f(w_host):.8e} tolerance {tol:.3e}")
            assert abs(f(w_dev[c]) - f(w_host)) <= tol
    finally:
        batch.close()
        prob.close()


def _grid():
    d = load("grid_64")
    return d["image"], round(float(d["apix"]), 4), np.array([-2.13, -1.37, -0.67]), np.linspace(4.31, 5.13, 3)


@pytest.mark.parametrize("pc", [0, -1])
def test_search_grid_elasticnet_vs_lsq_reconstruct(pc):
    from helicon_b200.grid import build_tasks, search_grid
    from helicon_b200.solver_linear_regression import lsq_reconstruct

    img, apix, tw, ri = _grid()
    alg = dict(model="elasticnet")
    out = search_grid(img, apix, tw, ri, positive_constraint=pc, top_k=3, algorithm=alg)
    tasks, _ = build_tasks(img.shape[0], img.shape[1], apix, tw, ri, positive_constraint=pc)
    ref = np.full(out["scores"].shape, np.nan, dtype=np.float64)
    for t in tasks:
        g = t.geom
        _, sc = lsq_reconstruct(img, g["s"], t.twist, t.rise / g["apix3d"], t.csym, positive_constraint=pc,
                                reconstruct_diameter_3d_inner_pixel=g["D3i"], reconstruct_diameter_2d_pixel=g["D2"],
                                reconstruct_length_2d_pixel=g["L2"], reconstruct_diameter_3d_pixel=g["D3"],
                                reconstruct_length_3d_pixel=g["L3"], sym_oversample=g["sym_oversample"], algorithm=alg)
        ref.reshape(-1)[t.ti] = float(sc)
    got = out["scores"].astype(np.float64)
    print(f"pc={pc}: max |score - lsq_reconstruct| {np.nanmax(np.abs(got - ref)):.2e}; itn {out['itn'].ravel()}")
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    assert np.nanmax(np.abs(got - ref)) <= 1e-4
    s = np.sort(ref[np.isfinite(ref)])[::-1]
    if s[0] - s[1] > 2e-4:
        assert np.nanargmax(got) == np.nanargmax(ref)


def test_cli_and_resume_with_a_model(tmp_path):
    from helicon_b200 import denovo3DBatch
    from helicon_b200.grid import search_grid

    img, apix, tw, ri = _grid()
    alg = dict(model="elasticnet")
    kw = dict(positive_constraint=0, batch_candidates=3, top_k=4, algorithm=alg)
    ref = search_grid(img, apix, tw, ri, **kw)
    # the CLI writes the same score map bit for bit
    mrc = str(tmp_path / "img.mrc")
    denovo3DBatch.write_mrc(mrc, img, apix)
    prefix = str(tmp_path / "cli")
    rc = denovo3DBatch.main([mrc, "--apix", str(apix), "--twist=" + ",".join(repr(float(v)) for v in tw),
                             "--rise=" + ",".join(repr(float(v)) for v in ri), "--positive-constraint", "0", "--top-k", "4",
                             "--model", "elasticnet", "--output", prefix])
    assert rc == 0
    cli = np.load(prefix + "_img0_scores.npz")
    assert np.array_equal(cli["scores"], ref["scores"], equal_nan=True) and np.array_equal(cli["itn"], ref["itn"])

    # an interrupted, then resumed model search equals the uninterrupted one
    class Stop(Exception):
        pass

    def die_after_first_batch(done, total):
        raise Stop()

    ck = str(tmp_path / "run.tiles")
    with pytest.raises(Stop):
        search_grid(img, apix, tw, ri, checkpoint=ck, progress=die_after_first_batch, **kw)
    out = search_grid(img, apix, tw, ri, checkpoint=ck, **kw)
    assert out["n_restored"] == 3 and out["n_solved_here"] == ref["n_candidates"] - 3
    assert np.array_equal(out["scores"], ref["scores"], equal_nan=True)
    assert np.array_equal(out["itn"], ref["itn"]) and np.array_equal(out["flags"], ref["flags"])
    assert [(e["ti"], e["score"]) for e in out["top"]] == [(e["ti"], e["score"]) for e in ref["top"]]

"""The 2-D score metrics of the grid search on the device (hb2_batch_score_metric, Batch.score_metric,
search_grid(score_metric=...)) against the host restatements in imageprep.py, scattered as _metric_2d scatters them."""
import numpy as np
import pytest

from tests.helpers import load

pytestmark = pytest.mark.gpu

METRICS = ("ssim", "ms_ssim", "mutual_information", "composite")


def _image(N, L=None, seed=5):
    L = N if L is None else L
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:N, 0:L]
    img = np.zeros((N, L), np.float32)
    for _ in range(14):
        cy, cx = rng.uniform(N * 0.3, N * 0.7), rng.uniform(1, L - 1)
        img += np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / 5.0).astype(np.float32)
    return img


def _host_parts(batch, c, x, image, clip):
    """[ssim, ms_ssim, mi] of imageprep on pred_2d scattered from apply_forward(x) exactly as _metric_2d does."""
    from helicon_b200 import imageprep as M

    D2, L2 = batch.problem.D2, batch.problem.L2
    pidx, kk, jj = batch.data_row_index(c)
    pred = batch.apply_forward(c, x)[pidx]
    if clip:
        pred = np.clip(pred, 0, None)
    ny, nx = image.shape
    region = image[ny // 2 - D2 // 2: ny // 2 + D2 // 2, nx // 2 - L2 // 2: nx // 2 + L2 // 2]
    pred_2d = np.zeros((L2, D2), dtype=np.float32)
    pred_2d.ravel()[(kk * D2 + jj).astype(np.int64)] = pred
    ref_2d = region.T
    return np.array([M.ssim_score(pred_2d, ref_2d), M.ms_ssim_score(pred_2d, ref_2d),
                     M.mutual_information_score(pred_2d, ref_2d)])


def _check(batch, image, clip, label):
    """Device parts of every candidate against the host; the scores of each metric from the same parts."""
    cos = batch.results["score"].copy()
    _, parts = batch.score_metric("composite", clip_pred=clip, parts=True)
    scores = {m: batch.score_metric(m, clip_pred=clip)["score"] for m in METRICS}
    xs = [batch.x(c) for c in range(batch.nc)]  # before apply_forward, which leaves the batch unsolved
    host = np.array([_host_parts(batch, c, xs[c], image, clip) for c in range(batch.nc)])
    print(f"{label}: device parts\n{parts}\nmax |device - host| {np.abs(parts[:, 1:] - host).max():.2e}")
    assert np.array_equal(parts[:, 0], cos.astype(np.float64))
    assert np.abs(parts[:, 1:] - host).max() <= 1e-9
    for q, m in enumerate(("ssim", "ms_ssim", "mutual_information")):
        assert np.abs(scores[m].astype(np.float64) - host[:, q]).max() <= 1e-6
    comp = (cos.astype(np.float64) + host.sum(axis=1)) / 4
    assert np.abs(scores["composite"].astype(np.float64) - comp).max() <= 1e-6
    return parts


def _nn_batch(img, L3, cands, so, pc):
    from helicon_b200.engine import Batch, Problem
    from helicon_b200.planner import MAX_EQUATIONS, CandidateSpec, positive_rule

    N, L = img.shape
    prob = Problem(img, 1.0, N, L, N, 0.0, N // 2 - 1)
    target = min(MAX_EQUATIONS, int(max(N * L, L3 * prob.ndisk) * so))
    specs = [CandidateSpec(tw, ri, cs, target, target, positive_rule(pc, ri, tw, L3)) for tw, ri, cs in cands]
    return prob, Batch(prob, L3, specs)


def _tie_case():
    d = load("solve_nn_unb_96_tie475")
    apix, twist, rise, csym, pc, so, L3 = d["args"]
    cands = [(float(twist), float(rise / apix), int(csym)), (float(twist) + 1.3, float(rise / apix) * 1.04, int(csym)),
             (float(twist) - 2.1, float(rise / apix) * 0.97, int(csym)), (float(twist) + 0.4, float(rise / apix), int(csym))]
    return d["image"], int(L3), cands, int(so)


def test_lsq_batch_with_tie_views_and_halton_duplicates():
    img, L3, cands, so = _tie_case()
    prob, batch = _nn_batch(img, L3, cands, so, 0)
    try:
        views = batch.plan.views
        assert (views["tie"] >= 0).any() and (views["dup_of"] >= 0).any(), "the case guards nothing"
        # the last-writer table, built a second way: walk the rows in the reference's order, keep the last one
        for c in range(batch.nc):
            pidx, kk, jj = batch.data_row_index(c)
            loop = np.full(batch.problem.L2 * batch.problem.D2, -1, dtype=np.int32)
            for r, pid in zip(pidx, kk * batch.problem.D2 + jj):
                loop[pid] = r
            t = batch.pixel_rows(c)
            assert np.array_equal(t, loop)
            assert len(pidx) > (t >= 0).sum(), "no pixel written twice: the case guards nothing"
        batch.solve()
        _check(batch, img, 0, "nn tie")
        from helicon_b200._lib import HeliconB200Error

        with pytest.raises(HeliconB200Error):  # a solve is required: apply_forward (inside _check) left it unsolved
            batch.score_metric("ssim")
    finally:
        batch.close()
        prob.close()


def test_clipped_prediction_and_model_batch():
    from helicon_b200.grid import prepare_image

    img, L3, cands, so = _tie_case()
    img = prepare_image(img, 0.1, img.shape[0], 1.0)
    prob, batch = _nn_batch(img, L3, cands[:3], so, 1)
    try:
        batch.solve(clip_pred=1)
        _check(batch, img, 1, "clip")
        batch.solve_model(dict(model="elasticnet"), clip_pred=1)
        _check(batch, img, 1, "elasticnet")
    finally:
        batch.close()
        prob.close()


def test_bilinear_and_explicit_batches():
    from helicon_b200.bilinear import BilinearBatch
    from helicon_b200.engine import ExplicitBatch, Problem
    from helicon_b200.planner import CandidateSpec

    N, L3 = 40, 6
    img = _image(N)
    prob = Problem(img, 1.0, N, N, N, 0.0, N // 2 - 1, interpolation="linear")
    specs = [CandidateSpec(23.7, 2.31, 1, 0, 30000, False), CandidateSpec(-31.3, 1.77, 1, 4000, 9000, False)]
    try:
        bb = BilinearBatch(prob, L3, specs)
        try:
            bb.solve()
            _check(bb, img, 0, "bilinear")
        finally:
            bb.close()
        eb = ExplicitBatch(prob, L3, specs[0], tilt_degree=3.0, psi_degree=2.0, interpolation="nn")
        try:
            eb.solve()
            _check(eb, img, 0, "explicit")
        finally:
            eb.close()
    finally:
        prob.close()


@pytest.mark.parametrize("shape", [(6, 16), (10, 10), (42, 50), (26, 34)])
def test_small_and_odd_sides(shape):
    """Sides below 7 (ssim 0) and below 8 (ms_ssim 0), one MS-SSIM scale, and odd sides on the way down
    (50 -> 25 -> 12, 42 -> 21 -> 10: round half to even)."""
    D2, L2 = shape
    img = _image(D2, L2, seed=3)
    prob, batch = _nn_batch(img, 4, [(-4.3, 1.73, 1), (7.1, 2.2, 1)], 4, 0)
    try:
        batch.solve()
        parts = _check(batch, img, 0, f"sides {shape}")
        if min(shape) < 7:
            assert (parts[:, 1] == 0).all()
        if min(shape) < 8:
            assert (parts[:, 2] == 0).all()
    finally:
        batch.close()
        prob.close()


def test_zero_image_gives_zero_metrics():
    """An all-zero image: b = 0, x = 0, so both images are constant: data range 0 (ssim, ms_ssim 0.0) and the
    histogram's widened range puts every sample in one bin (H(X, Y) = 0, the host's ZeroDivisionError -> 0.0)."""
    img = np.zeros((32, 32), np.float32)
    prob, batch = _nn_batch(img, 4, [(-4.3, 1.73, 1)], 4, 0)
    try:
        batch.solve()
        parts = _check(batch, img, 0, "zero")
        assert (parts[:, 1:] == 0).all()
    finally:
        batch.close()
        prob.close()


def test_batch_independence():
    img, L3, cands, so = _tie_case()
    prob, batch = _nn_batch(img, L3, cands, so, 0)
    try:
        batch.solve()
        _, all4 = batch.score_metric("composite", parts=True)
    finally:
        batch.close()
    for c in (0, 3):  # alone, the first and the last candidate of the batch of 4
        p1, one = _nn_batch(img, L3, [cands[c]], so, 0)
        try:
            one.solve()
            _, p = one.score_metric("composite", parts=True)
            assert np.array_equal(p[0], all4[c])
        finally:
            one.close()
            p1.close()
    prob.close()


def _grid():
    d = load("grid_64")
    return d["image"], round(float(d["apix"]), 4), np.array([-2.13, -1.37, -0.67]), np.linspace(4.31, 5.13, 3)


@pytest.mark.parametrize("pc", [0, -1])
def test_search_grid_vs_lsq_reconstruct(pc):
    from helicon_b200.grid import build_tasks, search_grid
    from helicon_b200.solver_linear_regression import lsq_reconstruct

    img, apix, tw, ri = _grid()
    tasks, _ = build_tasks(img.shape[0], img.shape[1], apix, tw, ri, positive_constraint=pc)
    for m in ("cosine",) + METRICS:
        out = search_grid(img, apix, tw, ri, positive_constraint=pc, top_k=3, score_metric=m)
        ref = np.full(out["scores"].shape, np.nan, dtype=np.float64)
        for t in tasks:
            g = t.geom
            _, sc = lsq_reconstruct(img, g["s"], t.twist, t.rise / g["apix3d"], t.csym, positive_constraint=pc,
                                    reconstruct_diameter_3d_inner_pixel=g["D3i"], reconstruct_diameter_2d_pixel=g["D2"],
                                    reconstruct_length_2d_pixel=g["L2"], reconstruct_diameter_3d_pixel=g["D3"],
                                    reconstruct_length_3d_pixel=g["L3"], sym_oversample=g["sym_oversample"],
                                    score_metric=m)
            ref.reshape(-1)[t.ti] = float(sc)
        got = out["scores"].astype(np.float64)
        print(f"pc={pc} {m}: max |search_grid - lsq_reconstruct| {np.nanmax(np.abs(got - ref)):.2e}")
        assert np.array_equal(np.isnan(got), np.isnan(ref))
        assert np.nanmax(np.abs(got - ref)) <= 1e-5
        s = np.sort(ref[np.isfinite(ref)])[::-1]
        if s[0] - s[1] > 1e-4:
            assert np.nanargmax(got) == np.nanargmax(ref)
            assert out["top"][0]["ti"] == int(np.nanargmax(ref))


def test_default_is_cosine_and_never_calls_the_metric(monkeypatch):
    from helicon_b200.engine import Batch
    from helicon_b200.grid import search_grid

    img, apix, tw, ri = _grid()
    a = search_grid(img, apix, tw, ri, positive_constraint=0, top_k=4)

    def refuse(*args, **kw):
        raise AssertionError("score_metric called on the cosine path")

    monkeypatch.setattr(Batch, "score_metric", refuse)
    b = search_grid(img, apix, tw, ri, positive_constraint=0, top_k=4, score_metric="cosine")
    for k in ("scores", "itn", "flags"):
        assert np.array_equal(a[k], b[k], equal_nan=True)
    assert [(e["ti"], e["score"]) for e in a["top"]] == [(e["ti"], e["score"]) for e in b["top"]]


def test_cli_and_resume_with_ssim(tmp_path):
    from helicon_b200 import denovo3DBatch
    from helicon_b200.grid import search_grid

    img, apix, tw, ri = _grid()
    kw = dict(positive_constraint=0, batch_candidates=3, top_k=4, score_metric="ssim")
    ref = search_grid(img, apix, tw, ri, **kw)
    mrc = str(tmp_path / "img.mrc")
    denovo3DBatch.write_mrc(mrc, img, apix)
    prefix = str(tmp_path / "cli")
    rc = denovo3DBatch.main([mrc, "--apix", str(apix), "--twist=" + ",".join(repr(float(v)) for v in tw),
                             "--rise=" + ",".join(repr(float(v)) for v in ri), "--positive-constraint", "0", "--top-k", "4",
                             "--score-metric", "ssim", "--output", prefix])
    assert rc == 0
    cli = np.load(prefix + "_img0_scores.npz")
    assert np.array_equal(cli["scores"], ref["scores"], equal_nan=True) and np.array_equal(cli["itn"], ref["itn"])
    import json

    assert json.load(open(prefix + "_top.json"))[0]["score_metric"] == "ssim"

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
    # the SSIM tiles are not reused by a cosine search, and cosine tiles not by an SSIM search
    cos = search_grid(img, apix, tw, ri, checkpoint=ck, **dict(kw, score_metric="cosine"))
    assert cos["n_restored"] == 0
    ssim = search_grid(img, apix, tw, ri, checkpoint=ck, **kw)
    assert ssim["n_restored"] == 0
    assert np.array_equal(ssim["scores"], ref["scores"], equal_nan=True)

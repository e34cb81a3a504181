"""CPU: the C-ABI library loads and exports every declared symbol, the LSMR
scalar recurrences (compiled host+device from the same source) follow scipy's
executed precision map, and the host planner restates the reference's ordering
logic.  No GPU compute."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from helicon_b200 import _lib, planner
from oracle import denovo3d_oracle as O
from tests.helpers import ROOT, load


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    hdr = open(os.path.join(ROOT, "include", "helicon_b200.h")).read()
    declared = set(re.findall(r"\b(hb2_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name


def test_struct_sizes_match_numpy_dtypes():
    assert _lib.CANDIDATE_DTYPE.itemsize == C.sizeof(_lib.Candidate) == 32
    assert _lib.PAIR_DTYPE.itemsize == 48 and _lib.VIEW_DTYPE.itemsize == C.sizeof(_lib.View) == 24


def test_no_gpu_means_loud_failure():
    lib = _lib.load()
    if lib.hb2_device_count() > 0:
        pytest.skip("GPU present")
    with pytest.raises(_lib.HeliconB200Error):
        _lib.require_gpu()
    from helicon_b200 import solver_linear_regression as solver

    with pytest.raises(_lib.HeliconB200Error):
        solver.lsq_reconstruct(np.ones((8, 8), np.float32), 1.0, 30, 2, reconstruct_diameter_3d_pixel=8,
                               reconstruct_length_3d_pixel=4)


def _solve_case(name):
    from scipy.sparse import vstack

    d = load(name)
    apix, twist, rise, csym, pc, so, L3 = d["args"]
    img = d["image"]
    N = img.shape[0]
    _, _, det = O.lsq_reconstruct(
        img, 1.0, float(twist), float(rise / apix), int(csym), positive_constraint=0,
        reconstruct_diameter_2d_pixel=N, reconstruct_length_2d_pixel=N, reconstruct_diameter_3d_pixel=N,
        reconstruct_length_3d_pixel=int(L3), sym_oversample=int(so), return_details=True)
    A = vstack((det["A_data"], det["A_hsym"])).tocsr()
    b = np.concatenate((det["b_data"], np.zeros(det["A_hsym"].shape[0], np.float32)))
    return A, b


@pytest.mark.parametrize("name", ["solve_nn_unb_32", "solve_nn_unb_48_t35"])
def test_scalar_recurrences_match_scipy_precision_map(name):
    """Drive the library's host build of the recurrences with (alpha, beta, normx)
    taken from the oracle's LSMR; coefficients and stop iteration must agree exactly."""
    lib = _lib.load()
    A, b = _solve_case(name)
    AT = A.T.tocsr()
    f = np.float32
    # re-run the oracle LSMR, recording alpha/beta/normx per iteration via the vectors
    trace = []
    x_ref, istop_ref, itn_ref, *_ = O.lsmr_mixed(A, b, trace=trace)
    state = np.zeros(64, dtype=np.float64)
    cfh, cfx, cfhh = C.c_float(), C.c_float(), C.c_float()
    tr = np.zeros(8)
    # initial alpha, beta exactly as lsmr.py:239-262
    u = b.astype(f).copy()
    beta0 = f(np.linalg.norm(u))
    u = f(1 / beta0) * u
    v = AT.dot(u)
    alpha0 = f(np.linalg.norm(v))
    lib.hb2_lsmr_scalar_step(_lib.ptr(state), 0, alpha0, beta0, 0.0, 1e-4, 1e-4, 1e8, 1000, C.byref(cfh), C.byref(cfx), C.byref(cfhh), _lib.ptr(tr))
    istop = 0
    for t in trace:
        lib.hb2_lsmr_scalar_step(_lib.ptr(state), 1, f(t["alpha"]), f(t["beta"]), 0.0, 1e-4, 1e-4, 1e8, 1000, C.byref(cfh), C.byref(cfx), C.byref(cfhh), _lib.ptr(tr))
        assert tr[0] == t["rho"] and tr[1] == t["rhobar"] and tr[2] == t["zeta"], t["itn"]
        assert tr[3] == t["normr"] and tr[4] == t["normA"], t["itn"]
        istop = lib.hb2_lsmr_scalar_step(_lib.ptr(state), 2, 0, 0, t["normx"], 1e-4, 1e-4, 1e8, 1000, C.byref(cfh), C.byref(cfx), C.byref(cfhh), _lib.ptr(tr))
        assert tr[5] == f(t["test1"]) and tr[6] == f(t["test2"]), t["itn"]
        if t["itn"] < itn_ref:
            assert istop == 0, t["itn"]
    assert istop == istop_ref


def test_planner_halton_and_pairs_match_reference_fixtures():
    d = load("halton")
    for k in d.files:
        assert np.array_equal(np.array(planner.halton_indices(int(k))), d[k])
    d = load("hsym_pairs")
    for i in range(5):
        tw, ri, cs, nz = d[f"case{i}_args"]
        res = planner.sorted_hsym_csym_pairs(float(tw), float(ri), int(cs), int(nz))
        arr = np.array([[e[0], e[1], e[2], e[3], e[4], e[5][0][0], e[5][0][1], e[5][1][0], e[5][1][1]] for e in res])
        assert np.array_equal(arr, d[f"case{i}"])


def test_planner_copies_match_oracle():
    for rise, csym, L3, L2 in [(2.4, 1, 6, 22), (3.1, 2, 8, 24), (1.9, 1, 4, 32), (3.654, 1, 12, 256), (0.7, 3, 4, 16)]:
        assert list(planner.data_copies(rise, csym, L3, L2)) == O.data_copies(rise, csym, L3, L2)


def test_rotation_entries_batch_equals_single_calls():
    from scipy.spatial.transform import Rotation as R

    angles = np.array([-1.2 * h for h in range(-40, 41)] + [30.0, 60.0, 90.0, 180.0, -179.5, 33.0 * 7 + 180.0])
    cs = planner.z_rotation_entries(angles)
    for a, (c, s) in zip(angles, cs):
        M = R.from_euler("z", a, degrees=True).as_matrix()
        assert c == M[0, 0] and s == M[1, 0] and M[0, 1] == -s and M[1, 1] == c


def test_column_slices_match_reference_tables():
    """Z of SLR:1578-1581 from the reference's own coordinate tables vs the planner's closed form."""
    img = np.zeros((24, 24), np.float32)
    for s, L2, L3, rise, h in [(1.0, 24, 8, 2.4, 3), (0.5, 24, 6, 1.9, -2), (1.0, 22, 6, 3.5, 1), (2.0, 16, 12, 2.2, 0)]:
        (X, Y, Z), _ = O.back_project_2d_coords_to_3d_coords(img, s, 12, L2)
        zref = np.rint(Z[:, 0, 6] - h * rise + L3 // 2).astype(int)  # central depth sample
        zi, tie = planner.column_slices(s, L2, L3, h * rise)
        ok = (zref >= 0) & (zref <= L3 - 1)
        if not tie:
            assert np.array_equal(np.where(ok, zref, -1), zi)
    zi, tie = planner.column_slices(1.0, 22, 6, 3.5)
    assert tie


@pytest.mark.parametrize("name", ["data_nn_tiez", "data_nn_csym2"])
def test_tie_views_reproduce_the_reference_slice_of_every_sample(name):
    """Column->slice ties (SURVEY F8): the planner's TieView tables (from planner.reference_z_table and the M22 of the
    copy's z-rotation) against the literal coordinate pipeline of the reference (SLR:1576-1581) for every ray j."""
    from scipy.spatial.transform import Rotation as R

    d = load(name)
    s, twist, rise, csym, D2, L2, D3, D3i, L3, mpl = d["args"]
    D2, L2, L3, csym = int(D2), int(L2), int(L3), int(csym)
    s, twist, rise = float(s), float(twist), float(rise)
    P = planner.BatchPlan(s, D2, L2, L3, [planner.CandidateSpec(twist, rise, csym, int(mpl), -1, False)])
    copies, aid, hidx, hs, ZI, ties = P._cand[0]
    assert P.has_ties and ties and not P.cand_tie_z[0]
    (X0, Y0, Z0), _ = O.back_project_2d_coords_to_3d_coords(d["image"], s, D2, L2)
    coords0 = np.vstack((X0.ravel(), Y0.ravel(), Z0.ravel())).T
    for (hi, c), tv in ties.items():
        h = hs[hi]
        cc = R.from_euler("z", twist * h + 360 * c / csym, degrees=True).apply(coords0, inverse=True)
        zi = np.rint(cc[:, 2].reshape(L2, D2, D2) - h * rise + L3 // 2).astype(np.int64)
        assert all(np.array_equal(zi[:, j, :], tv.zt) for j in range(D2)), (h, c)
        assert set(np.unique(tv.up)) <= {0, 1}


@pytest.mark.parametrize("N,s,angle", [(12, 1.0, 30.0), (16, 1.0, -60.0), (16, 0.5, 0.0), (14, 1.0, 150.0)])
def test_exact_map_requests_reproduce_the_reference_voxel_of_every_sample(N, s, angle):
    """In-plane ties (SURVEY F8): the x rows the planner hands to ``hb2_batch_add_exact_maps`` plus the kernel's
    arithmetic (fma(S, y0, C*x0) + D2//2, rint; restated here with exact rationals) against the literal coordinate
    pipeline of the reference (SLR:1576-1581) for every (column, ray, sample) -- and the x table carries no
    dependence on the ray j, the y table no noise at all."""
    from fractions import Fraction as F

    from scipy.spatial.transform import Rotation as R

    (X0, Y0, Z0), _ = O.back_project_2d_coords_to_3d_coords(np.zeros((N, N), np.float32), s, N, N)
    Xt, Zt = planner.reference_xz_tables(s, N, N)
    assert all(np.array_equal(X0[:, j, :], Xt) for j in range(N))
    assert all(np.array_equal(Z0[:, j, :], Zt) for j in range(N))
    assert np.array_equal(Y0, np.broadcast_to((s * (np.arange(N) - N // 2))[None, :, None], Y0.shape))
    coords0 = np.vstack((X0.ravel(), Y0.ravel(), Z0.ravel())).T
    cc = R.from_euler("z", angle, degrees=True).apply(coords0, inverse=True)
    Xr = np.rint(cc[:, 0].reshape(N, N, N) + N // 2)
    Yr = np.rint(cc[:, 1].reshape(N, N, N) + N // 2)
    C, S = planner.z_rotation_entries([angle])[0]
    fma = lambda a, b, c: float(F(a) * F(b) + F(c))
    y0 = s * (np.arange(N) - N // 2)
    varies = False
    for k in range(N):
        X = np.array([[fma(S, y0[j], C * Xt[k, i]) + N // 2 for i in range(N)] for j in range(N)])
        Y = np.array([[fma(C, y0[j], (-S) * Xt[k, i]) + N // 2 for i in range(N)] for j in range(N)])
        assert np.array_equal(np.rint(X), Xr[k]) and np.array_equal(np.rint(Y), Yr[k]), k
        varies |= not (np.array_equal(Xr[k], Xr[0]) and np.array_equal(Yr[k], Yr[0]))
    assert varies  # these are tie angles: the rounding really depends on the column


def test_mrc_writer_reader_round_trip(tmp_path):
    """denovo3DBatch.write_mrc <-> pipeline._read_mrc (the reference uses the mrcfile package for both)."""
    from helicon_b200 import pipeline
    from helicon_b200.denovo3DBatch import _axis, write_mrc

    vol = np.random.default_rng(0).random((3, 5, 7)).astype(np.float32)
    path = str(tmp_path / "v.mrc")
    write_mrc(path, vol, 1.3)
    data, apix = pipeline.get_images_from_file(path)
    assert np.array_equal(data, vol) and apix == 1.3
    assert np.array_equal(pipeline.read_image_2d(path, 1), vol[1])
    write_mrc(path, vol[0], 2.0)
    data, apix = pipeline.get_images_from_file(path)
    assert data.shape == (5, 7) and apix == 2.0
    assert np.allclose(_axis("-3:-1:5", "twist"), np.linspace(-3, -1, 5)) and list(_axis("4.7,4.8", "rise")) == [4.7, 4.8]


def test_transform_map_matches_reference_outputs():
    """helicon.transform_map (lib/transforms.py:168-235) on a small random volume: four argument sets generated by the
    unmodified reference (oracle/make_golden_task_tilt.py); same scipy calls -> identical to float32 round-off."""
    from helicon_b200 import transforms as T

    d = load("transform_map")
    for i in range(4):
        scale, rot, tilt, psi, dx, dy, dz = (float(v) for v in d[f"case{i}_args"])
        got = T.transform_map(d["vol"], scale=scale, rot=rot, tilt=tilt, psi=psi, dx=dx, dy=dy, dz=dz)
        ref = d[f"case{i}"]
        assert got.shape == ref.shape and got.dtype == ref.dtype
        assert np.allclose(got, ref, rtol=0, atol=1e-6), (i, float(np.abs(got - ref).max()))
    vol = d["vol"]
    assert T.transform_map(vol) is vol  # the identity returns its argument (lib/transforms.py:177-187)


def test_pad_to_size_centres_and_keeps_values():
    from helicon_b200 import transforms as T

    a = np.arange(12, dtype=np.float32).reshape(3, 4)
    p = T.pad_to_size(a, (4, 4))
    assert p.shape == (4, 4) and np.array_equal(p[0:3], a) and not p[3].any()
    assert T.pad_to_size(a, (3, 4)) is a


def test_down_scale_properties():
    """imageprep.down_scale restates skimage.transform.rescale(order=3, anti_aliasing=True) (parity unpinned: skimage is
    not installed): even output size of round(n * apix_orig / target), a constant image stays constant, the mean of a
    smooth image is kept, the value range is never exceeded, no change when the target is not coarser."""
    from helicon_b200 import imageprep as M

    yy, xx = np.mgrid[0:100, 0:140]
    img = (np.exp(-((yy - 50.0) ** 2) / 200.0) * (1 + 0.3 * np.cos(xx / 9.0))).astype(np.float32)
    out = M.down_scale(img, target_apix=5.0, apix_orig=1.3)
    assert out.shape == (26, 36) and out.shape[0] % 2 == 0 and out.shape[1] % 2 == 0
    assert out.min() >= img.min() - 1e-6 and out.max() <= img.max() + 1e-6
    assert abs(out[:, :36].mean() - img.mean()) < 0.02 * img.mean()
    c = M.down_scale(np.full((64, 64), 3.5, np.float32), 4.0, 1.0)
    assert c.shape == (16, 16) and np.allclose(c, 3.5)
    assert M.down_scale(img, 1.3, 1.3) is img and M.down_scale(img, 1.0, 1.3) is img
    odd = M.down_scale(np.ones((50, 50), np.float32), 2.0, 1.0)  # 25 -> padded to 26 with zeros (filters.py:408-411)
    assert odd.shape == (26, 26) and odd[:25, :25].min() > 0.99 or odd[1:, 1:].min() > 0.99


def test_2d_metrics_defining_properties():
    """SSIM = 1 / MS-SSIM = 1 for identical images, lower for a degraded copy, symmetric; MI of identical images = 1
    (normalised MI 2, minus 1) and ~0 for independent noise; constant images score 0 (lib/analysis.py:487-613)."""
    from helicon_b200 import imageprep as M

    rng = np.random.default_rng(3)
    yy, xx = np.mgrid[0:96, 0:96]
    a = (np.sin(xx / 5.0) * np.cos(yy / 7.0) + 1).astype(np.float32)
    noisy = (a + 0.4 * rng.standard_normal(a.shape)).astype(np.float32)
    assert abs(M.ssim_score(a, a) - 1) < 1e-9 and abs(M.ms_ssim_score(a, a) - 1) < 1e-9
    s = M.ssim_score(a, noisy)
    assert 0 < s < 0.9 and abs(s - M.ssim_score(noisy, a)) < 1e-12
    assert 0 < M.ms_ssim_score(a, noisy) < 1
    assert abs(M.mutual_information_score(a, a) - 1) < 1e-9
    ind = M.mutual_information_score(rng.random((96, 96)), rng.random((96, 96)))
    assert 0 <= ind < 0.2
    z = np.zeros((32, 32), np.float32)
    assert M.ssim_score(z, z) == 0.0 and M.ms_ssim_score(z, z) == 0.0
    with pytest.raises(ValueError):
        M.ssim_score(a, a[:10])


def test_horizontalize_and_diameter_estimate_on_a_synthetic_filament():
    """imageprep.estimate_helix_rotation_center_diameter / auto_horizontalize (lib/analysis.py:645-728,
    webApps/denovo3D/utils.py:383-426; scipy.ndimage restatement of the scikit-image calls, parity unpinned): a band of
    known width, rotated by a known angle and shifted, is brought back to horizontal and to the box centre."""
    from helicon_b200 import imageprep as M

    ny = nx = 128
    yy, xx = np.mgrid[0:ny, 0:nx].astype(np.float64)
    band = np.exp(-((yy - ny // 2) ** 2) / (2 * 6.0**2)) * (1 + 0.2 * np.cos(xx / 4.0))
    band[band < 0.05] = 0
    rot, sh, diam = M.estimate_helix_rotation_center_diameter(band)
    assert abs(rot) < 0.5 and abs(sh) < 0.5 and 25 <= diam <= 40
    tilted = M.rotate_shift_image(band, angle=12.0, post_shift=(5.0, 0.0), order=1)
    rot, sh, diam = M.estimate_helix_rotation_center_diameter(tilted)
    fixed, theta, shift = M.auto_horizontalize(tilted, refine=True)
    prof = fixed.sum(axis=1)
    assert abs(float((np.arange(ny) * prof).sum() / prof.sum()) - ny // 2) < 1.0      # centred
    r2, _, d2 = M.estimate_helix_rotation_center_diameter(np.where(fixed > 0.05, fixed, 0))  # cubic ripples off
    assert abs(r2) < 1.0 and abs(abs(theta) - 12.0) < 1.0 and 25 <= d2 <= 45            # horizontal again
    # transform_image: identity, and a pure rotation about the centre keeps the centre pixel's neighbourhood mass
    assert np.allclose(M.transform_image(band), band)
    assert abs(M.transform_image(band, rotation=90.0).sum() - band[:, 1:].sum()) < 0.05 * band.sum()


def test_tv_denoise_reduces_noise_and_keeps_the_mean():
    from helicon_b200 import imageprep as M

    rng = np.random.default_rng(0)
    clean = np.zeros((64, 64)); clean[20:44, 16:48] = 1.0
    noisy = clean + 0.3 * rng.standard_normal(clean.shape)
    out = M.denoise_tv_chambolle(noisy)
    assert np.abs(out - clean).mean() < 0.6 * np.abs(noisy - clean).mean()
    assert abs(out.mean() - noisy.mean()) < 1e-6


def test_bench_split_tail_keeps_the_candidates_and_whole_twist_rows():
    """bench.py deals the last step of every rank in pieces of whole twist rows: same candidates, same order."""
    import bench

    class T:
        def __init__(self, ti):
            self.ti = ti

    chunks = [("key", [T(i * 200 + j) for j in range(200)], 200.0) for i in range(8)]
    out = bench.split_tail(chunks, 2, 50)
    assert [len(c[1]) for c in out] == [200] * 6 + [50] * 8
    assert [t.ti for c in out for t in c[1]] == list(range(1600))
    assert all(c[1][0].ti % 50 == 0 for c in out) and abs(sum(c[2] for c in out) - 1600.0) < 1e-9
    assert [len(c[1]) for c in bench.split_tail(chunks, 2, 50, parts=2)] == [200] * 6 + [100] * 4
    assert bench.split_tail(chunks, 2, 50, parts=1) is chunks
    assert [len(c[1]) for c in bench.split_tail(chunks, 2, 10)] == [200] * 6 + [50] * 8  # cfg1: 5 rows of 10 rises
    ragged = [("key", [T(j) for j in range(24)], 1.0)] * 4  # cfg3: a twist row (600) exceeds the batch -> not split
    assert [len(c[1]) for c in bench.split_tail(ragged, 2, 600)] == [24] * 4


def test_bench_dump_outputs_writes_float_arrays_and_samples_above_the_limit(tmp_path):
    import bench

    n = 1000
    per = dict(candidate_index=np.arange(5, 5 + n, dtype=np.float64), scores=np.linspace(0, 1, n, dtype=np.float32))
    top = dict(top_scores=np.ones(3, np.float32), top_index=np.arange(3, dtype=np.float64))
    bench.dump_outputs(str(tmp_path / "all"), per, top)
    for k, v in {**per, **top}.items():
        got = np.load(tmp_path / "all" / (k + ".npy"))
        assert got.dtype == v.dtype and np.array_equal(got, v), k
    limit = 100 * 12 + 3 * 12 + 4 * bench.NPY_HEADER_BYTES  # 100 entries of 12 B, the top-K arrays, 4 headers
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), per, top, limit=limit)
    idx = np.load(tmp_path / "a" / "candidate_index.npy")
    assert len(idx) == 100 and np.array_equal(idx, np.load(tmp_path / "b" / "candidate_index.npy"))
    assert np.all(np.diff(idx) > 0) and np.array_equal(np.load(tmp_path / "a" / "scores.npy"), per["scores"][(idx - 5).astype(int)])
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= limit
    bench.dump_outputs(str(tmp_path / "c"), per, top, limit=limit - 1)  # one byte less: fewer entries, still inside
    assert sum(f.stat().st_size for f in (tmp_path / "c").iterdir()) <= limit - 1


def test_product_back_project_tables_equal_the_reference_outputs():
    """SURVEY 8(a1): the PRODUCT's host helper (not only the oracle's) against the reference's own outputs
    (tests/golden/backproject.npz, oracle/make_golden.py): coordinate tables and pixel values bit for bit."""
    from helicon_b200 import solver_linear_regression as S

    d = load("backproject")
    i = 0
    while f"case{i}_img" in d.files:
        N, s, D2, L2 = d[f"case{i}_args"]
        (X, Y, Z), pv = S.back_project_2d_coords_to_3d_coords(d[f"case{i}_img"], float(s), int(D2), int(L2))
        for got, key in ((X, "X"), (Y, "Y"), (Z, "Z"), (pv, "pix")):
            ref = d[f"case{i}_{key}"]
            assert np.asarray(got).dtype == ref.dtype and np.array_equal(got, ref), (i, key)
        i += 1
    assert i == 3

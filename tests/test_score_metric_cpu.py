"""Host side of search_grid(score_metric=...): validation, checkpoint fingerprint, the last-writer pixel table, and the
formulas the device kernels (csrc/hb2_metric.cuh) restate -- the 0.5 rescale of ms_ssim_score and histogramdd's edges --
checked against scipy / numpy on odd and even sides."""
import types

import numpy as np
import pytest

from helicon_b200 import imageprep as M


def test_unknown_metric_raises_before_any_gpu_work():
    from helicon_b200.grid import search_grid

    with pytest.raises(ValueError, match="unknown score_metric"):
        search_grid(np.zeros((32, 32), np.float32), 1.0, [1.0], [2.0], score_metric="no_such_metric")


def test_cli_refuses_an_unknown_metric():
    from helicon_b200 import denovo3DBatch

    with pytest.raises(SystemExit):
        denovo3DBatch.main(["x.mrc", "--twist", "1", "--rise", "2", "--score-metric", "no_such_metric"])


def test_fingerprint_gains_the_metric_only_when_not_cosine():
    from helicon_b200.checkpoint import fingerprint
    from helicon_b200.grid import metric_fingerprint

    img = np.arange(16, dtype=np.float32).reshape(4, 4)
    axes = (np.array([1.0]), np.array([1.0, 2.0]), np.array([3.0]))
    assert metric_fingerprint("cosine") == {}
    base = fingerprint(img, axes, apix=1.0)
    assert fingerprint(img, axes, apix=1.0, **metric_fingerprint("cosine")) == base
    fps = {m: fingerprint(img, axes, apix=1.0, **metric_fingerprint(m))
           for m in ("ssim", "ms_ssim", "mutual_information", "composite")}
    assert len(set(fps.values()) | {base}) == 5


def test_pixel_table_keeps_the_last_writer():
    """Batch.pixel_rows against a loop over the rows in the reference's order, with pixels written several times."""
    from helicon_b200.engine import Batch

    rng = np.random.default_rng(0)
    L2, D2, n = 6, 5, 80
    kk, jj = rng.integers(0, L2, n), rng.integers(0, D2, n)
    pidx = rng.permutation(1000)[:n]
    fake = types.SimpleNamespace(problem=types.SimpleNamespace(L2=L2, D2=D2), data_row_index=lambda c: (pidx, kk, jj))
    t = Batch.pixel_rows(fake, 0)
    loop = np.full(L2 * D2, -1, dtype=np.int32)
    for r, p in zip(pidx, kk * D2 + jj):
        loop[p] = r
    assert np.array_equal(t, loop) and (t == -1).any()


def _rescale_as_the_kernels(img):
    """_rescale(img, 0.5, order=1) with the index and weight formulas of hb2_metric.cuh."""
    img = np.asarray(img, dtype=np.float64)
    out = img
    for axis in (0, 1):
        n = img.shape[axis]
        z = n / float(int(np.round(n * 0.5)))
        sigma = max(0.0, (z - 1) / 2)
        r = int(4.0 * sigma + 0.5)
        w = np.exp(-0.5 / (sigma * sigma) * np.arange(-r, r + 1) ** 2.0)
        w = w / w.sum()
        a = np.moveaxis(out, axis, 0)
        idx = np.arange(n)

        def at(k):
            k = np.where(k < 0, -k - 1, np.where(k >= n, 2 * n - k - 1, k))
            return a[k]

        o = a * w[r]
        for k in range(r, 0, -1):
            o = o + (at(idx - k) + at(idx + k)) * w[r + k]
        out = np.moveaxis(o, 0, axis)
    H, W = img.shape
    Ho, Wo = int(np.round(H * 0.5)), int(np.round(W * 0.5))

    def coords(n_in, n_out):
        z = n_in / n_out
        c = (np.arange(n_out) + 0.5) * z - 0.5
        i0 = np.floor(c)
        w0 = 1.0 - (c - i0)
        return i0.astype(np.int64), w0, 1.0 - w0

    iy, wy0, wy1 = coords(H, Ho)
    ix, wx0, wx1 = coords(W, Wo)
    assert iy.min() >= 0 and iy.max() + 1 <= H - 1 and ix.min() >= 0 and ix.max() + 1 <= W - 1
    g = out
    t = 0.0
    t = t + g[iy][:, ix] * wy0[:, None] * wx0[None, :]
    t = t + g[iy][:, ix + 1] * wy0[:, None] * wx1[None, :]
    t = t + g[iy + 1][:, ix] * wy1[:, None] * wx0[None, :]
    t = t + g[iy + 1][:, ix + 1] * wy1[:, None] * wx1[None, :]
    return np.clip(t, img.min(), img.max())


@pytest.mark.parametrize("shape", [(8, 8), (9, 13), (25, 50), (42, 21), (100, 67), (200, 200), (511, 512)])
def test_rescale_formulas_match_scipy(shape):
    img = np.random.default_rng(shape[0]).standard_normal(shape)
    ref = M._rescale(img, 0.5, order=1)
    got = _rescale_as_the_kernels(img)
    assert got.shape == ref.shape == tuple(int(v) for v in np.round(np.asarray(shape) * 0.5))
    assert np.abs(got - ref).max() <= 1e-14


def _edges_as_the_kernels(v):
    """histogramdd's bin edges of float32 samples as hb2_metric.cuh computes them (float32 throughout)."""
    lo, hi = np.float32(v.min()), np.float32(v.max())
    if lo == hi:
        lo, hi = np.float32(lo - np.float32(0.5)), np.float32(hi + np.float32(0.5))
    step = np.float32(np.float32(hi - lo) / np.float32(64))
    e = (np.arange(65, dtype=np.float32) * step).astype(np.float32) + lo
    e[64] = hi
    return e.astype(np.float32)


def _bins_as_the_kernels(v, e):
    b = np.searchsorted(e, v, side="right") - 1
    b[v == e[64]] = 63
    return b


@pytest.mark.parametrize("kind", ["random", "clipped", "constant", "zero"])
def test_histogram_edges_and_bins_match_numpy(kind):
    rng = np.random.default_rng(1)
    x = rng.standard_normal(40 * 30).astype(np.float32)
    y = rng.random(40 * 30).astype(np.float32) * np.float32(3.3)
    if kind == "clipped":
        x = np.clip(x, 0, None)
    elif kind == "constant":
        x = np.full_like(x, np.float32(0.7))
    elif kind == "zero":
        x = np.zeros_like(x)
    hist, edges = np.histogramdd([x, y], bins=64)
    ex, ey = _edges_as_the_kernels(x), _edges_as_the_kernels(y)
    assert edges[0].dtype == np.float32 and np.array_equal(edges[0], ex) and np.array_equal(edges[1], ey)
    if kind in ("constant", "zero"):  # a zero range is widened to +-0.5 in float32
        assert ex[0] == np.float32(x[0] - np.float32(0.5)) and ex[64] == np.float32(x[0] + np.float32(0.5))
    counts = np.zeros((64, 64))
    np.add.at(counts, (_bins_as_the_kernels(x, ex), _bins_as_the_kernels(y, ey)), 1)
    assert np.array_equal(counts, hist)


def test_mutual_information_of_constant_images():
    """The host's values the device reproduces: one constant image gives 0, two give 0 (H(X, Y) = 0)."""
    y = np.random.default_rng(2).random((20, 20)).astype(np.float32)
    assert M.mutual_information_score(np.zeros_like(y), y) == 0.0
    assert M.mutual_information_score(np.zeros_like(y), np.ones_like(y)) == 0.0

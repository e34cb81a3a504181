"""Host-side image preparation and 2-D score metrics of the denovo3D task wrapper (SURVEY.md section 8f ranks 3-4).

``process_one_task`` / ``lsq_reconstruct`` run these once per TASK on one small 2-D image, on the host.  A grid search
scores every candidate, so ``search_grid(score_metric=...)`` runs the same three metrics on the device instead
(csrc/hb2_metric.cuh, Batch.score_metric), following these functions exactly.  The
reference implements them with scikit-image, which exists neither in the build container nor on the GPU box, so the
functions below RESTATE the published algorithms of the scikit-image 0.2x calls the reference makes with numpy /
scipy.ndimage.  **Parity unpinned**: the reference's own calls cannot be executed here (ImportError), so no golden
output exists; what is tested are the algorithms' defining properties (tests/test_host_cpu.py).

* ``down_scale``                -- lib/filters.py:375-412  (skimage.transform.rescale(order=3, anti_aliasing=True))
* ``ssim_score``                -- lib/analysis.py:487-514 (skimage.metrics.structural_similarity defaults)
* ``ms_ssim_score``             -- lib/analysis.py:517-582
* ``mutual_information_score``  -- lib/analysis.py:585-613 (skimage.metrics.normalized_mutual_information(bins=64) - 1)
"""

from __future__ import annotations

import numpy as np

from .transforms import pad_to_size


def _rescale(image, scale, order, anti_aliasing=True):
    """skimage.transform.rescale for a 2-D float image, mode="reflect", clip=True, preserve_range=False:
    output shape = round(scale * shape); Gaussian pre-filter sigma = max(0, (in/out - 1) / 2) per axis
    (resize(): anti_aliasing_sigma); ``scipy.ndimage.zoom(order, mode="reflect", grid_mode=True)`` (resize() since
    skimage 0.19); output clipped to the input's value range."""
    from scipy import ndimage as ndi

    image = np.asarray(image, dtype=np.float64)
    out_shape = tuple(int(v) for v in np.round(np.asarray(image.shape) * scale))
    factors = np.asarray(image.shape, dtype=np.float64) / np.asarray(out_shape, dtype=np.float64)
    filtered = image
    if anti_aliasing:
        sigma = np.maximum(0, (factors - 1) / 2)
        if np.any(sigma > 0):
            filtered = ndi.gaussian_filter(image, sigma, cval=0, mode="reflect")
    out = ndi.zoom(filtered, 1 / factors, order=order, mode="reflect", cval=0, grid_mode=True)
    if out.shape != out_shape:  # zoom rounds the same way; guard against a one-pixel disagreement
        out = pad_to_size(out[: out_shape[0], : out_shape[1]], out_shape)
    return np.clip(out, image.min(), image.max())


def down_scale(data, target_apix, apix_orig):
    """lib/filters.py:375-412: cubic, anti-aliased down-scaling to a larger pixel size; even output size (zero-padded)."""
    if target_apix == apix_orig or target_apix < apix_orig:
        return data
    out = _rescale(data, apix_orig / target_apix, order=3, anti_aliasing=True)
    ny, nx = out.shape
    return pad_to_size(out, shape=(ny + ny % 2, nx + nx % 2))


def _ssim(im1, im2, data_range, win_size=7, K1=0.01, K2=0.03):
    """skimage.metrics.structural_similarity with its defaults: 7 x 7 uniform window, sample covariance, mean of the
    SSIM map cropped by (win_size - 1) // 2 (Wang et al. 2004)."""
    from scipy.ndimage import uniform_filter

    im1 = np.asarray(im1, dtype=np.float64)
    im2 = np.asarray(im2, dtype=np.float64)
    if min(im1.shape) < win_size:
        raise ValueError("win_size exceeds image extent")
    NP = win_size**im1.ndim
    cov_norm = NP / (NP - 1)
    f = dict(size=win_size, mode="reflect")
    ux, uy = uniform_filter(im1, **f), uniform_filter(im2, **f)
    uxx, uyy, uxy = uniform_filter(im1 * im1, **f), uniform_filter(im2 * im2, **f), uniform_filter(im1 * im2, **f)
    vx, vy, vxy = cov_norm * (uxx - ux * ux), cov_norm * (uyy - uy * uy), cov_norm * (uxy - ux * uy)
    C1, C2 = (K1 * data_range) ** 2, (K2 * data_range) ** 2
    S = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux**2 + uy**2 + C1) * (vx + vy + C2))
    pad = (win_size - 1) // 2
    return float(S[pad:-pad, pad:-pad].mean(dtype=np.float64))


def ssim_score(img1, img2):
    """lib/analysis.py:487-514."""
    if img1.shape != img2.shape:
        raise ValueError(f"Image shapes must match: {img1.shape} vs {img2.shape}")
    try:
        data_range = max(img1.max() - img1.min(), img2.max() - img2.min())
        if data_range == 0:
            return 0.0
        return float(_ssim(img1, img2, data_range))
    except Exception:
        return 0.0


def ms_ssim_score(img1, img2):
    """lib/analysis.py:517-582: SSIM at up to five scales (each a rescale(0.5, anti_aliasing=True), bilinear), combined
    as a weighted geometric mean with the Wang et al. weights."""
    if img1.shape != img2.shape:
        raise ValueError(f"Image shapes must match: {img1.shape} vs {img2.shape}")
    try:
        data_range = max(img1.max() - img1.min(), img2.max() - img2.min())
        if data_range == 0:
            return 0.0
        all_weights = np.array([0.0448, 0.2856, 0.3001, 0.2363, 0.1333])
        vals = []
        for i in range(len(all_weights)):
            h, w = img1.shape
            if h < 8 or w < 8:
                break
            vals.append(max(_ssim(img1, img2, data_range), 0.0))
            if i < len(all_weights) - 1:
                img1 = _rescale(img1, 0.5, order=1)
                img2 = _rescale(img2, 0.5, order=1)
                data_range = max(img1.max() - img1.min(), img2.max() - img2.min())
                if data_range == 0:
                    break
        if not vals:
            return 0.0
        wts = all_weights[: len(vals)]
        wts = wts / wts.sum()
        out = 1.0
        for s, w in zip(vals, wts):
            out *= s**w
        return float(out)
    except Exception:
        return 0.0


def mutual_information_score(img1, img2):
    """lib/analysis.py:585-613: (H(X) + H(Y)) / H(X, Y) - 1 from a 64 x 64 joint histogram (Studholme et al. 1999)."""
    if img1.shape != img2.shape:
        raise ValueError(f"Image shapes must match: {img1.shape} vs {img2.shape}")
    try:
        hist, _ = np.histogramdd([np.reshape(img1, -1), np.reshape(img2, -1)], bins=64, density=True)

        def entropy(p):
            p = np.asarray(p, dtype=np.float64).ravel()
            p = p / p.sum()
            p = p[p > 0]
            return float(-(p * np.log(p)).sum())

        nmi = (entropy(hist.sum(axis=0)) + entropy(hist.sum(axis=1))) / entropy(hist)
        return float(nmi - 1.0)
    except Exception:
        return 0.0


# ---------------------------------------------------------------------------------------------------------------------
# prepare_data (pipeline.py:146-178) and the automatic tube diameter (pipeline.py:233-240): rotation / centring / size of
# the filament in the image.  scipy.ndimage stands in for the scikit-image calls (parity unpinned, see the header);
# rotate_shift_image is scipy in the reference as well.
# ---------------------------------------------------------------------------------------------------------------------
def _closing_ignore(bw):
    """skimage.morphology.closing(bw, mode="ignore") with the default footprint (3 x 3 cross): dilation then erosion,
    pixels beyond the border never decide (0 for the dilation, 1 for the erosion)."""
    from scipy import ndimage as ndi

    st = ndi.generate_binary_structure(2, 1)
    return ndi.binary_erosion(ndi.binary_dilation(bw, st, border_value=0), st, border_value=1)


def transform_image(image, scale=1.0, rotation=0.0, rotation_center=None, pre_translation=(0.0, 0.0),
                    post_translation=(0.0, 0.0), mode="constant", order=1):
    """lib/transforms.py:238-312: the affine map skimage composes there -- pre-translation, rotation / scale about
    ``rotation_center`` (default (ny/2, nx/2)), post-translation, all in (x, y) -- applied with
    ``scipy.ndimage.affine_transform`` (output pixel <- inverse-mapped input position, spline ``order``)."""
    from scipy.ndimage import affine_transform

    image = np.asarray(image, dtype=np.float64)
    cy, cx = (np.array(image.shape[:2]) / 2.0) if rotation_center is None else np.asarray(rotation_center, dtype=np.float64)
    sy, sx = (scale, scale) if np.isscalar(scale) else scale

    def T(tx, ty):
        return np.array([[1, 0, tx], [0, 1, ty], [0, 0, 1]], dtype=np.float64)

    a = np.deg2rad(rotation)
    RS = np.array([[sx * np.cos(a), -sy * np.sin(a), 0], [sx * np.sin(a), sy * np.cos(a), 0], [0, 0, 1]], dtype=np.float64)
    fwd = T(post_translation[1], post_translation[0]) @ T(cx, cy) @ RS @ T(-cx, -cy) @ T(pre_translation[1], pre_translation[0])
    inv = np.linalg.inv(fwd)  # (x, y) of the input for every (x, y) of the output
    M = np.array([[inv[1, 1], inv[1, 0]], [inv[0, 1], inv[0, 0]]])  # the same map in (row, column)
    off = np.array([inv[1, 2], inv[0, 2]])
    nd_mode = {"constant": "constant", "edge": "nearest", "symmetric": "reflect", "reflect": "mirror", "wrap": "grid-wrap"}[mode]
    return affine_transform(image, M, offset=off, order=order, mode=nd_mode, cval=0.0)


def rotate_shift_image(data, angle=0, pre_shift=(0, 0), post_shift=(0, 0), rotation_center=None, order=1):
    """lib/transforms.py:315-367 (scipy.ndimage.affine_transform in the reference as well; float32 matrix / offset)."""
    from scipy.ndimage import affine_transform

    if angle == 0 and pre_shift == [0, 0] and post_shift == [0, 0]:
        return data * 1.0
    ny, nx = data.shape
    if rotation_center is None:
        rotation_center = np.array((ny // 2, nx // 2), dtype=np.float32)
    ang = np.deg2rad(angle)
    m = np.array([[np.cos(ang), np.sin(ang)], [-np.sin(ang), np.cos(ang)]], dtype=np.float32)
    offset = -np.dot(m, np.array(post_shift, dtype=np.float32).T)
    offset += np.array(rotation_center, dtype=np.float32).T - np.dot(m, np.array(rotation_center, dtype=np.float32).T)
    offset += -np.array(pre_shift, dtype=np.float32).T
    return affine_transform(data, matrix=m, offset=offset, order=order, mode="constant")


def _periodic(v, lo=-180.0, hi=180.0):
    """lib/angular.py:84-108."""
    import math

    if lo <= v <= hi:
        return v
    t = math.fmod(v - lo, hi - lo)
    return t + lo if t >= 0 else t + hi


def estimate_helix_rotation_center_diameter(data, estimate_rotation=True, estimate_center=True, threshold=0):
    """lib/analysis.py:645-728: intensity-weighted second moments of the (morphologically closed) support -> rotation to
    horizontal (degrees), vertical shift to the box centre (pixels), diameter = vertical extent after the rotation."""
    data = np.asarray(data)
    ny, nx = data.shape

    def weighted(mask, inten):
        ys, xs = np.where(mask)
        if len(ys) < 2:
            return 0.0, 0.0, ny
        w = inten[ys, xs].astype(np.float64)
        w = w - w.min() + 1e-8
        cw = w.sum()
        cy, cx = (ys * w).sum() / cw, (xs * w).sum() / cw
        uy, ux = ys - cy, xs - cx
        i_yy, i_xx, i_xy = (uy * uy * w).sum() / cw, (ux * ux * w).sum() / cw, (uy * ux * w).sum() / cw
        angle = np.rad2deg(0.5 * np.arctan2(2.0 * i_xy, i_yy - i_xx)) + 90.0
        if abs(angle) > 90.0:
            angle -= 180.0
        return angle, (ny // 2 - cy) if estimate_center else 0.0, int(ys.max() - ys.min() + 1)

    mask = _closing_ignore(data > threshold)
    if not mask.any():
        return 0.0, 0.0, ny
    if estimate_rotation:
        rotation = _periodic(weighted(mask, data)[0])
        rotated = transform_image(data, rotation=rotation)
    else:
        rotation, rotated = 0.0, data
    mask_rot = _closing_ignore(rotated > threshold)
    if not mask_rot.any():
        return rotation, 0.0, ny
    _, shift_y, diameter = weighted(mask_rot, rotated)
    return rotation, shift_y, diameter


def auto_horizontalize(data, refine=False):
    """webApps/denovo3D/utils.py:383-426: rotate / shift the image so that the filament is horizontal and centred; with
    ``refine`` a Nelder-Mead search (scipy ``fmin``, xtol 1e-2) maximises the spread of the mirrored row-sum profile."""
    data_work = np.clip(data, 0, None)
    theta, shift_y, _ = estimate_helix_rotation_center_diameter(data)
    if refine:
        from scipy.optimize import fmin

        def score(x):
            tmp = rotate_shift_image(data_work, angle=x[0], post_shift=(x[1], 0))
            y = np.sum(tmp, axis=1)[1:]
            y = y + y[::-1]
            return -np.std(y)

        theta, shift_y = fmin(score, x0=(theta, shift_y), xtol=1e-2, disp=0)
    return rotate_shift_image(data, angle=theta, post_shift=(shift_y, 0), order=3), theta, shift_y


def denoise_tv_chambolle(image, weight=0.1, eps=2.0e-4, max_num_iter=200):
    """skimage.restoration.denoise_tv_chambolle with its defaults for one 2-D image (Chambolle 2004: projected
    gradient on the dual of the ROF model; same update, same stopping rule |dE| < eps * E0)."""
    image = np.asarray(image, dtype=np.float64)
    p = np.zeros((2,) + image.shape)
    g = np.zeros_like(p)
    d = np.zeros_like(image)
    out, E_prev, E0 = image, 0.0, None
    for i in range(max_num_iter):
        if i > 0:
            d = -p.sum(0)
            d[1:, :] += p[0, :-1, :]
            d[:, 1:] += p[1, :, :-1]
            out = image + d
        else:
            out = image
        E = float((d**2).sum())
        g[0, :-1, :] = np.diff(out, axis=0)
        g[1, :, :-1] = np.diff(out, axis=1)
        norm = np.sqrt((g**2).sum(axis=0))[np.newaxis, ...]
        E += weight * float(norm.sum())
        tau = 1.0 / (2.0 * image.ndim)
        norm = norm * (tau / weight) + 1.0
        p = (p - tau * g) / norm
        E /= float(image.size)
        if i == 0:
            E0, E_prev = E, E
        else:
            if abs(E_prev - E) < eps * E0:
                break
            E_prev = E
    return out

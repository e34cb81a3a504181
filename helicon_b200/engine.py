"""Python host objects over the C ABI: Problem (one image + in-plane geometry)
and Batch (candidates with a common 3-D length solved together on one GPU)."""

from __future__ import annotations

import ctypes as C

import numpy as np
from scipy.sparse import csr_matrix

from . import _lib
from .planner import BatchPlan, CandidateSpec

DEFAULT_OPTIONS = dict(
    max_iter=1000, atol=1e-4, btol=1e-4, conlim=1e8, check_every=8, clip_pred=0, trf_max_iter=200, trf_tol=1e-2,
    fixed_iters=0, profile=0, norm_mode=1,
)


MODELS = ("elasticnet", "lasso", "ridge")


def model_params(algorithm):
    """(kind, alpha, l1_ratio) of a sklearn-model ``algorithm`` dict with the reference's defaults (alpha 1 for ridge,
    1e-4 otherwise; l1_ratio 0.5), or None for ``None`` / ``{"model": "lsq"}``.  Raises before any GPU work."""
    model = "lsq" if algorithm is None else algorithm.get("model", "lsq")
    if model == "lsq":
        return None
    if model not in MODELS:
        raise NotImplementedError(f"helicon_b200: algorithm model {model!r} is not implemented on the CUDA path "
                                  "(lsq, elasticnet, lasso, ridge are; 'lreg' / 'ard' need the dense matrix)")
    alpha = float(algorithm.get("alpha", 1 if model == "ridge" else 1e-4))
    l1_ratio = 1.0 if model == "lasso" else (0.0 if model == "ridge" else float(algorithm.get("l1_ratio", 0.5)))
    if not alpha > 0 or not 0 <= l1_ratio <= 1:
        raise ValueError(f"helicon_b200: model {model!r} needs alpha > 0 and 0 <= l1_ratio <= 1 "
                         f"(got alpha={alpha}, l1_ratio={l1_ratio})")
    return model, alpha, l1_ratio


def _stream_handle(stream):
    if stream is None:
        return None
    if isinstance(stream, int):
        return C.c_void_p(stream)
    return C.c_void_p(int(stream.cuda_stream))  # torch.cuda.Stream or engine.Stream


class Stream:
    """A non-blocking CUDA stream owned by the library (``hb2_stream_create``)."""

    def __init__(self, device=0):
        lib = _lib.require_gpu()
        self.device = int(device)
        h = C.c_void_p()
        _lib.check(lib.hb2_stream_create(self.device, C.byref(h)))
        self.cuda_stream = int(h.value)

    def close(self):
        if getattr(self, "cuda_stream", None):
            _lib.load().hb2_stream_destroy(self.device, C.c_void_p(self.cuda_stream))
            self.cuda_stream = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ScoreMap:
    """Device-resident score map + iteration map of one search over ``n`` flat task indices, with the top-K selected
    by a CUDA kernel (include/helicon_b200.h: hb2_scoremap_*; the reference's host-side collect / sort / top-N of
    app.py:2482-2539).  ``scatter(batch, task_indices)`` after ``batch.solve()``; ``topk(k)``; ``read()``.
    ``__cuda_array_interface__`` exposes the 3*n int32 words (float32 scores, int32 iterations, uint32 flags) so that
    ``torch.as_tensor(score_map, device="cuda")`` is a zero-copy view NCCL can all-gather."""

    def __init__(self, n, device=0):
        lib = _lib.require_gpu()
        self.n, self.device = int(n), int(device)
        self._h = C.c_void_p()
        _lib.check(lib.hb2_scoremap_create(C.byref(self._h), self.n, self.device))
        ptr = lib.hb2_scoremap_device_ptr(self._h)
        self.__cuda_array_interface__ = dict(shape=(3 * self.n,), typestr="<i4", data=(int(ptr), False), version=3)

    def scatter(self, batch, task_indices, flags):
        idx = np.ascontiguousarray(task_indices, dtype=np.int64)
        fl = np.ascontiguousarray(flags, dtype=np.uint32)
        assert len(idx) == batch.nc == len(fl)
        _lib.check(_lib.load().hb2_batch_scatter_scores(batch._h, self._h, _lib.ptr(idx), _lib.ptr(fl)))

    def restore(self, task_indices, scores, itn, flags):
        """Entries of an interrupted search of the same grid (checkpoint.ScoreTileStore) written into the device maps."""
        idx = np.ascontiguousarray(task_indices, dtype=np.int64)
        sc = np.ascontiguousarray(scores, dtype=np.float32)
        it = np.ascontiguousarray(itn, dtype=np.int32)
        fl = np.ascontiguousarray(flags, dtype=np.uint32)
        assert len(idx) == len(sc) == len(it) == len(fl)
        _lib.check(_lib.load().hb2_scoremap_restore(self._h, len(idx), _lib.ptr(idx), _lib.ptr(sc), _lib.ptr(it), _lib.ptr(fl)))

    def merge(self, gathered_ptr, n_maps, stream=None):
        """Fold ``n_maps`` maps of other ranks (device buffer of n_maps x 3n words, e.g. filled by an all-gather) in."""
        _lib.check(_lib.load().hb2_scoremap_merge(self._h, C.c_void_p(int(gathered_ptr)), int(n_maps), _stream_handle(stream)))

    def topk(self, k, stream=None):
        sc = np.zeros(int(k), dtype=np.float32)
        ix = np.zeros(int(k), dtype=np.int64)
        _lib.check(_lib.load().hb2_scoremap_topk(self._h, int(k), _lib.ptr(sc), _lib.ptr(ix), _stream_handle(stream)))
        keep = ix >= 0
        return sc[keep], ix[keep]

    def read(self, stream=None):
        sc = np.empty(self.n, dtype=np.float32)
        it = np.empty(self.n, dtype=np.int32)
        fl = np.empty(self.n, dtype=np.uint32)
        _lib.check(_lib.load().hb2_scoremap_read(self._h, _lib.ptr(sc), _lib.ptr(it), _lib.ptr(fl), _stream_handle(stream)))
        return sc, it, fl

    def close(self):
        if getattr(self, "_h", None):
            _lib.load().hb2_scoremap_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Problem:
    """Image + the geometry that does not depend on (twist, rise, csym)."""

    def __init__(self, image, scale2d_to_3d, D2, L2, D3, rmin, rmax, device=0, stream=None, interpolation="nn"):
        lib = _lib.require_gpu()
        if interpolation not in ("nn", "linear"):
            raise NotImplementedError(
                f"helicon_b200: interpolation={interpolation!r} is not implemented on the CUDA path (only 'nn' and 'linear'); "
                "there is no CPU fallback"
            )
        image = np.ascontiguousarray(image, dtype=np.float32)
        ny, nx = image.shape
        # interpolation is a layout hint only (internal voxel order); every batch type runs on either order
        self.geom = _lib.Geometry(ny, nx, float(scale2d_to_3d), int(D2), int(L2), int(D3), float(rmin), int(rmax),
                                  1 if interpolation == "linear" else 0)
        self.device = int(device)
        self.stream = _stream_handle(stream)
        self._h = C.c_void_p()
        _lib.check(lib.hb2_problem_create(C.byref(self._h), _lib.ptr(image), C.byref(self.geom), self.device, self.stream))
        self.ndisk = lib.hb2_problem_ndisk(self._h)
        self.D2, self.L2, self.D3 = int(D2), int(L2), int(D3)
        self.s = float(scale2d_to_3d)

    def rank_table(self):
        out = np.empty(self.D2 * self.D2, dtype=np.int32)
        _lib.check(_lib.load().hb2_problem_rank_table(self._h, _lib.ptr(out)))
        return out.reshape(self.D2, self.D2)

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _lib.load().hb2_problem_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Batch:
    """Candidates (CandidateSpec) of one Problem with a common L3."""

    def __init__(self, problem: Problem, L3: int, specs, need_views=True, stream=None):
        """``stream``: the stream ALL work of this batch runs on (default: the problem's)."""
        lib = _lib.require_gpu()
        self.problem = problem
        self._stream_ref = stream  # keep the stream object alive as long as the batch
        self.L3 = int(L3)
        self.plan = BatchPlan(problem.s, problem.D2, problem.L2, self.L3, specs)
        nA = len(self.plan.angles)
        self.nvalid = np.zeros(nA, dtype=np.int32)
        self.tie = np.zeros(nA, dtype=np.int32)
        self._h = C.c_void_p()
        _lib.check(
            lib.hb2_batch_begin(
                C.byref(self._h), problem._h, self.L3, self.plan.MC, nA, _lib.ptr(self.plan.cos_sin),
                _lib.ptr(self.nvalid), _lib.ptr(self.tie), problem.stream if stream is None else _stream_handle(stream),
            )
        )
        req = self.plan.exact_map_requests(self.tie)
        if req is not None:  # in-plane tie views: exact per-column maps appended to the angle table
            nv_ex = np.zeros(len(req[0]), dtype=np.int32)
            _lib.check(lib.hb2_batch_add_exact_maps(self._h, len(req[0]), _lib.ptr(req[0]), _lib.ptr(req[1]), _lib.ptr(nv_ex)))
            self.nvalid = np.concatenate([self.nvalid, nv_ex])
            self.tie = np.concatenate([self.tie, np.zeros(len(nv_ex), dtype=np.int32)])
        self._amap_cache = {}
        self.plan.finalize(self.nvalid, lambda a: self.angle_map(a) >= 0)
        p = self.plan
        if p.n_tie:
            _lib.check(lib.hb2_batch_set_ties(self._h, p.n_tie, p.tie_TS, _lib.ptr(p.tie_zlo), _lib.ptr(p.tie_up),
                                              _lib.ptr(p.tie_rowvalid)))
        _lib.check(
            lib.hb2_batch_create(
                self._h, len(p.cands), _lib.ptr(p.cands), len(p.views), _lib.ptr(p.views), len(p.colk),
                _lib.ptr(p.colk), len(p.pairs), _lib.ptr(p.pairs),
            )
        )
        self.n = self.L3 * problem.ndisk
        self.nc = len(p.cands)
        self.results = None

    # -- half sets (fsc_test) -----------------------------------------------
    def set_pixel_masks(self, masks, cand_mask):
        """masks: (n_masks, L2*D2) uint8 over pixel ids pid = k*D2 + j; cand_mask[c] = mask index or -1."""
        masks = np.ascontiguousarray(masks, dtype=np.uint8).reshape(-1, self.problem.L2 * self.problem.D2)
        cand_mask = np.ascontiguousarray(cand_mask, dtype=np.int32)
        assert cand_mask.shape == (self.nc,)
        _lib.check(_lib.load().hb2_batch_set_pixel_masks(self._h, len(masks), _lib.ptr(masks), _lib.ptr(cand_mask)))

    # -- solve -------------------------------------------------------------
    def solve(self, **opts):
        o = dict(DEFAULT_OPTIONS)
        o.update(opts)
        so = _lib.SolveOptions(**o)
        res = np.zeros(self.nc, dtype=_lib.RESULT_DTYPE)
        _lib.check(_lib.load().hb2_batch_solve(self._h, C.byref(so), _lib.ptr(res)))
        res["n_data_rows"] = self.plan.cand_n_data_rows
        self.results = res
        return res

    def real_rows(self, c):
        """Mask of the real rows of candidate ``c`` over its padded rows (data rows of ``data_row_index`` and every
        symmetry row), as regularized._CenteredOperator builds it."""
        nd_pad, tot = self.rows_padded(c)
        real = np.zeros(tot, dtype=np.uint8)
        real[self.data_row_index(c)[0]] = 1
        real[nd_pad:] = 1
        return real

    def solve_model(self, algorithm, clip_pred=0, gap_factor=0.05, max_iter=4000, check_every=10):
        """ElasticNet / Lasso / Ridge (SLR:272-342) for every candidate at once on the device (hb2_batch_solve_model):
        the objectives, schedule and stop rules of regularized.solve_model; each candidate's positive constraint is its
        CandidateSpec.positive.  Returns the result array of ``solve`` (itn = iterations of the final fit, flags with
        HB2_FLAG_NOT_CONVERGED where max_iter ended it)."""
        model, alpha, l1_ratio = model_params(algorithm)
        lib = _lib.load()
        if not getattr(self, "_real_set", False):
            for c in range(self.nc):
                real = self.real_rows(c)
                _lib.check(lib.hb2_batch_set_real_rows(self._h, c, _lib.ptr(real), len(real)))
            self._real_set = True
        v = np.random.default_rng(0).standard_normal(self.n)
        v /= np.linalg.norm(v)
        o = _lib.ModelOptions(kind=_lib.MODEL_RIDGE if model == "ridge" else _lib.MODEL_ENET, alpha=alpha,
                              l1_ratio=l1_ratio, gap_factor=float(gap_factor), max_iter=int(max_iter),
                              check_every=int(check_every), clip_pred=int(clip_pred), power_start=_lib.ptr(v))
        res = np.zeros(self.nc, dtype=_lib.RESULT_DTYPE)
        _lib.check(lib.hb2_batch_solve_model(self._h, C.byref(o), _lib.ptr(res)))
        res["n_data_rows"] = self.plan.cand_n_data_rows
        self.results = res
        return res

    def model_info(self, c):
        """dict(alpha, iterations, gap, lipschitz) of candidate ``c``'s final fit (gap: the relative CG residual for
        ridge, the last relative update for ridge with the positive constraint; lipschitz 0 for CG)."""
        out = np.zeros(4, dtype=np.float64)
        _lib.check(_lib.load().hb2_batch_model_info(self._h, int(c), _lib.ptr(out)))
        return dict(alpha=float(out[0]), iterations=int(out[1]), gap=float(out[2]), lipschitz=float(out[3]))

    def pixel_rows(self, c):
        """Last-writer table of candidate ``c`` over the (L2, D2) image: for pixel id k*D2 + j the padded data row that
        _metric_2d's ``pred_2d.ravel()[pid] = pred`` leaves there (the last row of that pixel in the reference's order
        (copy, k, j); numpy's fancy assignment keeps the last of repeated indices), or -1."""
        pidx, kk, jj = self.data_row_index(c)
        D2 = self.problem.D2
        table = np.full(self.problem.L2 * D2, -1, dtype=np.int32)
        table[(kk * D2 + jj).astype(np.int64)] = pidx
        return table

    def set_pixel_rows(self):
        """Upload every candidate's pixel_rows table (hb2_batch_set_pixel_rows); the grid search does it on the
        pipeline's worker thread while the previous batch is being solved."""
        lib = _lib.load()
        for c in range(self.nc):
            t = self.pixel_rows(c)
            _lib.check(lib.hb2_batch_set_pixel_rows(self._h, c, _lib.ptr(t), self.problem.L2, self.problem.D2))
        self._pixel_rows_set = True

    def score_metric(self, metric, clip_pred=0, parts=False):
        """Replace every candidate's score by the 2-D ``metric`` ("ssim", "ms_ssim", "mutual_information",
        "composite") of _metric_2d, computed on the device (hb2_batch_score_metric) after ``solve`` or ``solve_model``.
        Returns the result array of that solve with the new scores; ``parts=True`` also returns [nc, 4] float64
        (cosine, ssim, ms_ssim, mutual information)."""
        if metric not in _lib.METRICS:
            raise ValueError(f"unknown score_metric {metric!r}")
        if self.results is None:
            raise _lib.HeliconB200Error("Batch.score_metric before a solve")
        if not getattr(self, "_pixel_rows_set", False):
            self.set_pixel_rows()
        sc = np.empty(self.nc, dtype=np.float32)
        out = np.empty((self.nc, 4), dtype=np.float64) if parts else None
        _lib.check(_lib.load().hb2_batch_score_metric(self._h, _lib.METRICS[metric], int(clip_pred), _lib.ptr(sc),
                                                      _lib.ptr(out) if parts else None))
        res = self.results.copy()
        res["score"] = sc
        self.results = res
        return (res, out) if parts else res

    def apply_all(self, xs=None, ys=None):
        """The MODE_PLAIN products over all candidates in one launch each (tests): ``xs`` [nc, n] -> list of row
        vectors, or ``ys`` (list of row vectors) -> [nc, n]."""
        lib = _lib.load()
        tots = [self.rows_padded(c)[1] for c in range(self.nc)]
        if xs is not None:
            x = np.ascontiguousarray(xs, dtype=np.float32).reshape(self.nc, self.n)
            y = np.empty(sum(tots), dtype=np.float32)
            _lib.check(lib.hb2_batch_apply_all(self._h, 0, _lib.ptr(x), _lib.ptr(y)))
            return np.split(y, np.cumsum(tots)[:-1])
        y = np.ascontiguousarray(np.concatenate([np.asarray(v, dtype=np.float32) for v in ys]))
        assert len(y) == sum(tots)
        x = np.empty((self.nc, self.n), dtype=np.float32)
        _lib.check(lib.hb2_batch_apply_all(self._h, 1, _lib.ptr(y), _lib.ptr(x)))
        return x

    def timing(self):
        out = np.zeros(16, dtype=np.float64)
        _lib.check(_lib.load().hb2_batch_timing(self._h, _lib.ptr(out)))
        return dict(lsmr_ms=out[0], trf_ms=out[1], score_ms=out[2], launches=int(out[3]), iterations=int(out[4]),
                    fwd_data_ms=out[5], fwd_sym_ms=out[6], adj_ms=out[7], update_ms=out[8], scalar_ms=out[9],
                    fwd_data_launches=int(out[10]), adj_launches=int(out[11]), update_launches=int(out[12]), norm_ms=out[14],
                    metric_ms=out[15])

    def trf_trace(self, c):
        out = np.zeros((24, 8), dtype=np.float64)
        rc = _lib.check(_lib.load().hb2_batch_trf_trace(self._h, int(c), _lib.ptr(out), 24))
        nit, status = rc // 16, rc % 16 - 1
        return out[: min(nit, 24)], nit, status

    def x(self, c):
        out = np.empty(self.n, dtype=np.float32)
        _lib.check(_lib.load().hb2_batch_get_x(self._h, int(c), _lib.ptr(out)))
        return out

    def mask2d(self):
        return self.problem_rank3d() >= 0

    def problem_rank3d(self):
        """disk rank table on the 3-D grid (D3 x D3)."""
        D3 = self.problem.D3
        g = self.problem.geom
        j = np.arange(D3) - D3 // 2
        Y, X = np.meshgrid(j, j, indexing="ij")
        r2 = X * X + Y * Y
        m = r2 < g.rmax * g.rmax
        if 0 < g.rmin < g.rmax:
            m &= r2 >= g.rmin * g.rmin
        rank = np.full((D3, D3), -1, dtype=np.int64)
        rank[m] = np.arange(int(m.sum()))
        return rank

    def rec3d(self, c):
        """Scatter x into the (L3, D3, D3) volume (SLR:532-538)."""
        D3 = self.problem.D3
        m = self.problem_rank3d() >= 0
        vol = np.zeros((self.L3, D3, D3), dtype=np.float32)
        vol[:, m] = self.x(c).reshape(self.L3, -1)
        return vol

    # -- exports (drop-in builders, tests) ---------------------------------
    def ray_valid(self):
        out = np.empty((len(self.nvalid), self.problem.D2), dtype=np.uint8)  # incl. exact-map angles
        _lib.check(_lib.load().hb2_batch_ray_valid(self._h, _lib.ptr(out)))
        return out

    def angle_map(self, a):
        """sample -> voxel map of angle a: [ray j, depth i] reference disk rank or -1 (cached)."""
        a = int(a)
        if a not in self._amap_cache:
            D2 = self.problem.D2
            out = np.empty(D2 * D2, dtype=np.int32)
            _lib.check(_lib.load().hb2_batch_angle_map(self._h, a, _lib.ptr(out)))
            self._amap_cache[a] = out.reshape(D2, D2)
        return self._amap_cache[a]

    def rows_padded(self, c):
        nd = C.c_int64()
        tot = _lib.load().hb2_batch_rows_padded(self._h, int(c), C.byref(nd))
        _lib.check(tot)
        return int(nd.value), int(tot)

    def rhs_padded(self, c):
        nd, _ = self.rows_padded(c)
        out = np.empty(nd, dtype=np.float32)
        _lib.check(_lib.load().hb2_batch_rhs(self._h, int(c), _lib.ptr(out)))
        return out

    def data_row_index(self, c):
        """For every real data row, in the reference's order (copy, k, j), its
        index in the padded layout [view slot][j][column slot] (row stride ZMP), plus (k, j)."""
        D2, L3, MC = self.problem.D2, self.L3, self.plan.MC
        ZMC = L3 * MC
        ZMP = (ZMC + 3) // 4 * 4
        rv = self.ray_valid()
        base = int(self.plan.cands[c]["view_begin"])
        idx, kk, jj = [], [], []
        for (a, zi, h, cc, nrows), slot in zip(self.plan.cand_views[c], self.plan.cand_view_slots[c]):
            vi = slot - base
            if zi.ndim == 1:
                js = np.nonzero(rv[a])[0]
                fill = np.zeros(L3, dtype=np.int64)
                for k in np.nonzero(zi >= 0)[0]:
                    z = int(zi[k])
                    zm = z * MC + fill[z]
                    fill[z] += 1
                    idx.append(vi * (D2 * ZMP) + js * ZMP + zm)
                    kk.append(np.full(len(js), k))
                    jj.append(js)
            else:  # tie view: column slots, per-(column, ray) validity
                va = self.angle_map(a) >= 0
                inside = (zi >= 0) & (zi < L3)
                cols = np.nonzero(inside.any(axis=1))[0]
                for t, k in enumerate(cols):
                    js = np.nonzero((va & inside[k][None, :]).any(axis=1))[0]
                    idx.append((vi + t // ZMC) * (D2 * ZMP) + js * ZMP + (t % ZMC))
                    kk.append(np.full(len(js), k))
                    jj.append(js)
        if not idx:
            return np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, np.int64)
        return np.concatenate(idx), np.concatenate(kk), np.concatenate(jj)

    def data_csr(self, c):
        """A_data, b, b_pid of SLR:1651-1654 assembled from the GPU-built maps."""
        D2, L3 = self.problem.D2, self.L3
        nd = self.problem.ndisk
        rv = self.ray_valid()
        rows, cols = [], []
        r0 = 0
        for a, zi, h, cc, nrows in self.plan.cand_views[c]:
            fm = self.angle_map(a)
            if zi.ndim == 1:
                js = np.nonzero(rv[a])[0]
                sub = fm[js]  # (nj, D2)
                hit = sub >= 0
                per_ray = hit.sum(axis=1)
                ray_local = np.repeat(np.arange(len(js)), per_ray)
                vox = sub[hit]
                for k in np.nonzero(zi >= 0)[0]:
                    z = int(zi[k])
                    rows.append(r0 + ray_local)
                    cols.append(z * nd + vox)
                    r0 += len(js)
            else:  # tie view: every sample carries its own slice (zi[k, i])
                inside = (zi >= 0) & (zi < L3)
                for k in np.nonzero(inside.any(axis=1))[0]:
                    hit = (fm >= 0) & inside[k][None, :]  # [j, i]
                    js = np.nonzero(hit.any(axis=1))[0]
                    sub = hit[js]
                    ray_local = np.repeat(np.arange(len(js)), sub.sum(axis=1))
                    jj_, ii_ = np.nonzero(sub)
                    rows.append(r0 + ray_local)
                    cols.append(zi[k][ii_] * nd + fm[js][jj_, ii_])
                    r0 += len(js)
        pidx, kk, jj = self.data_row_index(c)
        b = self.rhs_padded(c)[pidx] if len(pidx) else np.zeros(0, np.float32)
        if rows:
            rows, cols = np.concatenate(rows), np.concatenate(cols)
        else:
            rows, cols = np.zeros(0, np.int64), np.zeros(0, np.int64)
        A = csr_matrix((np.ones(len(rows), dtype=np.float32), (rows, cols)), shape=(r0, L3 * nd), dtype=np.float32)
        return A, b.astype(np.float32), (kk * D2 + jj).astype(np.int32)

    def sym_rows(self, c):
        n = C.c_int32()
        lib = _lib.load()
        _lib.check(lib.hb2_batch_sym_rows(self._h, int(c), C.byref(n), None, None, 0))
        a = np.empty(n.value, dtype=np.int32)
        b = np.empty(n.value, dtype=np.int32)
        if n.value:
            _lib.check(lib.hb2_batch_sym_rows(self._h, int(c), C.byref(n), _lib.ptr(a), _lib.ptr(b), n.value))
        return a, b

    def sym_row_order(self, c):
        """Position, inside the symmetry block of the padded row vectors, of the reference's r-th symmetry row."""
        n = C.c_int32()
        lib = _lib.load()
        _lib.check(lib.hb2_batch_sym_rows(self._h, int(c), C.byref(n), None, None, 0))
        order = np.zeros(max(n.value, 1), dtype=np.int32)
        if n.value:
            _lib.check(lib.hb2_batch_sym_order(self._h, int(c), _lib.ptr(order), n.value))
        return order[: n.value]

    def sym_csr(self, c):
        """A_hsym, b_hsym of SLR:1289-1298 (or (None, None))."""
        a, b = self.sym_rows(c)
        m = len(a)
        if m == 0:
            return None, None
        rows = np.repeat(np.arange(m), 2)
        cols = np.stack([a, b], axis=1).ravel()
        vals = np.tile(np.array([1, -1], dtype=np.float32), m)
        A = csr_matrix((vals, (rows, cols)), shape=(m, self.n), dtype=np.float32)
        return A, np.zeros(m, dtype=np.float32)

    def apply_forward(self, c, x):
        x = np.ascontiguousarray(x, dtype=np.float32)
        assert x.shape == (self.n,)
        _, tot = self.rows_padded(c)
        y = np.empty(tot, dtype=np.float32)
        _lib.check(_lib.load().hb2_batch_apply_forward(self._h, int(c), _lib.ptr(x), _lib.ptr(y)))
        return y

    def apply_adjoint(self, c, y):
        y = np.ascontiguousarray(y, dtype=np.float32)
        _, tot = self.rows_padded(c)
        assert y.shape == (tot,)
        x = np.empty(self.n, dtype=np.float32)
        _lib.check(_lib.load().hb2_batch_apply_adjoint(self._h, int(c), _lib.ptr(y), _lib.ptr(x)))
        return x

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            _lib.load().hb2_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class ExplicitBatch(Batch):
    """ONE candidate whose data rows are explicit (general orientation tilt/psi/dy and/or trilinear interpolation,
    ``hb2_batch_explicit_rows``): built on the GPU with the reference's float64 operation sequence, applied by CSR
    kernels; symmetry rows, LSMR/TRF and the score are the batch's usual kernels."""

    def __init__(self, problem: Problem, L3: int, spec: CandidateSpec, tilt_degree=0.0, psi_degree=0.0, dy_pixel=0.0,
                 interpolation="nn", stream=None, pixel_mask=None):
        from scipy.spatial.transform import Rotation as R

        from . import planner

        lib = _lib.require_gpu()
        if interpolation not in ("nn", "linear"):
            raise NotImplementedError(f"helicon_b200: interpolation={interpolation!r} (only 'nn' and 'linear')")
        self.problem = problem
        self._stream_ref = stream
        self.L3 = int(L3)
        D2, L2 = problem.D2, problem.L2
        linear = interpolation == "linear"
        # nearest neighbour: the batch's own symmetry rows (pairs from the planner); trilinear: explicit rows as well
        plan_spec = CandidateSpec(spec.twist, spec.rise_pixel, spec.csym, spec.min_projection_lines,
                                  -1 if linear else spec.min_sym_pairs, spec.positive)
        self.plan = BatchPlan(problem.s, D2, L2, self.L3, [plan_spec], exact_ties=False)
        st = problem.stream if stream is None else _stream_handle(stream)
        dummy = np.array([[1.0, 0.0]], dtype=np.float64)  # the in-plane maps are not used by explicit rows
        self.nvalid = np.zeros(1, dtype=np.int32)
        self.tie = np.zeros(1, dtype=np.int32)
        self._h = C.c_void_p()
        _lib.check(lib.hb2_batch_begin(C.byref(self._h), problem._h, self.L3, 1, 1, _lib.ptr(dummy), _lib.ptr(self.nvalid),
                                       _lib.ptr(self.tie), st))
        self.tie[:] = 0
        copies = planner.data_copies(spec.rise_pixel, spec.csym, self.L3, L2)
        ang = np.array([spec.twist * h + 360 * c / spec.csym for h, c in copies], dtype=np.float64)
        mats = np.ascontiguousarray(R.from_euler("z", ang.reshape(-1, 1), degrees=True).as_matrix().reshape(-1, 9))
        zshift = np.array([h * spec.rise_pixel for h, _ in copies], dtype=np.float64)
        geo = _lib.ExplicitGeometry()
        geo.interpolation = 1 if interpolation == "linear" else 0
        geo.dy_pixel = float(dy_pixel)
        myx = R.from_euler("yx", (tilt_degree, psi_degree), degrees=True).as_matrix().reshape(-1)
        for q in range(9):
            geo.rot_yx[q] = float(myx[q])
        Xt, Zt = planner.reference_xz_tables(problem.s, D2, L2)
        if pixel_mask is not None:  # half set (fsc_test): rows of the other half are dropped after the early stop
            pm = np.ascontiguousarray(pixel_mask, dtype=np.uint8).reshape(L2 * D2)
            _lib.check(lib.hb2_batch_explicit_pixel_mask(self._h, _lib.ptr(pm)))
        used, m, nnz = C.c_int32(), C.c_int64(), C.c_int64()
        self.rows_per_copy = np.zeros(len(copies), dtype=np.int32)
        _lib.check(lib.hb2_batch_explicit_rows(
            self._h, C.byref(geo), len(copies), _lib.ptr(mats), _lib.ptr(zshift), _lib.ptr(Xt), _lib.ptr(Zt),
            int(spec.min_projection_lines), C.byref(used), _lib.ptr(self.rows_per_copy), C.byref(m), C.byref(nnz)))
        self.copies_used, self.m_rows, self.nnz = int(used.value), int(m.value), int(nnz.value)
        self.m_sym_explicit = 0
        if linear and spec.min_sym_pairs >= 0:
            if problem.D3 != D2:
                raise NotImplementedError("helicon_b200: trilinear rows need reconstruct_diameter_3d == 2d diameter")
            tab = planner.trilinear_pair_table(spec.twist, spec.rise_pixel, spec.csym, self.L3)
            ms = C.c_int64()
            _lib.check(lib.hb2_batch_explicit_sym_rows(self._h, len(tab), _lib.ptr(tab), int(spec.min_sym_pairs),
                                                       C.byref(ms)))
            self.m_sym_explicit = int(ms.value)
        # pairs (symmetry rows) from the planner; views replaced by pseudo views over the explicit rows
        p = self.plan
        p.finalize(np.zeros(len(p.angles), dtype=np.int64))
        ZMP = (self.L3 + 3) // 4 * 4
        rpv = D2 * ZMP
        nv = (self.m_rows + self.m_sym_explicit + rpv - 1) // rpv
        views = np.zeros(nv, dtype=_lib.VIEW_DTYPE)
        views["angle"] = 0
        views["tie"] = 0
        views["dup_of"] = -1
        views["mult"] = 1
        views["col_begin"] = 0
        colk = np.full(self.L3, -1, dtype=np.int32)
        p.cands[0]["view_begin"], p.cands[0]["view_count"] = 0, nv
        p.cands[0]["flags_in"] = 0
        p.views, p.colk = views, colk
        p.cand_n_data_rows = np.array([self.m_rows], dtype=np.int64)
        _lib.check(lib.hb2_batch_create(self._h, 1, _lib.ptr(p.cands), nv, _lib.ptr(views), len(colk), _lib.ptr(colk),
                                        len(p.pairs), _lib.ptr(p.pairs)))
        self.n = self.L3 * problem.ndisk
        self.nc = 1
        self.results = None
        self._amap_cache = {}

    def data_csr(self, c=0):
        """A_data, b, b_pid (SLR:1651-1654) downloaded from the GPU-built rows (duplicates summed by scipy)."""
        m, nnz = self.m_rows, self.nnz
        indptr = np.zeros(m + 1, dtype=np.int64)
        indices = np.zeros(max(nnz, 1), dtype=np.int32)
        data = np.zeros(max(nnz, 1), dtype=np.float32)
        b = np.zeros(max(m, 1), dtype=np.float32)
        pid = np.zeros(max(m, 1), dtype=np.int32)
        _lib.check(_lib.load().hb2_batch_explicit_export(self._h, _lib.ptr(indptr), _lib.ptr(indices), _lib.ptr(data),
                                                         _lib.ptr(b), _lib.ptr(pid)))
        A = csr_matrix((data[:nnz], indices[:nnz], indptr), shape=(m, self.n), dtype=np.float32)
        return A, b[:m], pid[:m]

    def data_b(self):
        """b_data of the explicit rows (SLR:1548) without downloading the matrix."""
        b = np.zeros(max(self.m_rows, 1), dtype=np.float32)
        _lib.check(_lib.load().hb2_batch_explicit_export(self._h, None, None, None, _lib.ptr(b), None))
        return b[:self.m_rows]

    def predict(self, x):
        """A_data @ x on the GPU (x in the reference's voxel order)."""
        return self.apply_forward(0, x)[:self.m_rows]

    def sym_csr(self, c=0):
        if not self.m_sym_explicit:
            return super().sym_csr(c)
        return trilinear_sym_csr(self._h, self.m_sym_explicit, self.n)

    def data_row_index(self, c=0):
        _, _, pid = self.data_csr(0)
        D2 = self.problem.D2
        return np.arange(self.m_rows, dtype=np.int64), (pid // D2).astype(np.int64), (pid % D2).astype(np.int64)


def trilinear_sym_csr(handle, m, n):
    """A_hsym, b_hsym (SLR:1289-1298) from the GPU-built trilinear symmetry rows (duplicates summed by scipy)."""
    if m == 0:
        return None, None
    cols = np.zeros(16 * m, dtype=np.int32)
    w = np.zeros(16 * m, dtype=np.float32)
    _lib.check(_lib.load().hb2_batch_explicit_sym_export(handle, _lib.ptr(cols), _lib.ptr(w)))
    A = csr_matrix((w, cols, np.arange(m + 1, dtype=np.int64) * 16), shape=(m, n), dtype=np.float32)
    A.sum_duplicates()
    return A, np.zeros(m, dtype=np.float32)


def build_trilinear_sym_rows(problem: Problem, nz, twist, rise_pixel, csym, min_sym_pairs):
    """build_A_helical_sym_matrix with interpolation "linear": rows built on the GPU, nothing else of a batch."""
    from . import planner

    lib = _lib.require_gpu()
    h = C.c_void_p()
    dummy = np.array([[1.0, 0.0]], dtype=np.float64)
    nvalid, tie = np.zeros(1, dtype=np.int32), np.zeros(1, dtype=np.int32)
    _lib.check(lib.hb2_batch_begin(C.byref(h), problem._h, int(nz), 1, 1, _lib.ptr(dummy), _lib.ptr(nvalid), _lib.ptr(tie),
                                   problem.stream))
    try:
        tab = planner.trilinear_pair_table(twist, rise_pixel, csym, int(nz))
        ms = C.c_int64()
        _lib.check(lib.hb2_batch_explicit_sym_rows(h, len(tab), _lib.ptr(tab), int(min_sym_pairs), C.byref(ms)))
        return trilinear_sym_csr(h, int(ms.value), int(nz) * problem.ndisk)
    finally:
        lib.hb2_batch_destroy(h)

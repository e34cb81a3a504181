"""Batched (twist x rise [x csym]) grid search -- the driver the reference runs
as a ThreadPoolExecutor over ``process_one_task`` (webApps/denovo3D/app.py:
2286-2523) -- with thousands of candidates resident on the GPU at once.

Geometry derivation follows ``pipeline.process_one_task`` (pipeline.py:253-349)
for the no-rescale case (target_apix2d <= apix2d_orig); the per-candidate
semantics are those of ``lsq_reconstruct`` (solver_linear_regression.py:31-547).
"""

from __future__ import annotations

import itertools
import logging
import time

from concurrent.futures import ThreadPoolExecutor

import numpy as np

from .engine import Batch, ExplicitBatch, Problem, ScoreMap, Stream, model_params
from .planner import MAX_EQUATIONS, CandidateSpec, positive_rule

logger = logging.getLogger(__name__)


def _version():
    from . import __version__

    return __version__


class BatchPipeline:
    """Double-buffered batch preparation.

    ``for i, batch in pipe.run(prob, L3, chunks)`` yields ready ``Batch`` objects in
    order while a worker thread plans and sets up the NEXT chunk (host planner,
    in-plane maps, right-hand side, symmetry rows) on the other of two non-blocking
    streams, so that it overlaps the solve of the current batch: the C calls
    release the GIL, the GPU work of the two batches runs on different streams.
    The caller closes each batch when it is done with it.
    """

    _STREAMS = {}  # device -> the two library streams, kept for the life of the process: their memory arenas stay warm

    def __init__(self, device=0, pipelined=True):
        self.device = int(device)
        self.pipelined = bool(pipelined)
        if self.device not in BatchPipeline._STREAMS:
            BatchPipeline._STREAMS[self.device] = [Stream(device), Stream(device)]
        self.streams = BatchPipeline._STREAMS[self.device]
        self._ex = ThreadPoolExecutor(max_workers=1) if pipelined else None

    def run(self, prob, L3, chunks):
        """Batches of one Problem: ``chunks`` is a list of spec lists."""
        for i, (_, batch) in enumerate(self.run_items((prob, L3, ch, None) for ch in chunks)):
            yield i, batch

    def run_items(self, items, factory=None):
        """``items`` yields ``(prob, L3, specs, tag)`` lazily -- e.g. pulled from a ``ChunkQueue`` shared by several
        ranks: the NEXT item is fetched (and its batch built) by the worker thread while the current batch is being
        solved by the caller.  Yields ``(tag, batch)`` in order.  ``factory(prob, L3, specs, stream)`` builds the batch
        (default: the nearest-neighbour ``Batch``)."""
        it = iter(items)
        if factory is None:
            factory = lambda prob, L3, specs, stream: Batch(prob, L3, specs, stream=stream)
        streams = self.streams
        count = [0]

        def make_next():
            try:
                prob, L3, specs, tag = next(it)
            except StopIteration:
                return None
            i = count[0]
            count[0] += 1
            return tag, factory(prob, L3, specs, streams[i % 2])

        if not self.pipelined:
            while True:
                nb = make_next()
                if nb is None:
                    return
                yield nb
        fut = self._ex.submit(make_next)
        while True:
            cur = fut.result()
            if cur is None:
                return
            fut = self._ex.submit(make_next)
            try:
                yield cur
            except GeneratorExit:
                try:
                    pend = fut.result()
                    if pend is not None:
                        pend[1].close()
                except Exception:
                    pass
                raise

    def close(self):
        if self._ex is not None:
            self._ex.shutdown(wait=True)
            self._ex = None


def derive_geometry(ny, nx, apix2d_orig, rise, rise_max, tube_diameter, tube_diameter_inner, tube_length,
                    reconstruct_length, target_apix2d, target_apix3d, sym_oversample, return_3d=False, tilt_max=0.0):
    """Integer geometry of one task, pipeline.py:253-349 (image already at target_apix2d)."""
    reconstruct_diameter = tube_diameter if 0 < tube_diameter < ny * apix2d_orig else ny * apix2d_orig
    reconstruct_diameter_inner = tube_diameter_inner if 0 < tube_diameter_inner < reconstruct_diameter else 0
    if reconstruct_length < rise:
        reconstruct_length = max(min(3 * rise_max, tube_length),
                                 round(np.tan(np.deg2rad(abs(tilt_max))) * tube_diameter * 3))
    if target_apix2d < apix2d_orig:
        target_apix2d = apix2d_orig
    if target_apix2d != apix2d_orig:
        raise NotImplementedError("helicon_b200: image down-scaling (target_apix2d > apix2d_orig, skimage rescale) "
                                  "is outside the CUDA hot path; pass an image already at the target pixel size")
    if target_apix3d < 0:
        vol = reconstruct_length * (reconstruct_diameter**2 - reconstruct_diameter_inner**2) / 4 * np.pi
        target_apix3d = max(target_apix2d, round(np.power(vol / (nx * ny), 1 / 3) + 0.5))
    elif target_apix3d == 0:
        target_apix3d = target_apix2d
    D3 = int(round(reconstruct_diameter / target_apix3d))
    D3 += D3 % 2
    D3i = int(round(tube_diameter_inner / target_apix3d))
    D2 = int(round(reconstruct_diameter / target_apix2d))
    D2 += D2 % 2
    reconstruct_length_2d = tube_length if 0 < tube_length < nx * target_apix2d else nx * target_apix2d
    L2 = int(reconstruct_length_2d / target_apix2d)
    L2 += L2 % 2
    if reconstruct_length > 0:
        L3 = max(int(np.ceil(rise / target_apix3d)), int(np.ceil(reconstruct_length / target_apix3d)))
        L3 += L3 % 2
    else:
        L3 = int(L2 * target_apix2d / target_apix3d + 0.5)
        L3 += L3 % 2
    if sym_oversample <= 0:
        n_voxels = L3 * (D3**2 - D3i**2)
        ratio = 2**20 / n_voxels
        if ratio < 10:
            sym_oversample = max(1, int(round(ratio)))
        elif ratio < 100:
            sym_oversample = max(1, int(round(ratio / 10)) * 10)
        else:
            sym_oversample = max(1, int(round(ratio / 100)) * 100)
        if return_3d:
            sym_oversample *= 2
    return dict(D2=D2, L2=L2, D3=D3, D3i=D3i, L3=L3, sym_oversample=sym_oversample, apix2d=target_apix2d,
                apix3d=target_apix3d, s=target_apix2d / target_apix3d)


def _periodic(v, lo=-180.0, hi=180.0):
    """lib/angular.py:84-108 ``set_to_periodic_range``."""
    import math

    if lo <= v <= hi:
        return v
    tmp = math.fmod(v - lo, hi - lo)
    return tmp + lo if tmp >= 0 else tmp + hi


class ChunkQueue:
    """Dealer of work chunks to ranks (SURVEY 8e: cost-sorted deal / dynamic chunk queue per GPU).

    With an initialised ``torch.distributed`` of world size > 1 the chunks are dealt DYNAMICALLY: one atomic counter in
    the process group's key-value store (``store.add``; rank 0's TCPStore, host side, a few hundred microseconds per
    pull) hands out chunk indices in cost-sorted order, so a rank that drew cheap candidates simply takes more of them
    and no rank waits for another inside a search -- there is NO data-path collective.  Without a process group the
    deal is static: chunk i of the cost-sorted list goes to rank ``i % world`` (``shard=(rank, world)``).
    Every rank must create its queues in the same order (the counter key is derived from a per-process sequence)."""

    _seq = 0

    def __init__(self, n_chunks, shard=(0, 1), dist=None):
        self.n = int(n_chunks)
        self.rank, self.world = int(shard[0]), int(shard[1])
        self.store = None
        self._next = self.rank
        if dist is not None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            from torch.distributed import distributed_c10d

            self.store = distributed_c10d._get_default_store()
            self.key = f"hb2_chunk_queue_{ChunkQueue._seq}"
            ChunkQueue._seq += 1

    def next(self):
        """Index of the next chunk for this rank, or None when the list is exhausted."""
        if self.store is not None:
            i = int(self.store.add(self.key, 1)) - 1
        else:
            i = self._next
            self._next += self.world
        return i if i < self.n else None

    def __iter__(self):
        while True:
            i = self.next()
            if i is None:
                return
            yield i


def prepare_image(image, thresh_fraction, reconstruct_diameter, apix):
    """pipeline.py:276-284: with ``thresh_fraction >= 0`` the background (median of the two image rows just outside the
    reconstruction diameter) is set to 0, values below ``thresh_fraction * max`` are cut and the maximum is scaled to 1.
    Returns a new float32 array (the reference mutates its argument)."""
    data = np.array(image, dtype=np.float32, copy=True)
    if thresh_fraction >= 0:
        ny = data.shape[0]
        nr = min(ny // 2 - 1, int(np.ceil(reconstruct_diameter / 2 / apix) + 1))
        data -= np.median(data[(ny // 2 - nr, ny // 2 + nr), :])
        thresh = data.max() * thresh_fraction
        data = np.clip(data, thresh, None) - thresh
        data /= np.max(data)
    return np.ascontiguousarray(data, dtype=np.float32)


class GridTask:
    __slots__ = ("ti", "twist", "rise", "csym", "geom", "spec")

    def __init__(self, ti, twist, rise, csym, geom, spec):
        self.ti, self.twist, self.rise, self.csym, self.geom, self.spec = ti, twist, rise, csym, geom, spec


def build_tasks(ny, nx, apix, twists, rises, csyms=(1,), reconstruct_length_rise=3, tube_diameter=None,
                tube_diameter_inner=0.0, tube_length=None, target_apix3d=0, sym_oversample=-1,
                positive_constraint=-1, ndisk_of=None):
    """Task list in the reference's order (twist-major, app.py:2338) with its skip rules (app.py:2389-2403)."""
    tube_diameter = ny * apix if tube_diameter is None else tube_diameter
    tube_length = nx * apix if tube_length is None else tube_length
    rises = list(rises)
    tasks = []
    ti = 0
    for csym in csyms:
        for twist, rise in itertools.product(twists, rises):
            twist = float(np.round(_periodic(float(twist)), 6))  # app.py:2360
            this = ti
            ti += 1
            if abs(twist) < 0.01 or abs(rise) < 0.01 or abs(rise) >= tube_length / 2:
                continue
            g = derive_geometry(ny, nx, apix, rise, max(rises), tube_diameter, tube_diameter_inner, tube_length,
                                reconstruct_length_rise * rise, apix, target_apix3d, sym_oversample)
            tasks.append(GridTask(this, twist, float(rise), int(csym), g, None))
    return tasks, ti


def _bytes_per_candidate(n, md, cap, model=False):
    """Device bytes of one candidate; ``model``: hb2_batch_solve_model adds xbar, w_new, rhs and the CG residual
    (float64 n-vectors) and the one-byte real-row mask."""
    extra = 32 * n + (md + cap) if model else 0
    return 8 * (md + cap) + 48 * n + 16 * cap + 8 * cap + 32 * (2 * cap + 17) + 16 * n + 12 * (n + 1) + extra


def check_algorithm(algorithm, interpolation="nn"):
    """model_params of ``algorithm``, refusing what the batched model path does not cover (before any GPU work)."""
    params = model_params(algorithm)
    if params is not None and interpolation != "nn":
        raise NotImplementedError("helicon_b200: a grid search with a sklearn model runs on nearest-neighbour batches "
                                  "only (interpolation='linear' with a model is not implemented)")
    return params


def make_chunks(tasks, ndisk_of, batch_candidates=None, mem_budget_bytes=48 << 30, pipelined=True, positive_constraint=-1,
                interpolation="nn", model=False):
    """Cut the (twist-major) task list into the chunks that are solved as one batch each, most expensive first.

    Tasks that share a Problem/Batch shape (D2, L2, D3, D3i, s, L3) are grouped; every group is cut into runs of
    consecutive tasks (whole twist rows: the candidates of a run share most view angles, so their in-plane maps are
    built once).  Chunks are sorted by an a-priori cost -- unknowns x candidates, i.e. larger L3 (larger rise) first --
    so that a static round-robin deal is balanced and a dynamic deal ends with the cheap chunks (LPT rule)."""
    groups = {}
    for t in tasks:
        g = t.geom
        groups.setdefault((g["D2"], g["L2"], g["D3"], g["D3i"], g["s"], g["L3"]), []).append(t)
    chunks = []
    for key, tl in groups.items():
        D2, L2, D3, D3i, s, L3 = key
        n3 = L3 * ndisk_of(key)
        for t in tl:
            target = min(MAX_EQUATIONS, int(max(D2 * L2, n3) * t.geom["sym_oversample"]))
            rise_px = t.rise / t.geom["apix3d"]
            t.spec = CandidateSpec(t.twist, rise_px, t.csym, target, target,
                                   positive_rule(positive_constraint, rise_px, t.twist, L3))
        md_est = int((L3 + L2) / max(min(x.spec.rise_pixel for x in tl), 1e-3) + 3) * L3 * D2
        cap_est = min(max(x.spec.min_sym_pairs for x in tl) + n3, 64 * n3)
        per_cand = _bytes_per_candidate(n3, md_est, cap_est, model) * (2 if pipelined else 1)  # two batches resident
        bs = batch_candidates or max(1, min(512, int(mem_budget_bytes // per_cand)))
        if interpolation != "nn":
            # trilinear rows: matrix-free batches where the factorisation applies (bilinear.py; ~0.3 GB per candidate:
            # 16-entry symmetry rows + their transpose), else one candidate at a time on explicit rows
            mf = s == 1.0 and D3 == D2 and L3 <= 16
            bs = max(1, min(batch_candidates or 50, int(mem_budget_bytes // (per_cand + 40 * 16 * cap_est)))) if mf else 1
        for i0 in range(0, len(tl), bs):
            ch = tl[i0:i0 + bs]
            chunks.append((key, ch, float(n3) * len(ch)))
    chunks.sort(key=lambda c: -c[2])  # stable: equal-cost chunks keep the grid order
    return chunks


def search_grid(image, apix, twists, rises, csyms=(1,), reconstruct_length_rise=3, tube_diameter=None,
                tube_diameter_inner=0.0, tube_length=None, target_apix3d=0, sym_oversample=-1,
                positive_constraint=-1, thresh_fraction=-1, top_k=10, device=0, stream=None, batch_candidates=None,
                mem_budget_bytes=48 << 30, shard=(0, 1), return_x_top=False, progress=None, pipelined=True,
                interpolation="nn", dist=None, checkpoint=None, checkpoint_seconds=30.0, algorithm=None,
                score_metric="cosine"):
    """Solve + score every candidate of the grid on one GPU (or this rank's share of it).

    ``interpolation="nn"`` runs batches of candidates through the matrix-free projector; ``"linear"`` (trilinear rows,
    SLR:1403-1510 / 910-1138) through the matrix-free bilinear-footprint x slice-blend operator (bilinear.py) when
    scale2d_to_3d = 1 and L3 <= 16, else one candidate at a time on explicit GPU-built rows (engine.ExplicitBatch).

    Several GPUs split the grid by CHUNKS (batches of consecutive candidates) without any data-path communication:
    ``shard=(rank, world)`` deals the cost-sorted chunk list round-robin; with ``dist`` (an initialised
    ``torch.distributed``, NCCL) the deal is dynamic through ``ChunkQueue`` (an atomic counter) and the per-rank score
    maps are all-gathered ONCE at the end, so every rank returns the whole grid and the global top-K.  The score map,
    iteration map and top-K selection are device-resident (``engine.ScoreMap``: one scatter kernel per solved batch,
    one top-K kernel per search).  ``thresh_fraction >= 0``
    applies the image preparation of ``process_one_task`` (pipeline.py:276-284) and clips the predictions at 0
    (SLR:502-503).  ``checkpoint=path`` makes the search resumable (checkpoint.ScoreTileStore): the tiles of solved
    batches are written to ``path`` (``path.rank<r>`` per rank) every ``checkpoint_seconds``; a later call with the same
    image, grid and parameters restores them into the device maps (``hb2_scoremap_restore``) and solves only the rest
    (``n_restored`` in the result; ``return_x_top`` volumes exist only for candidates solved in this call).
    ``algorithm`` (the app's solver choice, SLR:272-342): None or ``{"model": "lsq"}`` runs LSMR (+ the bounded branch);
    ``{"model": "elasticnet" | "lasso" | "ridge", "alpha": .., "l1_ratio": ..}`` the batched model solver
    (Batch.solve_model) with the reference's defaults; other models and ``interpolation="linear"`` with a model raise
    NotImplementedError before any GPU work.
    ``score_metric`` (SLR:484-525): "cosine" (default, the solve's own score) or "ssim" / "ms_ssim" /
    "mutual_information" / "composite", computed for every candidate on the device after its batch's solve
    (Batch.score_metric) with the semantics of ``lsq_reconstruct(..., score_metric=...)``; the score map, top-K,
    checkpoint tiles and ``return_x_top`` then rank by it.
    Returns dict(scores[(n_csym,) T, R] (NaN = not solved here / skipped task), itn, flags, top,
    n_candidates, seconds).
    """
    mparams = check_algorithm(algorithm, interpolation)
    check_score_metric(score_metric)
    ny, nx = np.asarray(image).shape
    tube_d = ny * apix if tube_diameter is None else tube_diameter
    image = prepare_image(image, thresh_fraction, tube_d if 0 < tube_d < ny * apix else ny * apix, apix)
    twists = np.atleast_1d(np.asarray(twists, dtype=np.float64))
    rises = np.atleast_1d(np.asarray(rises, dtype=np.float64))
    tasks, ntot = build_tasks(ny, nx, apix, twists, rises, csyms, reconstruct_length_rise, tube_diameter,
                              tube_diameter_inner, tube_length, target_apix3d, sym_oversample, positive_constraint)
    t0 = time.perf_counter()
    probs = {}
    store = None
    if checkpoint is not None:
        from .checkpoint import ScoreTileStore, agree_across_ranks, fingerprint

        rank, world = shard
        if dist is not None and dist.is_available() and dist.is_initialized():
            rank, world = dist.get_rank(), dist.get_world_size()
        fp = fingerprint(image, (np.asarray(csyms, dtype=np.float64), twists, rises), apix=float(apix),
                         reconstruct_length_rise=reconstruct_length_rise, tube_diameter=tube_diameter,
                         tube_diameter_inner=tube_diameter_inner, tube_length=tube_length, target_apix3d=target_apix3d,
                         sym_oversample=sym_oversample, positive_constraint=positive_constraint,
                         clip_pred=int(thresh_fraction >= 0), interpolation=str(interpolation), library=_version(),
                         **model_fingerprint(mparams), **metric_fingerprint(score_metric))
        store = ScoreTileStore(checkpoint, fp, ntot, rank=rank, world=world, flush_seconds=checkpoint_seconds)
        if world > 1 and dist is not None and dist.is_available() and dist.is_initialized():
            agree_across_ranks(store, dist, device)  # every rank must filter the SAME tasks
        tasks_all = len(tasks)
        tasks = [t for t in tasks if not store.is_done(t.ti)]
        logger.info("search_grid: %d of %d candidates restored from %s", tasks_all - len(tasks), tasks_all, checkpoint)

    def problem(key):
        if key not in probs:
            D2, L2, D3, D3i, s, L3 = key
            probs[key] = Problem(image, s, D2, L2, D3, D3i / 2, D3 // 2 - 1, device=device, stream=stream,
                                 interpolation="linear" if interpolation != "nn" else "nn")
        return probs[key]

    chunks = make_chunks(tasks, lambda key: problem(key).ndisk, batch_candidates, mem_budget_bytes, pipelined,
                         positive_constraint, interpolation, model=mparams is not None)
    queue = ChunkQueue(len(chunks), shard=shard, dist=dist)
    smap = ScoreMap(ntot, device=device)  # score / iteration / flag maps + top-K live on the device
    top_x = {}
    done = [0]
    if store is not None and store.n_restored:
        r = np.flatnonzero(store.restored)
        smap.restore(r, store.scores[r], store.itn[r], store.flags[r])

    def on_result(chunk, res, batch):
        done[0] += len(chunk)
        smap.scatter(batch, [x.ti for x in chunk], res["flags"])
        if store is not None:
            store.add([x.ti for x in chunk], res["score"], res["itn"], res["flags"])
        if return_x_top and top_k:  # keep the volumes of this batch's best candidates while the batch is alive
            for c in np.argsort(-res["score"], kind="stable")[:top_k]:
                top_x[chunk[c].ti] = (float(res[c]["score"]), batch.rec3d(int(c)))
            if len(top_x) > top_k:
                for ti in sorted(top_x, key=lambda t: (-top_x[t][0], t))[top_k:]:
                    del top_x[ti]
        if progress:
            progress(done[0], len(tasks))

    try:
        stats = solve_chunks(chunks, queue, problem, device=device, pipelined=pipelined, interpolation=interpolation,
                             clip_pred=int(thresh_fraction >= 0), on_result=on_result, algorithm=algorithm if mparams else None,
                             score_metric=score_metric)
        n_solved = stats["n_candidates"]
        if dist is not None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            # the ONLY collective of a search: every rank's maps all-gathered (NCCL), folded and ranked on the device
            import torch

            world = dist.get_world_size()
            with torch.cuda.device(device):
                mine = torch.as_tensor(smap, device=f"cuda:{device}")
                buf = torch.empty(world * mine.numel(), dtype=mine.dtype, device=mine.device)
                dist.all_gather_into_tensor(buf, mine)
                cur = torch.cuda.current_stream()
                smap.merge(buf.data_ptr(), world, stream=cur)
                cur.synchronize()
        scores, itn, flags = smap.read()
        if dist is not None and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            n_solved = int(np.isfinite(scores).sum()) - (store.n_restored if store is not None else 0)
        top = []
        if top_k:
            axes = (tuple(int(c) for c in csyms), twists, rises)
            from .distributed import entry_from_index

            tsc, tix = smap.topk(top_k)
            for sc_, ti in zip(tsc.tolist(), tix.tolist()):
                ent = entry_from_index(ti, sc_, axes)
                if ti in top_x:
                    ent["rec3d"] = top_x[ti][1]
                top.append(ent)
    finally:
        if store is not None:
            store.close()  # also after an interrupted search: what was solved so far is on disk
        smap.close()
        for pr in probs.values():
            pr.close()
    shape = (len(csyms), len(twists), len(rises))
    out = dict(scores=scores.reshape(shape), itn=itn.reshape(shape), flags=flags.reshape(shape), top=top,
               n_candidates=n_solved, n_solved_here=stats["n_candidates"], seconds=time.perf_counter() - t0,
               kernel_ms=stats["kernel_ms"], launches=stats["launches"] + 2 * stats["n_chunks"] + 2,
               axes=(tuple(int(c) for c in csyms), twists, rises), n_restored=store.n_restored if store is not None else 0)
    return out


TIMING_KEYS = ("lsmr_ms", "trf_ms", "score_ms", "fwd_data_ms", "fwd_sym_ms", "adj_ms", "update_ms", "scalar_ms", "norm_ms",
               "metric_ms", "launches", "fwd_data_launches", "adj_launches", "update_launches")


def model_fingerprint(mparams):
    """Checkpoint parameters of the solver model: none for lsq, so that the tiles of existing lsq searches resume."""
    if mparams is None:
        return {}
    model, alpha, l1_ratio = mparams
    return dict(model=model, alpha=float(alpha), l1_ratio=float(l1_ratio))


def check_score_metric(score_metric):
    """The score metrics lsq_reconstruct accepts; raises before any GPU work."""
    if score_metric not in ("cosine", "ssim", "ms_ssim", "mutual_information", "composite"):
        raise ValueError(f"unknown score_metric {score_metric!r}")


def metric_fingerprint(score_metric):
    """Checkpoint parameter of the score metric: none for cosine, so that the tiles of existing searches resume."""
    return {} if score_metric == "cosine" else dict(score_metric=str(score_metric))


def solve_chunks(chunks, queue, problem_of, device=0, pipelined=True, interpolation="nn", clip_pred=0, profile=0,
                 on_result=None, solve_options=None, algorithm=None, score_metric="cosine"):
    """Solve the chunks ``queue`` deals to this rank: ``chunks[i] = (problem key, [GridTask], cost)`` (make_chunks).

    The batch of chunk i+1 is planned and set up by a worker thread (second stream) while chunk i is being solved
    (BatchPipeline).  ``on_result(chunk_tasks, results, batch)`` is called per solved batch, before it is closed.
    Returns the summed library timings (``profile=1`` adds the per-kernel-class device times).  ``algorithm``: a
    sklearn-model dict solves every batch with Batch.solve_model instead of LSMR.  ``score_metric`` other than "cosine":
    every batch is re-scored with Batch.score_metric after its solve; its pixel tables are built with the batch on the
    worker thread."""
    pipe = BatchPipeline(device=device, pipelined=pipelined)
    stats = dict.fromkeys(TIMING_KEYS, 0.0)
    stats.update(n_candidates=0, n_chunks=0, itn_sum=0, chunk_ids=[])
    opts = dict(solve_options or {})
    batches = None
    try:
        factory = None
        if interpolation != "nn":
            from . import bilinear

            def factory(prob, L3, specs, stream):
                if bilinear.supported(prob, L3):  # matrix-free trilinear rows, many candidates per batch
                    return bilinear.BilinearBatch(prob, L3, specs, stream=stream)
                if len(specs) != 1:
                    raise AssertionError("explicit rows: one candidate per batch")
                return ExplicitBatch(prob, L3, specs[0], interpolation=interpolation, stream=stream)

        if score_metric != "cosine":
            build = factory or (lambda prob, L3, specs, stream: Batch(prob, L3, specs, stream=stream))

            def factory(prob, L3, specs, stream):
                batch = build(prob, L3, specs, stream)
                try:
                    batch.set_pixel_rows()
                except BaseException:
                    batch.close()
                    raise
                return batch

        batches = pipe.run_items(((problem_of(chunks[ci][0]), chunks[ci][0][5], [x.spec for x in chunks[ci][1]], ci)
                                  for ci in queue), factory)
        for ci, batch in batches:
            chunk = chunks[ci][1]
            try:
                if algorithm is not None:
                    res = batch.solve_model(algorithm, clip_pred=clip_pred, **opts)
                else:
                    res = batch.solve(clip_pred=clip_pred, profile=int(profile), **opts)
                if score_metric != "cosine":
                    res = batch.score_metric(score_metric, clip_pred=clip_pred)
                tm = batch.timing()
                for k in TIMING_KEYS:
                    stats[k] += tm.get(k, 0.0)
                stats["itn_sum"] += int(res["itn"].sum())
                if on_result is not None:
                    on_result(chunk, res, batch)
            finally:
                batch.close()
            stats["n_candidates"] += len(chunk)
            stats["n_chunks"] += 1
            stats["chunk_ids"].append(ci)
    finally:
        if batches is not None and hasattr(batches, "close"):
            batches.close()  # closes a batch the worker thread may still be building, BEFORE the problems go away
        pipe.close()
    stats["kernel_ms"] = stats["lsmr_ms"] + stats["trf_ms"] + stats["score_ms"] + stats["metric_ms"]
    stats["launches"] = int(stats["launches"])
    return stats


def search_images(images, apix, twists, rises, csyms=(1,), shard=(0, 1), dist=None, gather_device="cuda", **kw):
    """BASELINE config 4: an independent (twist x rise [x csym]) grid search per image (e.g. 2-D class averages).

    Images are dealt round-robin over ranks (``shard=(rank, world)``): every rank runs ``search_grid`` on its images
    with the whole grid, so there is no data-path communication; with ``dist`` (an initialised ``torch.distributed``)
    the per-image score maps are all-gathered at the end.  Returns ``dict(scores[n_img, (n_csym,) T, R], best=[(score,
    twist, rise, csym)] per image, n_candidates, seconds)``; entries of images solved by other ranks are NaN / None
    unless gathered.
    """
    rank, world = shard
    t0 = time.perf_counter()
    n_img = len(images)
    shape = (len(csyms), len(np.atleast_1d(twists)), len(np.atleast_1d(rises)))
    scores = np.full((n_img,) + shape, np.nan, dtype=np.float32)
    best = [None] * n_img
    ncand = 0
    for ii in range(rank, n_img, world):
        out = search_grid(images[ii], apix, twists, rises, csyms=csyms, **kw)
        scores[ii] = out["scores"]
        ncand += out["n_candidates"]
        if out["top"]:
            e = out["top"][0]
            best[ii] = (e["score"], e["twist"], e["rise"], e["csym"])
    if dist is not None and dist.is_initialized() and dist.get_world_size() > 1:
        import torch

        t = torch.from_numpy(scores.reshape(n_img, -1)).to(gather_device)
        parts = [torch.empty_like(t) for _ in range(dist.get_world_size())]
        dist.all_gather(parts, t)
        allsc = torch.stack(parts).cpu().numpy()  # [world, n_img, grid]
        own = np.arange(n_img) % dist.get_world_size()
        scores = allsc[own, np.arange(n_img)].reshape((n_img,) + shape)
        tw, ri = np.atleast_1d(twists), np.atleast_1d(rises)
        for ii in range(n_img):
            if best[ii] is None and np.any(np.isfinite(scores[ii])):
                c, a, b = np.unravel_index(np.nanargmax(scores[ii]), shape)
                best[ii] = (float(scores[ii][c, a, b]), float(tw[a]), float(ri[b]), int(csyms[c]))
        nt = torch.tensor([ncand], device=gather_device)
        dist.all_reduce(nt)
        ncand = int(nt.item())
    return dict(scores=scores, best=best, n_candidates=ncand, seconds=time.perf_counter() - t0)

#!/usr/bin/env python
"""denovo3D candidates/sec (solve + score) on N B200s vs the reference CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2|cfg1|cfg3]
                    [--dump-outputs DIR]

Workload (default, BASELINE.json configs[1]): one synthetic amyloid-like filament image, 256x256 px at 1.3 A/px (true
twist -1.2 deg, rise 4.75 A); dense 1000 twist x 50 rise grid; interpolation "nn", algorithm {"model": "lsq"}, cosine
score, and the reference's DEFAULT positive-constraint rule (positive_constraint=-1, SLR:352-355: every candidate of
this grid then also runs scipy's bounded TRF branch).  ``--positive 0`` times the unbounded LSMR path alone; the default
run reports it as the co-equal ``unbounded_path`` line.

A "step" = one chunk of the grid = one batch of consecutive candidates (default 4 twist rows x 50 rises = 200).  The
job's chunks are a FIXED pseudo-random sample of the grid's twist rows (seeded permutation), so that the work per step
is statistically the same whatever the number of GPUs; the N*K chunks of a run are dealt to the ranks dynamically
through an atomic counter (grid.ChunkQueue, no data-path collective), the last step of every rank in quarters (whole
twist rows) so that the job ends on small chunks; every rank keeps its scores in a device score map
and ONE NCCL all-gather + a device top-K kernel end the timed region (weak scaling: per-GPU work fixed).

JSON line keys follow the driver contract (task statement / DESIGN.md section 6).
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"  # NCCL prints its version banner on stdout; rank 0's stdout is ONE JSON line

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

APIX = 1.3
N_IMG = 256
TRUE_TWIST, TRUE_RISE = -1.2, 4.75
N_TWIST, N_RISE = 1000, 50
TWISTS = np.linspace(-3.0, -0.2, N_TWIST)
RISES = np.linspace(4.4, 5.1, N_RISE)

# BASELINE.json configs (SURVEY 8d).  cfg2 is the bench line; cfg1 / cfg3 are selectable for the other shapes.
CONFIGS = {
    "cfg1": dict(n=200, twists=np.linspace(-2.19, -0.21, 100), rises=np.linspace(4.5, 4.95, 10), csyms=(1,), batch=200,
                 image="filament",
                 workload="cfg1: synthetic amyloid-like filament 200x200 px @1.3 A/px (true twist -1.2 deg, rise 4.75 A), "
                          "100 twist x 10 rise grid"),
    "cfg2": dict(n=N_IMG, twists=TWISTS, rises=RISES, csyms=(1,), batch=200, image="filament",
                 workload="cfg2: synthetic amyloid-like filament 256x256 px @1.3 A/px (true twist -1.2 deg, rise 4.75 A), "
                          "1000 twist x 50 rise grid"),
    "cfg3": dict(n=512, twists=np.linspace(-60.0, 60.0, 2000), rises=np.linspace(4.75, 20.0, 100), csyms=(1, 2, 3, 4, 5, 6),
                 batch=24, image="tube",
                 workload="cfg3: synthetic tube-like helix 512x512 px @1.3 A/px (true twist 27.3 deg, rise 9.1 A, csym 3), "
                          "2000 twist x 100 rise x csym 1-6 grid"),
}


def synthetic_filament(n=N_IMG, apix=APIX, twist=TRUE_TWIST, rise=TRUE_RISE, seed=7, n_atoms=30, diameter=100.0,
                       ball_radius=3.0, csym=1, tube=False):
    """Helical assembly of Gaussian balls projected along y (same recipe as the
    reference's utils.simulate_helical_projection:31-189, restated; the
    reference itself is not available on the GPU box).  ``tube=True`` puts the atoms of the asymmetric unit on a ring
    (BASELINE config 3: a tube-like helix); ``csym`` adds the cyclic copies."""
    rng = np.random.default_rng(seed)
    # asymmetric unit: a planar-ish chain of atoms inside the tube cross-section
    t = np.cumsum(rng.normal(0, 1, (n_atoms, 2)), axis=0)
    t -= t.mean(axis=0)
    t *= (diameter / 2 * 0.8) / np.abs(t).max()
    if tube:
        ang = rng.uniform(0, 2 * np.pi / csym, n_atoms)
        rad = diameter / 2 * rng.uniform(0.85, 1.0, n_atoms)
        t = np.stack([rad * np.cos(ang), rad * np.sin(ang)], axis=1)
    au = np.stack([t[:, 0], t[:, 1], rng.normal(0, 0.3, n_atoms)], axis=1)  # x, y, z (A)
    length = n * apix
    hmax = int(np.ceil(length / 2 / rise)) + 2
    img = np.zeros((n, n), dtype=np.float64)
    yy = (np.arange(n) - n // 2) * apix
    xx = (np.arange(n) - n // 2) * apix
    sig2 = (ball_radius / 1.5) ** 2
    for h in range(-hmax, hmax + 1):
        for c in range(csym):
            a = np.deg2rad(twist * h + 360.0 * c / csym)
            ca, sa = np.cos(a), np.sin(a)
            x = ca * au[:, 0] - sa * au[:, 1]
            z = au[:, 2] + h * rise
            # image rows = x (across the filament), columns = z (along the axis); projection along y
            gy = np.exp(-(yy[:, None] - x[None, :]) ** 2 / (2 * sig2))
            gx = np.exp(-(xx[:, None] - z[None, :]) ** 2 / (2 * sig2))
            img += gy @ gx.T
    return np.ascontiguousarray(img, dtype=np.float32)


def config_image(cfg):
    if cfg["image"] == "tube":
        return synthetic_filament(n=cfg["n"], twist=27.3, rise=9.1, n_atoms=6, diameter=0.6 * cfg["n"] * APIX,
                                  ball_radius=6.0, csym=3, tube=True)
    return synthetic_filament(n=cfg["n"])


def grid_tasks():
    """The whole cfg2 task list (kept for profiles/*.py)."""
    from helicon_b200.grid import build_tasks

    tasks, ntot = build_tasks(N_IMG, N_IMG, APIX, TWISTS, RISES, csyms=(1,), reconstruct_length_rise=3,
                              target_apix3d=0, sym_oversample=-1)
    return tasks


def job_chunks(cfg, n_chunks, batch, positive, ndisk_of, seed=2026):
    """The first ``n_chunks`` chunks of the job: twist rows (all rises, all csyms of a twist) in a seeded pseudo-random
    order, cut into batches of <= ``batch`` candidates that share a batch shape (grid.make_chunks), in row order."""
    from helicon_b200.grid import build_tasks, make_chunks

    order = np.random.default_rng(seed).permutation(len(cfg["twists"]))
    per_row = len(cfg["rises"]) * len(cfg["csyms"])
    rows_per_block = max(1, batch // per_row) if per_row <= batch else 1
    chunks, pos, base = [], 0, 0
    while len(chunks) < n_chunks:
        rows = [order[(pos + i) % len(order)] for i in range(rows_per_block * 4)]
        pos += len(rows)
        tasks, ntot = build_tasks(cfg["n"], cfg["n"], APIX, np.sort(cfg["twists"][rows]), cfg["rises"], csyms=cfg["csyms"],
                                  reconstruct_length_rise=3, target_apix3d=0, sym_oversample=-1)
        for t in tasks:
            t.ti += base  # flat candidate index inside the job
        base += ntot
        new = make_chunks(tasks, ndisk_of, batch_candidates=batch, positive_constraint=positive)
        new.sort(key=lambda c: c[1][0].ti)  # grid order inside the block (make_chunks sorts by cost)
        chunks += new
    return chunks[:n_chunks], base


def split_tail(chunks, world, per_row, parts=4):
    """The LAST step of the timed region (one chunk per rank) is dealt in quarters (whole twist rows): the ranks pull
    chunks from the atomic counter as they finish, so what a rank can be late by at the end of the job is one small
    chunk instead of one whole step (cost-sorted / dynamic deal of SURVEY 8e: big chunks first, small ones last).
    The candidates -- and their total -- are the same at every N, N = 1 included."""
    if len(chunks) < world or parts <= 1:
        return chunks
    out = list(chunks[:-world])
    for key, tl, cost in chunks[-world:]:
        piece = max(per_row, len(tl) // parts) // per_row * per_row if per_row > 0 else 0
        if piece <= 0 or len(tl) < 2 * piece:
            out.append((key, tl, cost))
            continue
        for i0 in range(0, len(tl), piece):
            part = tl[i0:i0 + piece]
            out.append((key, part, cost * len(part) / len(tl)))
    return out


# ---------------------------------------------------------------------------
# clocks sampling during the timed region (B200_PROFILING.md)
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index):
        self.idx = device_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=float(max(mx)) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------
# CPU arm: the reference's own implementation of the path on the host cores -- the UNMODIFIED reference when
# oracle/_ref holds it (kind "reference"; shipped by oracle/build_ref.py), else the oracle port (kind "port")
# ---------------------------------------------------------------------------
def _cpu_full_candidate(job):
    """One FULL candidate on one core: system build, scipy lsq_linear exactly as the reference calls it (LSMR to its own
    stopping point, bounded TRF branch when the positive rule fires), reprojection + cosine score.  Returns a dict with
    the wall time and what the parity gate compares (score, LSMR iterations, TRF iterations, score of the LSMR stage)."""
    os.environ["OMP_NUM_THREADS"] = "1"  # the reference forces this at import (lib/transforms.py:14)
    import importlib
    import tempfile
    import warnings

    warnings.filterwarnings("ignore")
    img, g, twist, rise, csym, positive, warm = job
    LL = importlib.import_module("scipy.optimize._lsq.lsq_linear")
    spy = dict(lsmr=[], trf=[])
    real_lsmr, real_trf = LL.lsmr, LL.trf_linear
    if not hasattr(real_lsmr, "_hb2_spy"):
        def lsmr_spy(*a, **k):
            r = real_lsmr(*a, **k)
            spy["lsmr"].append((int(r[2]), r[0]))
            return r

        def trf_spy(*a, **k):
            r = real_trf(*a, **k)
            spy["trf"].append(int(r.nit))
            return r

        lsmr_spy._hb2_spy = True
        LL.lsmr, LL.trf_linear = lsmr_spy, trf_spy
    kw = dict(scale2d_to_3d=g["s"], twist_degree=twist, rise_pixel=rise / g["apix3d"], csym=csym,
              positive_constraint=positive, reconstruct_diameter_3d_inner_pixel=g["D3i"],
              reconstruct_diameter_2d_pixel=g["D2"], reconstruct_length_2d_pixel=g["L2"],
              reconstruct_diameter_3d_pixel=g["D3"], reconstruct_length_3d_pixel=g["L3"],
              sym_oversample=g["sym_oversample"], interpolation="nn")
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    kind = "port"
    S = None
    if os.path.isdir(os.path.join(ref_dir, "helicon")):
        try:
            tmp = tempfile.mkdtemp(prefix="hb2_ref_")
            os.environ["HELION_CACHE_DIR"] = tmp   # the reference memoises its builders on disk (lib/cache.py): fresh dir
            os.environ.setdefault("NUMBA_CACHE_DIR", os.path.join(tempfile.gettempdir(), "hb2_numba_cache"))
            if ref_dir not in sys.path:
                sys.path.insert(0, ref_dir)
            from helicon.webApps.denovo3D import solver_linear_regression as S  # noqa: N812

            kind = "reference"
        except Exception:
            S = None
    t0 = time.perf_counter()
    if S is not None:
        (rec, _, _), score = S.lsq_reconstruct(projection_image=img, algorithm=dict(model="lsq"), cpu=1, **kw)
    else:
        from oracle import denovo3d_oracle as O

        (rec, _, _), score = O.lsq_reconstruct(img, fast=True, **kw)
    dt = time.perf_counter() - t0
    LL.lsmr, LL.trf_linear = real_lsmr, real_trf
    out = dict(seconds=dt, score=float(score), kind=kind, itn=spy["lsmr"][0][0] if spy["lsmr"] else -1,
               trf_nit=spy["trf"][0] if spy["trf"] else 0, warm=bool(warm))
    if spy["lsmr"] and not warm:
        # score of the unconstrained LSMR stage (the first thing lsq_linear computes): rebuild the prediction with the
        # oracle's data rows (pinned bit-exact to the reference's builder)
        from oracle import denovo3d_oracle as O

        n3 = int(np.count_nonzero(O.cylindrical_mask(g["L3"], g["D3"], g["D3"], g["D3i"] / 2, g["D3"] // 2 - 1)))
        target = min(O.MAX_EQUATIONS, int(max(g["D2"] * g["L2"], n3) * g["sym_oversample"]))
        A_d, b_d, _ = O.build_A_data_matrix_fast(img, g["s"], twist, rise / g["apix3d"], csym, g["D2"], g["L2"], g["D3"],
                                                 g["D3i"], g["L3"], target)
        out["score_lsmr_stage"] = float(O.cosine_similarity(A_d.dot(spy["lsmr"][0][1].astype(np.float32)), b_d))
    return out


def _small_job(positive):
    from helicon_b200.grid import derive_geometry

    small = synthetic_filament(n=64, apix=APIX * 4)
    g = derive_geometry(64, 64, APIX * 4, 4.75, 4.75, 64 * APIX * 4, 0.0, 64 * APIX * 4, 3 * 4.75, APIX * 4, 0, -1)
    return (small, g, -1.3, 4.75, 1, positive, True)


def reference_arm(args, cfg, img, rank):
    """--impl reference: the reference's CPU implementation of the path with all host cores: one FULL candidate per
    core in parallel processes (real iteration counts, nothing extrapolated); throughput = sum over workers of
    1 / (seconds per candidate)."""
    from concurrent.futures import ProcessPoolExecutor

    if rank != 0:
        return 0
    cores = len(os.sched_getaffinity(0))
    workers = max(1, min(cores, args.ref_workers or cores))
    chunks, _ = job_chunks(cfg, 1 + args.warmup, args.batch or cfg["batch"], args.positive, lambda key: _ndisk(key))
    cands = [t for ch in chunks[args.warmup:] for t in ch[1]]
    stride = max(1, len(cands) // workers)
    picks = [cands[(i * stride) % len(cands)] for i in range(workers)]
    jobs = [(img, t.geom, t.twist, t.rise, t.csym, args.positive, False) for t in picks]
    with ProcessPoolExecutor(max_workers=workers) as ex:
        for _ in range(max(1, min(args.warmup, 2))):  # warm-up: imports, numba JIT, page cache (a small problem per worker)
            list(ex.map(_cpu_full_candidate, [_small_job(args.positive)] * workers))
        t0 = time.perf_counter()
        outs = list(ex.map(_cpu_full_candidate, jobs))
        wall = time.perf_counter() - t0
    value = float(sum(1.0 / o["seconds"] for o in outs))
    kind = outs[0]["kind"]
    secs = [o["seconds"] for o in outs]
    line = dict(
        impl="reference", metric="denovo3D candidates/sec (solve+score)", value=value, unit="candidates/s",
        n_gpus=args.gpus, steps=args.steps, warmup=args.warmup, ms_per_step=wall * 1e3, higher_is_better=True,
        scaling="weak", vs_baseline=None, dtype="f32 (u,v,h) / f64 (x,hbar; bounded branch), as scipy executes it",
        data="synthetic",
        config=dict(workload=cfg["workload"] + ", nn interpolation, model=lsq, cosine score", positive_constraint=args.positive,
                    steps_run=1, mean_lsmr_iterations=float(np.mean([o["itn"] for o in outs])),
                    mean_trf_iterations=float(np.mean([o["trf_nit"] for o in outs]))),
        cpu_baseline=dict(value=value, unit="candidates/s", cores=workers, kind=kind,
                          sample=f"{workers} grid candidates solved COMPLETELY, one per core in parallel processes "
                                 f"({'the unmodified reference lsq_reconstruct from oracle/_ref' if kind == 'reference' else 'the oracle port (oracle/_ref absent)'}"
                                 f": system build + scipy lsq_linear to its own stopping point + score); "
                                 f"{min(secs):.0f}-{max(secs):.0f} s per candidate, wall {wall:.0f} s; value = sum of 1/seconds. "
                                 f"A step of the GPU arm ({args.batch or cfg['batch']} candidates) would take "
                                 f"{(args.batch or cfg['batch']) / value / 3600:.1f} h here, so the K steps are bounded to this one round."),
        e2e=dict(value=value, unit="candidates/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
    )
    print(json.dumps(line))
    return 0


DUMP_LIMIT_BYTES = 64 << 20
NPY_HEADER_BYTES = 256  # np.save writes 128 B of header before a 1-D array; the limit counts whole files


def dump_outputs(out_dir, per_candidate, top, limit=DUMP_LIMIT_BYTES, seed=2026):
    """Write the results of the timed region as ``out_dir/<name>.npy`` so that two builds can be compared output for
    output.  ``per_candidate`` maps names to arrays of equal length (one entry per slot of the score map);
    ``candidate_index.npy`` gives the flat job index of each entry.  When these would exceed ``limit`` bytes, a fixed
    seeded sample of the entries is written instead (``limit`` counts whole files, headers included).  ``top`` maps names
    to the (short) top-K arrays."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v) for k, v in per_candidate.items()}
    top = {k: np.asarray(v) for k, v in top.items()}
    n = len(arrays["candidate_index"])
    row_bytes = sum(a.dtype.itemsize for a in arrays.values())
    room = limit - sum(a.nbytes for a in top.values()) - NPY_HEADER_BYTES * (len(arrays) + len(top))
    if n * row_bytes > room:
        keep = np.sort(np.random.default_rng(seed).choice(n, room // row_bytes, replace=False))
        arrays = {k: a[keep] for k, a in arrays.items()}
    for name, a in {**arrays, **top}.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _ndisk(key):
    D2, L2, D3, D3i, s, L3 = key
    c = np.arange(D3) - D3 // 2
    r2 = np.add.outer(c * c, c * c)
    return int(np.count_nonzero((r2 < (D3 // 2 - 1) ** 2) & (r2 >= (D3i / 2) ** 2)))


# ---------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="candidates per step (default: the config's, 200 for cfg2)")
    ap.add_argument("--positive", type=int, default=-1,
                    help="positive_constraint passed to the solver (-1 = the reference's default rule; 0 = unbounded LSMR path)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU baseline + parity gate (full oracle solve)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the unbounded-path and trilinear secondary measurements")
    ap.add_argument("--no-pipeline", action="store_true", help="prepare and solve batches strictly one after the other")
    ap.add_argument("--tail-split", type=int, default=4, help="pieces the last step of every rank is dealt in (1 = whole steps)")
    ap.add_argument("--e2e-calls", type=int, default=3, help="timed search_grid() calls of the e2e measurement")
    ap.add_argument("--e2e-batches", type=int, default=2, help="batches per rank and search_grid() call of the e2e measurement")
    ap.add_argument("--ref-workers", type=int, default=0, help="--impl reference: worker processes (default: all cores)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the score map and top-K the timed steps computed as DIR/<name>.npy (float32/float64, "
                         "<= 64 MB; a fixed seeded sample of a larger map)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg = CONFIGS[args.config]
    batch_size = args.batch or cfg["batch"]
    img = config_image(cfg)

    if args.impl == "reference":
        return reference_arm(args, cfg, img, rank)

    import torch

    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from helicon_b200.engine import Problem, ScoreMap
    from helicon_b200.grid import ChunkQueue, search_grid, solve_chunks

    stream = torch.cuda.current_stream()
    probs = {}

    def problem(key):
        if key not in probs:
            D2, L2, D3, D3i, s, L3 = key
            probs[key] = Problem(img, s, D2, L2, D3, D3i / 2, D3 // 2 - 1, device=local_rank, stream=stream)
        return probs[key]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    W, K = args.warmup, args.steps
    chunks, n_job = job_chunks(cfg, (W + K) * world, batch_size, args.positive, lambda key: problem(key).ndisk)
    warm_chunks, timed_chunks = chunks[:W * world], chunks[W * world:]
    n_timed_steps = len(timed_chunks)
    timed_chunks = split_tail(timed_chunks, world, len(cfg["rises"]) * len(cfg["csyms"]), args.tail_split)

    # ---- CPU baseline + parity gate: ONE full candidate of the timed block through the reference's CPU path, started
    # now in a background process so that its ~2-3 minutes overlap the GPU measurements (rank 0, N = 1 only) --------
    cpu_future, cpu_pool, gate = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from concurrent.futures import ProcessPoolExecutor

        gate = timed_chunks[0][1][len(timed_chunks[0][1]) // 3]
        cpu_pool = ProcessPoolExecutor(max_workers=1)
        cpu_pool.submit(_cpu_full_candidate, _small_job(args.positive)).result()  # imports / JIT warm-up, untimed
        cpu_future = cpu_pool.submit(_cpu_full_candidate, (img, gate.geom, gate.twist, gate.rise, gate.csym, args.positive, False))

    def run_block(block, positive_override=None, profile=True):
        """Deal ``block`` to the ranks, solve, keep the scores in a device map; one all-gather + top-K at the end."""
        queue = ChunkQueue(len(block), shard=(rank, world), dist=dist)
        lo = min(t.ti for ch in block for t in ch[1])
        hi = max(t.ti for ch in block for t in ch[1]) + 1
        smap = ScoreMap(hi - lo, device=local_rank)
        md = []

        def on_result(chunk, res, batch):
            smap.scatter(batch, [x.ti - lo for x in chunk], res["flags"])
            md.append((float(np.mean([batch.rows_padded(c)[0] for c in range(0, batch.nc, max(1, batch.nc // 8))])),
                       batch.n, res["itn"].astype(np.float64), res["n_sym_rows"].astype(np.float64), res["trf_nit"].astype(np.float64),
                       int(np.count_nonzero(batch.plan.views["dup_of"] < 0)) / max(1, batch.nc), batch.problem.ndisk, batch.L3))

        t_s0 = time.perf_counter()
        stats = solve_chunks(block, queue, problem, device=local_rank, pipelined=not args.no_pipeline, profile=int(profile),
                             on_result=on_result)
        stats["solve_wall_ms"] = 1e3 * (time.perf_counter() - t_s0)  # this rank's own work, before it waits in the all-gather
        if dist is not None:
            mine = torch.as_tensor(smap, device=f"cuda:{local_rank}")
            buf = torch.empty(world * mine.numel(), dtype=mine.dtype, device=mine.device)
            dist.all_gather_into_tensor(buf, mine)
            smap.merge(buf.data_ptr(), world, stream=stream)
        top_sc, top_ix = smap.topk(10, stream=stream)  # device kernel; synchronises the stream
        stats["launches"] += 2 * stats["n_chunks"] + 2 + (1 if dist is not None else 0)
        return stats, smap, lo, md, (top_sc, top_ix + lo)

    # ---- kernel-path timing: image resident, candidates -> scores -------------
    if warm_chunks:
        st_w, sm_w, _, _, _ = run_block(warm_chunks, profile=False)
        sm_w.close()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    stats, smap, lo, md, top = run_block(timed_chunks)
    torch.cuda.synchronize()  # the batches run on the library's own streams
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    t_ms = e0.elapsed_time(e1)
    red = torch.tensor([t_ms, float(stats["n_candidates"]), float(stats["itn_sum"]), float(stats["launches"])], device="cuda",
                       dtype=torch.float64)
    if dist is not None:
        mx = red.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(red, op=dist.ReduceOp.SUM)
        t_ms = float(mx[0].item())
    total_cands, itn_total, launches_total = int(red[1].item()), float(red[2].item()), int(red[3].item())
    value = total_cands / (t_ms / 1e3)
    # per-rank decomposition of the timed region (where a scaling loss comes from: uneven chunk deal, slower GPUs, host)
    mine_pr = torch.tensor([stats["solve_wall_ms"], stats["lsmr_ms"] + stats["trf_ms"] + stats["score_ms"],
                            float(stats["n_chunks"]), float(stats["n_candidates"]), float(stats["itn_sum"]),
                            float(clocks.get("sm_mhz") or 0.0), float("sw_power_cap" in clocks.get("reasons", []))],
                           device="cuda", dtype=torch.float64)
    if dist is not None:
        all_pr = torch.empty(world * mine_pr.numel(), device="cuda", dtype=torch.float64)
        dist.all_gather_into_tensor(all_pr, mine_pr)
    else:
        all_pr = mine_pr
    per_rank = [dict(solve_wall_ms=round(r[0], 1), kernel_ms=round(r[1], 1), chunks=int(r[2]), candidates=int(r[3]),
                     lsmr_iterations=int(r[4]), sm_mhz=r[5], sw_power_cap=bool(r[6])) for r in all_pr.reshape(-1, 7).tolist()]
    sc_all, itn_all, fl_all = smap.read()
    smap.close()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs,
                     dict(candidate_index=np.arange(lo, lo + len(sc_all), dtype=np.float64), scores=sc_all,
                          itn=itn_all.astype(np.float64), flags=fl_all.astype(np.float64)),
                     dict(top_scores=top[0].astype(np.float32), top_index=top[1].astype(np.float64)))
    per_rank_cands = stats["n_candidates"]

    # ---- algorithmic bytes of this rank's launches (SURVEY 8d) -----------------------------------------------------
    fwd_bytes = iter_bytes = gather_bytes = 0.0
    trf_total = 0.0
    for md_mean, n3, itn_c, msym_c, trf_c, views_nd, ndisk, L3 in md:
        fwd_bytes += float(itn_c.sum()) * (4.0 * n3 + 8.0 * md_mean)  # read v (4n) + read/write u (8 m_data)
        iter_bytes += float(np.sum(itn_c * (56.0 * n3 + 12.0 * (md_mean + msym_c))))  # B_iter = 56 n + 12 m
        # on chip: every sample of every non-duplicate view moves its L3P slices (4 B each) from L1/L2 to registers
        gather_bytes += float(itn_c.sum()) * views_nd * ndisk * ((L3 + 3) // 4 * 4) * 4.0
        trf_total += float(trf_c.sum())

    # ---- end-to-end through the public API: host image in, host scores out ----
    e2e_vals, e2e_best = [], None
    per_row = len(cfg["rises"]) * len(cfg["csyms"])
    rows_per_call = max(1, batch_size // per_row) * args.e2e_batches * world
    e2e_rises = cfg["rises"]
    if per_row > batch_size:  # a twist row is larger than a batch (cfg3: 100 rises x 6 csyms): one row, every n-th rise
        rows_per_call = 1
        n_r = max(1, (batch_size * args.e2e_batches * world) // len(cfg["csyms"]))
        e2e_rises = cfg["rises"][np.unique(np.linspace(0, len(cfg["rises"]) - 1, min(n_r, len(cfg["rises"]))).astype(int))]
    order = np.random.default_rng(77).permutation(len(cfg["twists"]))
    launches_e2e = 0
    for s in range(args.e2e_calls + 1):  # the first call is the warm-up
        rows = np.sort(order[(s * rows_per_call + np.arange(rows_per_call)) % len(order)])
        barrier()
        t0 = time.perf_counter()
        out = search_grid(np.array(img, copy=True), APIX, cfg["twists"][rows], e2e_rises, csyms=cfg["csyms"],
                          positive_constraint=args.positive, device=local_rank, stream=stream, batch_candidates=batch_size,
                          pipelined=not args.no_pipeline, shard=(rank, world), dist=dist)
        best = float(np.nanmax(out["scores"]))  # host read of the call's result (every rank holds the gathered map)
        barrier()
        tt = torch.tensor([time.perf_counter() - t0], device="cuda", dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if s > 0:
            e2e_vals.append(out["n_candidates"] / float(tt.item()))
            e2e_best, launches_e2e = best, out["launches"]
    e2e_val = float(np.mean(e2e_vals))
    d2h = int(out["scores"].size * 12)

    # ---- co-equal line: the unbounded LSMR path alone (positive_constraint=0) -------------------------------------
    unb = None
    if args.positive != 0 and not args.no_secondary:
        blk, _ = job_chunks(cfg, (1 + min(K, 4)) * world, batch_size, 0, lambda key: problem(key).ndisk, seed=4052)
        st_w, sm_w, _, _, _ = run_block(blk[:world], profile=False)
        sm_w.close()
        barrier()
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record(stream)
        st_u, sm_u, _, _, _ = run_block(blk[world:], profile=False)
        torch.cuda.synchronize()
        u1.record(stream)
        barrier()
        ru = torch.tensor([u0.elapsed_time(u1), float(st_u["n_candidates"]), float(st_u["itn_sum"])], device="cuda", dtype=torch.float64)
        if dist is not None:
            mxu = ru.clone()
            dist.all_reduce(mxu, op=dist.ReduceOp.MAX)
            dist.all_reduce(ru, op=dist.ReduceOp.SUM)
            ru[0] = mxu[0]
        sm_u.close()
        unb = dict(value=float(ru[1].item() / (ru[0].item() / 1e3)), unit="candidates/s", steps=min(K, 4),
                   mean_lsmr_iterations=float(ru[2].item() / max(1.0, ru[1].item())),
                   note="the same timed region with positive_constraint=0 (LSMR only, no bounded branch)")

    # ---- secondary: trilinear interpolation (the app's default mode) through the same call ------------------------
    trilinear = None
    if rank == 0 and not args.no_secondary and args.config == "cfg2":
        # matrix-free trilinear rows (helicon_b200/bilinear.py): batches of 25 candidates; one small warm-up call, then a timed one
        search_grid(np.array(img, copy=True), APIX, TWISTS[[400]], RISES[[10, 30]], positive_constraint=0,
                    device=local_rank, stream=stream, interpolation="linear")
        t0 = time.perf_counter()
        outl = search_grid(np.array(img, copy=True), APIX, TWISTS[[398, 402]], RISES, positive_constraint=0,
                           device=local_rank, stream=stream, interpolation="linear", batch_candidates=50)
        dtl = time.perf_counter() - t0
        trilinear = dict(value=outl["n_candidates"] / dtl, unit="candidates/s", candidates=int(outl["n_candidates"]),
                         n_gpus=1, mean_lsmr_iterations=float(np.nanmean(np.where(np.isfinite(outl["scores"]), outl["itn"], np.nan))),
                         best_score=float(np.nanmax(outl["scores"])), kernel_ms=float(outl["kernel_ms"]),
                         note="search_grid(interpolation='linear', positive_constraint=0) on one GPU: 2 twists x 50 rises in "
                              "batches of 50 candidates through the matrix-free trilinear operator (bilinear footprint maps x "
                              "slice blends, csrc/hb2_bilinear.cuh), host image -> host score map, one warmed call")

    # ---- parity gate against the CPU run of the same candidate ----------------------------------------------------
    parity, cpu_line = None, None
    if cpu_future is not None:
        from helicon_b200 import solver_linear_regression as S

        g = gate.geom
        kw = dict(reconstruct_diameter_3d_inner_pixel=g["D3i"], reconstruct_diameter_2d_pixel=g["D2"],
                  reconstruct_length_2d_pixel=g["L2"], reconstruct_diameter_3d_pixel=g["D3"],
                  reconstruct_length_3d_pixel=g["L3"], sym_oversample=g["sym_oversample"], interpolation="nn",
                  device=local_rank, return_info=True)
        (_, _, _), sc_unb, info_u = S.lsq_reconstruct(img, g["s"], gate.twist, gate.rise / g["apix3d"], gate.csym,
                                                      positive_constraint=0, **kw)
        cpu = cpu_future.result()
        cpu_pool.shutdown()
        gi = gate.ti - lo
        parity = dict(candidate=dict(twist=gate.twist, rise=gate.rise, csym=gate.csym),
                      dscore=abs(float(sc_all[gi]) - cpu["score"]), ditn=int(itn_all[gi]) - cpu["itn"],
                      gpu_score=float(sc_all[gi]), cpu_score=cpu["score"], gpu_itn=int(itn_all[gi]), cpu_itn=cpu["itn"],
                      cpu_trf_nit=cpu["trf_nit"], positive_constraint=args.positive,
                      dscore_lsmr_stage=abs(float(sc_unb) - cpu.get("score_lsmr_stage", float("nan"))),
                      gpu_score_lsmr_stage=float(sc_unb), cpu_score_lsmr_stage=cpu.get("score_lsmr_stage"),
                      tolerance="gate: LSMR stage |dscore| <= 1e-5 and |ditn| <= 2, and the final score within 1e-5 when the "
                                "candidate stayed unbounded.  When scipy's bounded TRF branch ran, the final score is "
                                "REPORTED (bounded_dscore_within_1e-4) but only sanity-gated (5e-2): the reference's own "
                                "result moves by 1e-3...2e-2 on some candidates when its equations are merely "
                                "re-ordered (tests/golden/bounded_band_cfg2.npz, DESIGN section 5), while the CUDA TRF "
                                "equals scipy's to 1e-7 from the same LSMR start (profiles/r2_summary.md)",
                      cpu_kind=cpu["kind"])
        bounded = bool(int(fl_all[gi]) & 4)
        parity["bounded"] = bounded
        parity["bounded_dscore_within_1e-4"] = bool(parity["dscore"] <= 1e-4) if bounded else None
        parity["ok"] = bool(parity["dscore_lsmr_stage"] <= 1e-5 and abs(parity["ditn"]) <= 2 and
                            parity["dscore"] <= (5e-2 if bounded else 1e-5))
        cpu_line = dict(value=1.0 / cpu["seconds"], unit="candidates/s", cores=1, kind=cpu["kind"],
                        sample=f"1 grid candidate (twist={gate.twist}, rise={gate.rise:.4f}) solved COMPLETELY by "
                               f"{'the unmodified reference (oracle/_ref)' if cpu['kind'] == 'reference' else 'the oracle port'} "
                               f"on one core: build + scipy lsq_linear ({cpu['itn']} LSMR iterations, {cpu['trf_nit']} TRF "
                               f"iterations) + score = {cpu['seconds']:.1f} s, concurrently with the GPU measurements")

    for pr in probs.values():
        pr.close()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    fwd_ms, fwd_launches = stats["fwd_data_ms"], max(1, int(stats["fwd_data_launches"]))
    achieved = fwd_bytes / (fwd_ms / 1e3) / 1e9 if fwd_ms > 0 else 0.0
    itn_rank = float(stats["itn_sum"])
    traffic, traffic_note = None, "no capture"
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
        per_cand = sum(tj["dram_bytes_per_launch"][k] for k in ("k_fwd_band", "k_fwd_band_reduce")) / tj["candidates_per_launch"]
        traffic = per_cand * itn_rank / fwd_launches
        traffic_note = ("dram__bytes_read.sum + dram__bytes_write.sum of the kernel from " + tj["source"] +
                        f": {per_cand / 1e6:.2f} MB per candidate-pass x {itn_rank / fwd_launches:.1f} active candidates per "
                        "launch in this run")
    except Exception:
        pass
    sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
    lsu_peak = 148 * 128.0 * sm_hz  # 128 B/clk/SM through the L1 / shared-memory data pipe (B300_MICROARCH.md)
    pass_us = fwd_ms * 1e3 / max(1.0, itn_rank)
    floor_us = gather_bytes / max(1.0, itn_rank) / lsu_peak * 1e6
    line = dict(
        metric="denovo3D candidates/sec (solve+score)", value=value, unit="candidates/s", n_gpus=world,
        steps=K, warmup=W, ms_per_step=t_ms / K, higher_is_better=True, scaling="weak",
        vs_baseline=None, dtype="f32 (u,v,h) / f64 (x,hbar; bounded branch), as scipy executes it", data="synthetic",
        config=dict(workload=cfg["workload"] + ", nn interpolation, model=lsq, cosine score",
                    step=f"one chunk of {batch_size} grid candidates (whole twist rows, seeded pseudo-random row order); "
                         f"{K} steps per GPU dealt by an atomic-counter chunk queue, the last step of every GPU in "
                         f"{args.tail_split} pieces ({n_timed_steps} chunks of the job -> {len(timed_chunks)} dealt pieces, same candidates at "
                         f"every N)", pipelined=not args.no_pipeline,
                    positive_constraint=args.positive,
                    bounded_fraction=float(np.mean((fl_all[np.isfinite(sc_all)] & 4) != 0)) if np.isfinite(sc_all).any() else 0.0,
                    cache="inputs of every step are new candidates; per-step working set >> L2 (126 MB)",
                    mean_lsmr_iterations=itn_total / max(1, total_cands),
                    mean_trf_iterations=trf_total / max(1, per_rank_cands),
                    candidate_iterations_per_s=itn_total / (t_ms / 1e3),
                    norm_mode="LSMR norms accumulated like numpy/OpenBLAS sdot (reference-faithful, DESIGN section 5)"),
        clocks=clocks, gpu_launches=int(launches_total),
        e2e=dict(value=e2e_val, unit="candidates/s", h2d_bytes_per_step=int(img.nbytes), d2h_bytes_per_step=d2h,
                 candidates_per_call=int(out["n_candidates"]), calls=len(e2e_vals), per_call=e2e_vals, best_score=e2e_best,
                 launches_per_call=int(launches_e2e),
                 note="search_grid(): host image -> Problem upload, host planning, solve, device score map + top-K, ONE "
                      "all-gather at N > 1, maps copied back; bytes are per search_grid() call"),
        roofline=dict(bound="hbm", kernel="k_fwd_band + k_fwd_band_reduce (forward projector u <- A v - alpha u: voxel bands "
                                         "staged in shared memory by TMA, partial ray sums, streaming row epilogue)",
                      achieved=achieved,
                      peak=peak, unit="GB/s", frac=achieved / peak if peak else None, traffic=traffic,
                      traffic_source=traffic_note,
                      algorithmic_bytes_per_launch=fwd_bytes / fwd_launches,
                      on_chip="the kernel is bound on chip, not by HBM (see roofline_onchip and profiles/r2_summary.md): the "
                              "time goes into moving the gathered slices through the shared-memory data pipe (82 % busy); "
                              "DRAM traffic above the algorithmic bytes = the partial ray sums of the band decomposition "
                              "(written once, read once)",
                      peak_source=peak_src, avg_launch_ms=fwd_ms / fwd_launches,
                      note="achieved = algorithmic bytes (4n + 8 m_data per active candidate-iteration) / summed "
                           "CUDA-event time of the two kernels' launches inside the timed region (rank 0)"),
        roofline_onchip=dict(kernel="k_fwd_band + k_fwd_band_reduce", bytes_gathered_per_pass=gather_bytes / max(1.0, itn_rank),
                             lsu_wavefronts_per_pass=gather_bytes / max(1.0, itn_rank) / 128.0,
                             floor_us=floor_us, achieved_us=pass_us, frac=floor_us / pass_us if pass_us > 0 else None,
                             note="floor = (non-duplicate views x in-disk samples x L3P slices x 4 B) / (148 SMs x 128 B/clk "
                                  "x SM clock): every gathered slice value crosses the shared-memory data pipe once; achieved "
                                  "= device time of the two kernels per active candidate-pass (ncu, profiles/r2_summary.md: "
                                  "2.8 M wavefronts per pass = 2.3x the floor -- ragged ray segments, pure-column steps, map "
                                  "shuffles)"),
        roofline_iteration=dict(
            bound="hbm", achieved=iter_bytes / (stats["lsmr_ms"] / 1e3) / 1e9 if stats["lsmr_ms"] > 0 else 0.0, peak=peak,
            unit="GB/s", frac=(iter_bytes / (stats["lsmr_ms"] / 1e3) / 1e9 / peak) if stats["lsmr_ms"] > 0 and peak else None,
            note="all kernels of the LSMR phase together: algorithmic bytes B_iter = 56 n + 12 m per active "
                 "candidate-iteration (SURVEY 8d) / device time of the LSMR phase"),
        kernel_share=dict(lsmr_phase_ms=stats["lsmr_ms"], trf_phase_ms=stats["trf_ms"], score_ms=stats["score_ms"],
                          fwd_data_ms=fwd_ms, fwd_sym_ms=stats["fwd_sym_ms"], adjoint_ms=stats["adj_ms"],
                          update_ms=stats["update_ms"], blas_norm_chain_ms=stats["norm_ms"], scalar_ms=stats["scalar_ms"],
                          note="rank 0, device time by kernel class inside the timed region (LSMR phase classes; the bounded "
                               "branch's float64 kernels are in trf_phase_ms)"),
        top=dict(best_score=float(top[0][0]) if len(top[0]) else None, best_index=int(top[1][0]) if len(top[1]) else None,
                 note="selected by the device top-K kernel over the all-gathered score map"),
    )
    line["per_rank"] = per_rank
    if unb is not None:
        line["unbounded_path"] = unb
    if trilinear is not None:
        line["e2e_trilinear"] = trilinear
    if parity is not None:
        line["parity_check"] = parity
        line["cpu_baseline"] = cpu_line
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    if parity is not None and not parity["ok"]:
        print("bench.py: PARITY GATE FAILED: " + json.dumps(parity), file=sys.stderr)
        return 3
    return 0


if __name__ == "__main__":
    sys.exit(main())

"""Cost of the 2-D score metrics of the grid search (Batch.score_metric, hb2_batch_score_metric) at bench.py's cfg2 shape.

One 200-candidate cfg2 batch (bench.job_chunks chunk 0, the reference's default positive rule), solved once with LSMR
(+ the bounded branch); then every metric is run on it twice (warm-up, timed).  Prints one JSON object:

  * solve: device ms of the solve (LSMR + bounded branch + cosine score) per candidate
  * metrics[m]: device ms of the metric stage per candidate (CUDA events around hb2_batch_score_metric) and its share
    of the solve's device time
  * e2e[m]: candidates/s of search_grid(score_metric=m) over the chunk's twist rows, host clock, against cosine
  * host_metric_ms: _metric_2d on the host (the per-candidate path of lsq_reconstruct) for two candidates, per metric
  * gpu: card name, power limit and maximum SM clock, read in the same run

usage: python profiles/score_metric_grid.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from helicon_b200.engine import Batch, Problem  # noqa: E402
from helicon_b200.grid import search_grid  # noqa: E402
from helicon_b200.solver_linear_regression import _metric_2d  # noqa: E402

METRICS = ("ssim", "ms_ssim", "mutual_information", "composite")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    cfg = bench.CONFIGS["cfg2"]
    img = bench.config_image(cfg)
    probs = {}

    def problem(key):
        if key not in probs:
            D2, L2, D3, D3i, s, L3 = key
            probs[key] = Problem(img, s, D2, L2, D3, D3i / 2, D3 // 2 - 1)
        return probs[key]

    chunks, _ = bench.job_chunks(cfg, 1, cfg["batch"], -1, lambda key: problem(key).ndisk)
    key, tasks = chunks[0][0], chunks[0][1]
    specs = [t.spec for t in tasks]
    nc = len(specs)
    b = Batch(problem(key), key[5], specs)
    b.solve()
    tm = b.timing()
    solve_ms = tm["lsmr_ms"] + tm["trf_ms"] + tm["score_ms"]
    t0 = time.perf_counter()
    b.set_pixel_rows()
    table_s = time.perf_counter() - t0
    metrics = {}
    for m in METRICS:
        b.score_metric(m)  # warm-up
        torch.cuda.synchronize()
        b.score_metric(m)
        ms = b.timing()["metric_ms"]
        metrics[m] = dict(device_ms=ms, device_ms_per_candidate=ms / nc, share_of_solve=ms / solve_ms)
    # the host path: prediction downloaded, scattered and scored with numpy / scipy, per candidate
    D2, L2 = key[0], key[1]
    host = {}
    xs = {c: b.x(c) for c in (0, nc // 2)}  # before apply_forward, which leaves the batch unsolved
    for m in METRICS:
        ts = []
        for c in (0, nc // 2):
            pidx, kk, jj = b.data_row_index(c)
            pred = b.apply_forward(c, xs[c])[pidx]
            t1 = time.perf_counter()
            _metric_2d(m, pred, b.rhs_padded(c)[pidx], kk * D2 + jj, img, D2, L2, -1)
            ts.append((time.perf_counter() - t1) * 1e3)
        host[m] = float(np.mean(ts))
    b.close()
    for p in probs.values():
        p.close()
    twists = np.unique([t.twist for t in tasks])
    e2e = {}
    for m in ("cosine",) + METRICS:
        search_grid(np.array(img, copy=True), bench.APIX, twists[:1], cfg["rises"][:4], score_metric=m)  # warm-up
        t0 = time.perf_counter()
        out = search_grid(np.array(img, copy=True), bench.APIX, twists, cfg["rises"], score_metric=m)
        s = time.perf_counter() - t0
        e2e[m] = dict(candidates_per_s=out["n_candidates"] / s, candidates=int(out["n_candidates"]), seconds=s,
                      kernel_ms=float(out["kernel_ms"]))
    result = dict(
        workload=f"cfg2 chunk 0: {nc} candidates, L3={key[5]}, D2={D2}, L2={L2}, default positive rule, LSMR",
        gpu=gpu,
        solve=dict(device_ms=solve_ms, device_ms_per_candidate=solve_ms / nc),
        pixel_tables_s=table_s,
        metrics=metrics,
        e2e=e2e,
        host_metric_ms_per_candidate=host,
    )
    print(json.dumps(result))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()

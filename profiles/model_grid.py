"""Throughput of the batched ElasticNet solver (Batch.solve_model) at bench.py's cfg2 shape.

One 200-candidate cfg2 batch (bench.job_chunks chunk 0, the reference's default positive rule), elasticnet with the
reference's defaults (alpha 1e-4, l1_ratio 0.5).  One warm-up solve of the same batch, then a timed one.  Prints one
JSON object:

  * device: candidates/s from the library's device time (model iterations + score) of the timed solve
  * e2e: candidates/s of search_grid(algorithm=elasticnet) over the same twist rows (setup, solve, score map), host clock
  * iterations: distribution of the final fit's iterations, candidates that hit max_iter, refits (alpha < 1e-4)
  * host_path: regularized.solve_model (host-driven FISTA, one host round trip per product) on two of the candidates
  * gpu: card name and power limit, read in the same run

usage: python profiles/model_grid.py [--out FILE]
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
from helicon_b200 import _lib  # noqa: E402
from helicon_b200.engine import Batch, Problem  # noqa: E402
from helicon_b200.grid import search_grid  # noqa: E402
from helicon_b200.regularized import solve_model  # noqa: E402

ALG = dict(model="elasticnet")


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
    b = Batch(problem(key), key[5], specs)
    b.solve_model(ALG)  # warm-up: module load, allocations
    torch.cuda.synchronize()
    b.close()
    b = Batch(problem(key), key[5], specs)
    t0 = time.perf_counter()
    res = b.solve_model(ALG)
    wall = time.perf_counter() - t0
    tm = b.timing()
    infos = [b.model_info(c) for c in range(b.nc)]
    it = res["itn"].astype(np.int64)
    device_ms = tm["lsmr_ms"] + tm["score_ms"]
    # the host-driven path on two of the same candidates
    host = []
    for c in (0, b.nc // 2):
        info = {}
        t1 = time.perf_counter()
        solve_model(b, c, ALG, bool(b.plan.cands[c]["positive"]), info=info)
        host.append(dict(candidate=c, seconds=time.perf_counter() - t1, iterations=int(info["iterations"]),
                         device_iterations=int(it[c]), alpha=float(info["alpha"])))
    b.close()
    for p in probs.values():
        p.close()
    # end to end: search_grid over the twist rows of the same chunk
    twists = np.unique([t.twist for t in tasks])
    search_grid(np.array(img, copy=True), bench.APIX, twists[:1], cfg["rises"][:4], algorithm=ALG)  # warm-up
    t0 = time.perf_counter()
    out = search_grid(np.array(img, copy=True), bench.APIX, twists, cfg["rises"], algorithm=ALG)
    e2e_s = time.perf_counter() - t0
    result = dict(
        workload=f"cfg2 chunk 0: {len(specs)} candidates, L3={key[5]}, elasticnet alpha 1e-4 l1_ratio 0.5, "
                 "default positive rule",
        gpu=gpu,
        device=dict(candidates_per_s=len(specs) / (device_ms / 1e3), device_ms=device_ms, model_ms=tm["lsmr_ms"],
                    score_ms=tm["score_ms"], batch_iterations=tm["iterations"], launches=tm["launches"],
                    wall_s=wall, us_per_candidate_iteration=device_ms * 1e3 / max(1, int(it.sum()))),
        e2e=dict(candidates_per_s=out["n_candidates"] / e2e_s, candidates=int(out["n_candidates"]), seconds=e2e_s),
        iterations=dict(min=int(it.min()), median=float(np.median(it)), mean=float(it.mean()), max=int(it.max()),
                        p90=float(np.percentile(it, 90)), hit_max_iter=int((res["flags"] & _lib.HB2_FLAG_NOT_CONVERGED != 0).sum()),
                        refitted=int(sum(i["alpha"] < 1e-4 * 0.99 for i in infos)),
                        positive=int(sum(bool(s.positive) for s in specs))),
        host_path=host,
    )
    print(json.dumps(result))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()

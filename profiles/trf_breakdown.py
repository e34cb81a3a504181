"""Where the bounded (TRF) branch spends its device time, for one bench-shape batch.

Solves one batch of bench.py's cfg2 job (bench.job_chunks, 200 candidates, the reference's default positive rule, so
every candidate runs the float64 TRF branch after LSMR) under torch.profiler with CUDA activities, after one unprofiled
solve of the same batch as warm-up.  Kernel time is grouped by class.  Prints one JSON object:

  * us_per_candidate_trf_iteration: TRF-phase kernel time / sum of the candidates' trf_nit
  * per_outer_iteration: launches of each class per lock-step outer iteration of the batch
  * algorithmic forwards/adjoints per candidate outer iteration, from the per-iteration traces
  * step_kinds: how often each select_step outcome was taken (full step = the one that still runs a step forward)
  * trf_nit per candidate

usage: python profiles/trf_breakdown.py [--repo TREE] [--chunk I] [--label NAME] [--out FILE]
``--repo`` profiles the package of another checkout (e.g. a parent build) with this script; ``--out`` merges the
result into FILE under ``--label``.
"""
import argparse
import json
import os
import re
import subprocess
import sys

ap = argparse.ArgumentParser()
ap.add_argument("--repo", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--chunk", type=int, default=0, help="index into bench.job_chunks (default 0)")
ap.add_argument("--label", default="this")
ap.add_argument("--out", default="")
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.repo))

import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

import bench  # noqa: E402
from helicon_b200 import _lib  # noqa: E402
from helicon_b200.engine import Batch, Problem  # noqa: E402

CLASSES = ("fwd64", "fwd64_sym", "adj64", "elementwise", "mspace", "reduce_scalar")
MSPACE_OPS = None  # k_trf_pass<OP> ids of the m-space passes, read from the source of the profiled tree


def mspace_ops(repo):
    src = open(os.path.join(repo, "helicon_b200", "csrc", "hb2_trf.cuh")).read()
    m = re.search(r"enum \{\s*EW_START = 0,(.*?)\};", src, re.S)
    if m is None or "k_trf_pass" not in src:
        return set()
    names = ["EW_START"] + re.findall(r"^\s*(\w+),?\s*(?://.*)?$", m.group(1), re.M)
    return {i for i, n in enumerate(names) if n.startswith("MW_")}


def kernel_class(name):
    if "double" in name or "TD" in name:
        if re.search(r"\bk_fwd64_sym\b", name):
            return "fwd64_sym"
        if re.search(r"\bk_(fwd_band|fwd_band_reduce|fwd64_data|fwd_tie|fwd_csr|fwd_bil|fwd_lsym)\b", name) and "double" in name:
            return "fwd64"
        if re.search(r"\bk_(adj_tile|adj64|adj_tie|adj_csc|adj_bil|adj_bil_tile|bil_unblend|adj_lsym)\b", name) and (
                "double" in name or "k_adj64" in name):
            return "adj64"
    if re.search(r"\bk_trf_(reduce|scal)\b", name):
        return "reduce_scalar"
    if re.search(r"\bk_trf_mw\b", name):
        return "mspace"
    m = re.search(r"\bk_trf_pass<(\d+)>", name)
    if m:
        return "mspace" if int(m.group(1)) in MSPACE_OPS else "elementwise"
    if re.search(r"\bk_trf_(ew|start_apply)\b", name):
        return "elementwise"
    return None


def main():
    global MSPACE_OPS
    MSPACE_OPS = mspace_ops(os.path.abspath(args.repo))
    cfg = bench.CONFIGS["cfg2"]
    img = bench.config_image(cfg)
    probs = {}

    def problem(key):
        if key not in probs:
            D2, L2, D3, D3i, s, L3 = key
            probs[key] = Problem(img, s, D2, L2, D3, D3i / 2, D3 // 2 - 1)
        return probs[key]

    chunks, _ = bench.job_chunks(cfg, args.chunk + 1, cfg["batch"], -1, lambda key: problem(key).ndisk)
    key, tasks = chunks[args.chunk][0], chunks[args.chunk][1]
    specs = [t.spec for t in tasks]

    def solve():
        b = Batch(problem(key), key[5], specs)
        res = b.solve()
        torch.cuda.synchronize()
        return b, res

    b, _ = solve()  # warm-up: module load, allocations
    b.close()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        b, res = solve()
    tm = np.zeros(16, dtype=np.float64)
    _lib.check(_lib.load().hb2_batch_timing(b._h, _lib.ptr(tm)))
    traces = [b.trf_trace(c) for c in range(b.nc)]
    b.close()
    for p in probs.values():
        p.close()

    ms, n = dict.fromkeys(CLASSES, 0.0), dict.fromkeys(CLASSES, 0)
    for ev in prof.key_averages():
        k = kernel_class(ev.key)
        if k is None or ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        ms[k] += t / 1e3
        n[k] += ev.count
    trf_nit = res["trf_nit"].astype(int)
    outer = int(tm[13])
    total = sum(ms.values())
    kinds = np.zeros(4, dtype=int)
    inner, fwd_alg, adj_alg, n_it = 0.0, 0.0, 0.0, 0
    split = bool(MSPACE_OPS)  # the tree forms A*step from the select_step products and takes A^T r from the gradient
    for tr, nit, status in traces:
        for row in tr:
            if row[2] == 0 and row[0] == 0:
                continue  # iteration that stopped before its inner solve
            kind, k_in = int(row[3]), float(row[2])
            kinds[kind] += 1
            inner += k_in
            n_it += 1
            if split:  # inner + select_step (A D RH, A D PH, A ag; a full step only A D PH) + residual
                fwd_alg += k_in + (1 if kind == 0 else 3) + 1
                adj_alg += k_in + 1
            else:  # inner + select_step (none for a full step) + step + residual; inner-init adjoint + gradient
                fwd_alg += k_in + (0 if kind == 0 else 3) + 2
                adj_alg += k_in + 2
    sm = torch.cuda.get_device_properties(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable: {e}"
    out = dict(
        tree=args.label, card=sm.name, nvidia_smi=q, chunk=args.chunk, candidates=int(b.nc),
        trf_phase_ms_event=round(float(tm[1]), 2), trf_kernel_ms=round(total, 2),
        kernel_ms={k: round(v, 2) for k, v in ms.items()}, launches={k: n[k] for k in CLASSES},
        lockstep_outer_iterations=outer,
        per_outer_iteration={k: round(n[k] / max(1, outer), 2) for k in CLASSES},
        sum_trf_nit=int(trf_nit.sum()), mean_trf_nit=round(float(trf_nit.mean()), 3),
        us_per_candidate_trf_iteration=round(1e3 * total / max(1, int(trf_nit.sum())), 1),
        candidate_outer_iterations=n_it, mean_inner_iterations=round(inner / max(1, n_it), 3),
        forwards_per_candidate_outer_iteration=round(fwd_alg / max(1, n_it), 3),
        adjoints_per_candidate_outer_iteration=round(adj_alg / max(1, n_it), 3),
        step_kinds=dict(full=int(kinds[0]), p=int(kinds[1]), r=int(kinds[2]), ag=int(kinds[3])),
        trf_nit=trf_nit.tolist(),
    )
    print(json.dumps(out))
    if args.out:
        data = json.load(open(args.out)) if os.path.exists(args.out) else {}
        data[args.label] = out
        json.dump(data, open(args.out, "w"), indent=1)


if __name__ == "__main__":
    main()

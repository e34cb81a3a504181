"""denovo3DBatch -- command line driver of the batched grid search (helicon's README.md:27 announces a
``denovo3DBatch`` tool; the reference repository ships only the Shiny app, whose "run" handler (app.py:2330-2523) this
mirrors): read 2-D images from an MRC file, search the (twist x rise [x csym]) grid on all visible GPUs, write the
score table, the top-K list and -- optionally -- the symmetrised map of the best candidate (app.py:1267-1287).

One process per GPU: ``python -m helicon_b200.denovo3DBatch ...`` for one GPU, or
``python -m torch.distributed.run --nproc-per-node N -m helicon_b200.denovo3DBatch ...`` to shard the grid over N
GPUs (ranks take disjoint candidates; NCCL only all-gathers score tiles and top-K).  There is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import struct
import sys

import numpy as np


def write_mrc(path, vol, apix):
    """Minimal MRC2014 writer (mode 2, little-endian), the counterpart of ``pipeline._read_mrc``: what the reference
    does with ``mrcfile.new(...).set_data(vol); mrc.voxel_size = apix`` (app.py:1280-1284)."""
    vol = np.ascontiguousarray(vol, dtype="<f4")
    if vol.ndim == 2:
        vol = vol[None]
    nz, ny, nx = vol.shape
    hdr = bytearray(1024)
    struct.pack_into("<4i", hdr, 0, nx, ny, nz, 2)
    struct.pack_into("<3i", hdr, 28, nx, ny, nz)                       # mx, my, mz
    struct.pack_into("<3f", hdr, 40, nx * apix, ny * apix, nz * apix)  # cell dimensions (A)
    struct.pack_into("<3f", hdr, 52, 90.0, 90.0, 90.0)
    struct.pack_into("<3i", hdr, 64, 1, 2, 3)                          # mapc, mapr, maps
    struct.pack_into("<3f", hdr, 76, float(vol.min()), float(vol.max()), float(vol.mean()))
    struct.pack_into("<i", hdr, 88, 1)                                 # ispg
    hdr[104:108] = b"\x00\x00\x00\x00"
    struct.pack_into("<i", hdr, 108, 20140)                            # nversion
    hdr[208:212] = b"MAP "
    hdr[212:216] = bytes([0x44, 0x44, 0x00, 0x00])                     # little-endian machine stamp
    struct.pack_into("<f", hdr, 216, float(vol.std()))
    with open(path, "wb") as f:
        f.write(bytes(hdr))
        f.write(vol.tobytes())


def _axis(spec, name):
    """'lo:hi:n' (linspace), 'a,b,c' (list) or a single number."""
    if ":" in spec:
        lo, hi, n = spec.split(":")
        return np.linspace(float(lo), float(hi), int(n))
    vals = np.array([float(v) for v in spec.split(",")], dtype=np.float64)
    if len(vals) == 0:
        raise SystemExit(f"--{name}: empty")
    return vals


def main(argv=None):
    ap = argparse.ArgumentParser(prog="denovo3DBatch", description=__doc__.split("\n\n")[0])
    ap.add_argument("image", help="MRC file with one 2-D image or a stack of 2-D class averages")
    ap.add_argument("--index", default="all", help="image indices in the stack: 'all' or a comma list (default all)")
    ap.add_argument("--apix", type=float, default=0.0, help="pixel size in Angstrom (default: from the MRC header)")
    ap.add_argument("--twist", required=True, help="twist grid in degrees: 'lo:hi:n', a comma list or one value "
                                                   "(negative values: --twist=-3:-0.2:100)")
    ap.add_argument("--rise", required=True, help="rise grid in Angstrom: 'lo:hi:n', a comma list or one value")
    ap.add_argument("--csym", default="1", help="cyclic symmetries to search, comma list (default 1)")
    ap.add_argument("--tube-diameter", type=float, default=None, help="Angstrom (default: image height)")
    ap.add_argument("--tube-diameter-inner", type=float, default=0.0)
    ap.add_argument("--tube-length", type=float, default=None, help="Angstrom (default: image width)")
    ap.add_argument("--reconstruct-length-rise", type=float, default=3, help="reconstruct length in units of rise (app default 3)")
    ap.add_argument("--sym-oversample", type=int, default=-1)
    ap.add_argument("--positive-constraint", type=int, default=-1, help="-1 auto (reference rule), 0 off, 1 on")
    ap.add_argument("--interpolation", default="nn", choices=["nn", "linear"])
    ap.add_argument("--top-k", type=int, default=10)
    ap.add_argument("--output", default="denovo3DBatch_out", help="output prefix")
    ap.add_argument("--save-map", action="store_true", help="write the symmetrised 3-D map of the best candidate per image")
    ap.add_argument("--batch-candidates", type=int, default=0, help="candidates per batch (default: sized from GPU memory)")
    ap.add_argument("--resume", action="store_true", help="keep the score tiles of solved batches in <output>_img<i>.tiles"
                    "[.rank<r>].npz and restart an interrupted search from them (same image, grid and parameters)")
    ap.add_argument("--model", default="lsq", choices=["lsq", "elasticnet", "lasso", "ridge"],
                    help="solver model (app.py algorithm; default lsq)")
    ap.add_argument("--alpha", type=float, default=None, help="model alpha (default: 1 for ridge, 1e-4 otherwise)")
    ap.add_argument("--l1-ratio", type=float, default=None, help="elastic-net l1_ratio (default 0.5)")
    ap.add_argument("--score-metric", default="cosine",
                    choices=["cosine", "ssim", "ms_ssim", "mutual_information", "composite"],
                    help="score that ranks the candidates (app.py score_metric; default cosine)")
    args = ap.parse_args(argv)
    algorithm = None
    if args.model != "lsq":
        algorithm = dict(model=args.model)
        if args.alpha is not None:
            algorithm["alpha"] = args.alpha
        if args.l1_ratio is not None:
            algorithm["l1_ratio"] = args.l1_ratio
    elif args.alpha is not None or args.l1_ratio is not None:
        ap.error("--alpha / --l1-ratio need --model elasticnet, lasso or ridge")

    from . import distributed, pipeline, transforms
    from .grid import check_algorithm, search_grid

    check_algorithm(algorithm, args.interpolation)  # before any GPU work

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist

        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    data, apix_hdr = pipeline.get_images_from_file(args.image)
    apix = args.apix if args.apix > 0 else apix_hdr
    if apix <= 0:
        raise SystemExit("pixel size unknown: pass --apix")
    stack = data if data.ndim == 3 else data[None]
    idx = range(len(stack)) if args.index == "all" else [int(v) for v in args.index.split(",")]
    twists, rises = _axis(args.twist, "twist"), _axis(args.rise, "rise")
    csyms = tuple(int(v) for v in args.csym.split(","))
    report = []
    for i in idx:
        img = np.ascontiguousarray(stack[i], dtype=np.float32)
        if pipeline.is_vertical(img):  # the reference transposes vertical filaments (pipeline.py:159-161)
            img = np.ascontiguousarray(img.T)
        out = search_grid(img, apix, twists, rises, csyms=csyms, reconstruct_length_rise=args.reconstruct_length_rise,
                          tube_diameter=args.tube_diameter, tube_diameter_inner=args.tube_diameter_inner,
                          tube_length=args.tube_length, sym_oversample=args.sym_oversample,
                          positive_constraint=args.positive_constraint, top_k=args.top_k, device=local_rank,
                          shard=(rank, world), return_x_top=args.save_map, interpolation=args.interpolation, dist=dist,
                          checkpoint=f"{args.output}_img{i}.tiles" if args.resume else None,
                          batch_candidates=args.batch_candidates or None, algorithm=algorithm,
                          score_metric=args.score_metric)
        # with more than one process the per-rank score maps were all-gathered inside search_grid (one NCCL call)
        if rank != 0:
            continue
        prefix = f"{args.output}_img{i}"
        np.savez_compressed(prefix + "_scores.npz", scores=out["scores"], itn=out["itn"], flags=out["flags"], twists=twists,
                            rises=rises, csyms=np.array(csyms))
        top = [dict(score=e["score"], twist=e["twist"], rise=e["rise"], csym=e["csym"]) for e in out["top"]]
        report.append(dict(image=i, n_candidates=int(np.isfinite(out["scores"]).sum()), seconds=out["seconds"], top=top,
                           n_restored=int(out.get("n_restored", 0)), score_metric=args.score_metric))
        best = out["top"][0] if out["top"] else None
        if best is not None:
            print(f"image {i}: best twist={best['twist']:.4f} rise={best['rise']:.4f} csym={best['csym']} "
                  f"score={best['score']:.6f} ({report[-1]['n_candidates']} candidates, {out['seconds']:.1f} s)", flush=True)
        if args.save_map and best is not None and "rec3d" not in best:
            # the best candidate was solved by another rank: solve it again here (one candidate) for its volume
            from .grid import build_tasks
            from .solver_linear_regression import lsq_reconstruct

            t, _ = build_tasks(img.shape[0], img.shape[1], apix, [best["twist"]], [best["rise"]], csyms=(best["csym"],),
                               reconstruct_length_rise=args.reconstruct_length_rise, tube_diameter=args.tube_diameter,
                               tube_diameter_inner=args.tube_diameter_inner, tube_length=args.tube_length,
                               sym_oversample=args.sym_oversample)
            g = t[0].geom
            (best["rec3d"], _, _), _ = lsq_reconstruct(
                img, g["s"], best["twist"], best["rise"] / g["apix3d"], best["csym"],
                positive_constraint=args.positive_constraint, reconstruct_diameter_3d_inner_pixel=g["D3i"],
                reconstruct_diameter_2d_pixel=g["D2"], reconstruct_length_2d_pixel=g["L2"],
                reconstruct_diameter_3d_pixel=g["D3"], reconstruct_length_3d_pixel=g["L3"],
                sym_oversample=g["sym_oversample"], interpolation=args.interpolation, device=local_rank,
                algorithm=algorithm or dict(model="lsq"))
        if args.save_map and best is not None and "rec3d" in best:
            ny, nx = img.shape
            vol = transforms.apply_helical_symmetry(best["rec3d"], apix, best["twist"], best["rise"], csym=best["csym"],
                                                    new_size=(nx, ny, ny), new_apix=apix)
            write_mrc(prefix + "_best_map.mrc", vol, apix)
    if rank == 0:
        with open(args.output + "_top.json", "w") as f:
            json.dump(report, f, indent=1)
    if dist is not None:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())

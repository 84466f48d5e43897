"""Cost of FPFH features (apc_compute_fpfh / apc_compute_fpfh_knn) and feature matching
(apc_correspondences_from_features) on one GPU: the time of every kernel of a call (CUDA events, ``ctx.profile(True)``)
and of the whole call (CUDA events around RUNS calls, profiler off), with the GPU's name and power limit read in the
same run.

Inputs: a 128 x 2048 synthetic LiDAR scan (262 144 points) and its 0.2 m voxel downsampling, with a copy of the
downsampled cloud moved by 10 degrees and 1 m.  Normals: ``estimate_normals`` hybrid (30 within 0.5 m) on the GPU.
FPFH: hybrid (100 within 1.0 m) and KNN (100) on the full scan and on the downsampled cloud.  Matching: the
downsampled cloud's FPFH against the moved copy's, without and with the mutual filter; its operation count is
n_src * n_tgt * dim * 3 (subtract, multiply, add) per direction, reported next to the time.  ``true_fraction``: the
share of mutual pairs whose target point is the source point's image (within 1 cm).
Usage: python profiles/features.py [out.json]   (default profiles/features.json)"""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from wide_neighbors import gpu_info
from registration import call_us, profiled, to_xyzi, RUNS
from autodriver_pointcloud_preprocessor_b200 import engine, synth
from oracle import registration as reg
from oracle import voxel


def fpfh_case(ctx, name, p, nrm, max_nn, radius):
    xyzi = to_xyzi(p)
    run = lambda: ctx.compute_fpfh(xyzi, nrm, max_nn, radius)
    run()
    ctx.check()
    per, launches = profiled(ctx, run)
    return dict(name=name, points=int(p.shape[0]), max_nn=max_nn, radius=radius, call_us=call_us(run),
                kernels_us={k: v for k, v in per.items() if k.startswith("k_fpfh") or k.startswith("k_grid")},
                launches={k: v for k, v in launches.items() if k.startswith("k_fpfh")})


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "features.json")
    res = dict(gpu_info(), runs_per_config=RUNS, fpfh=[], matching=[])
    scan = synth.lidar_scan(seed=3, n_beams=128, n_az=2048, nan_frac=0.0)["positions"].astype(np.float32)
    scan = np.ascontiguousarray(scan)
    down = np.ascontiguousarray(voxel.voxel_down_sample(scan, 0.2, None, fixed=True)["positions"])
    T = reg.pose_to_transformation([0.0, 0.0, np.deg2rad(10.0), 1.0, -0.5, 0.1])
    moved = np.ascontiguousarray(reg.transform_points(down, T))
    ctx = engine.Context(max_points=scan.shape[0])
    normals = {}
    for key, p in (("scan", scan), ("down", down), ("moved", moved)):
        nrm, _, _ = ctx.estimate_normals(to_xyzi(p), 30, 0.5)
        ctx.check()
        normals[key] = nrm.contiguous()
    for key, p in (("full scan", scan), ("0.2 m voxels", down)):
        nrm = normals["scan" if key == "full scan" else "down"]
        res["fpfh"].append(fpfh_case(ctx, f"{key}, hybrid", p, nrm, 100, 1.0))
        res["fpfh"].append(fpfh_case(ctx, f"{key}, KNN", p, nrm, 100, None))
    fs, _, _ = ctx.compute_fpfh(to_xyzi(down), normals["down"], 100, 1.0)
    ft, _, _ = ctx.compute_fpfh(to_xyzi(moved), normals["moved"], 100, 1.0)
    ctx.check()
    fs, ft = fs.contiguous(), ft.contiguous()
    for mutual in (False, True):
        run = lambda: ctx.correspondences_from_features(fs, ft, mutual, 0.1)
        pairs, info, _ = run()
        ctx.check()
        count, fell_back = (int(v) for v in info.cpu().tolist())
        pr = pairs[:count].cpu().numpy()
        img = reg.transform_points(down[pr[:, 0]], T)
        true = float(np.mean(np.linalg.norm(img - moved[pr[:, 1]], axis=1) < 0.01)) if count else 0.0
        per, launches = profiled(ctx, run)
        us = call_us(run)
        ops = fs.shape[0] * ft.shape[0] * fs.shape[1] * 3 * (2 if mutual else 1)
        res["matching"].append(dict(n_src=int(fs.shape[0]), n_tgt=int(ft.shape[0]), dim=int(fs.shape[1]),
                                    mutual_filter=mutual, pairs=count, fell_back=bool(fell_back),
                                    true_fraction=round(true, 4), call_us=us, kernels_us=per, launches=launches,
                                    flops=ops, gflops_per_s=round(ops / us * 1e-3, 1)))
    ctx.close()
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

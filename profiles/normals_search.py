"""Cost of estimate_normals with one search bound (KNN: max_nn only; radius: radius only) next to the hybrid
search, on one GPU, with every kernel bracketed by CUDA events (``ctx.profile(True)``).

Clouds: the C2 frame of bench.py (262 144-point scan) through the front end of the reference's default set
(NaN skip, duplicate removal, non-finite filter, ROI crop), voxelized at 0.1 m and at the reference's default
0.01 m.  On each: KNN at max_nn in {30, 100, 1024}, radius search at r in {0.1, 0.5, 1.0} m, and the hybrid
search (r = 0.5 m, max_nn = 30) for comparison.  Per configuration one warm-up call, then RUNS profiled calls;
the JSON holds the mean time per launch of every kernel of the call, their sum, and the neighbour counts
(mean / max), with the GPU's name and power limit.

``--wide-ab BEFORE AFTER``: two outputs of ``profiles/wide_neighbors.py`` taken in the same session (before
and after a change); their k_knn_query_wide rows at k = 65 and 1024 on C4 are copied into the result.
Usage: python profiles/normals_search.py [out.json] [--wide-ab BEFORE.json AFTER.json]
(default profiles/normals_search.json)"""
import json, os, sys
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
import bench
from wide_neighbors import gpu_info
from autodriver_pointcloud_preprocessor_b200 import _capi, engine

RUNS = 10
KERNELS = ("k_grid_insert", "k_grid_assign", "k_grid_scatter", "k_normals_knn", "k_normals_knn_stragglers",
           "k_normals_radius", "k_normals_cov", "k_normals_query", "k_normals_wide", "k_normals_eigen", "k_grid_clean")


def voxel_cloud(ctx, desc, fcfg, voxel_size):
    xyzi, _, _, cnt = ctx.frontend([desc], fcfg, want_src=False)
    out, _, _, vcnt = ctx.voxel_downsample(xyzi[:int(cnt.item())], voxel_size)
    ctx.check()
    return out[:int(vcnt.item())].clone()


def profile_call(ctx, fn):
    fn()                                                                 # warm-up (allocations, module load)
    ctx.check()
    ctx.profile(True)
    for _ in range(RUNS):
        _, cnt, _ = fn()
    rep = ctx.profile_report()
    ctx.profile(False)
    ctx.check()
    per = {k: round(ms / n * 1e3, 1) for k, (ms, n) in rep.items() if k in KERNELS}
    c = cnt.double()
    return dict(kernels_us=per, call_us=round(sum(per.values()), 1),
                neighbours_mean=round(float(c.mean().item()), 1), neighbours_max=int(c.max().item()))


def main():
    args = sys.argv[1:]
    wide = None
    if "--wide-ab" in args:
        i = args.index("--wide-ab")
        wide = args[i + 1:i + 3]
        del args[i:i + 3]
    path = args[0] if args else os.path.join(ROOT, "profiles", "normals_search.json")
    res = dict(gpu_info(), runs_per_config=RUNS, clouds=[])
    m = bench.make_frames(1, seed0=3)[0]
    ctx = engine.Context(max_points=m.width)
    desc = engine.make_cloud_desc(m.fields, m.point_step, m.width, torch.frombuffer(bytearray(m.data), dtype=torch.uint8).cuda())
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=_capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True, crop=bench.CROP)
    for voxel_size in (0.1, 0.01):
        xyzi = voxel_cloud(ctx, desc, fcfg, voxel_size)
        cloud = dict(voxel_size=voxel_size, points=int(xyzi.shape[0]), runs=[])
        configs = [("knn", dict(max_nn=k), lambda k=k: ctx.estimate_normals_knn(xyzi, k, want_counts=True)) for k in (30, 100, 1024)]
        configs += [("radius", dict(radius=r), lambda r=r: ctx.estimate_normals_radius(xyzi, r, want_counts=True))
                    for r in (0.1, 0.5, 1.0)]
        configs.append(("hybrid", dict(radius=0.5, max_nn=30), lambda: ctx.estimate_normals(xyzi, 30, 0.5, want_counts=True)))
        for mode, params, fn in configs:
            r = dict(mode=mode, **params, **profile_call(ctx, fn))
            print(voxel_size, json.dumps(r), flush=True)
            cloud["runs"].append(r)
        res["clouds"].append(cloud)
    ctx.close()
    if wide:
        rows = {}
        for side, f in zip(("before", "after"), wide):
            stat = json.load(open(f))["statistical"]
            rows[side] = {str(r["k"]): r["kernels_us"]["k_knn_query_wide"] for r in stat if r["k"] in (65, 1024)}
        res["k_knn_query_wide_c4_us"] = rows
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()

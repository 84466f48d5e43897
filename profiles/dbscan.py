"""Cost of cluster_dbscan (apc_cluster_dbscan) on one GPU: the time of every kernel of the call (CUDA events,
``ctx.profile(True)``) and of the whole call (CUDA events around RUNS calls, profiler off), with the GPU's name and
power limit read in the same run.

Inputs:
  (a) a C2-shaped scan (``synth.lidar_scan``, 128 x 2048) voxelised at 0.1 m, with the ground removed by
      ``segment_plane`` (0.2 m, ransac_n 3, 200 iterations), at eps in {0.3, 0.5, 1.0} m x min_points in {5, 10};
  (b) the raw 262 144-point scan at eps = 0.5 m, min_points = 10, where neighbourhoods are large;
  (c) ``dense_patch`` of tests/test_gpu_normals_search.py (6 003 points, neighbourhoods above 1 024) at eps = 0.45.
Next to each time: ``neighbour_tests`` = sum |N(i)| (the distance tests a walk over exactly the neighbourhoods
makes), whether labels, cluster count and neighbour counts equal ``oracle.dbscan``, and the oracle's host time
(scipy, one CPU run) as a CPU reference point only.
Usage: python profiles/dbscan.py [out.json]   (default profiles/dbscan.json)"""
import json, os, sys, time
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from wide_neighbors import gpu_info
from test_gpu_normals_search import dense_patch
from autodriver_pointcloud_preprocessor_b200 import engine, geometry as o3d, synth
from oracle import dbscan as odb
from oracle import voxel

RUNS = 20
KERNELS = ("k_grid_insert", "k_grid_assign", "k_grid_scatter", "k_dbscan_core", "k_dbscan_union", "k_dbscan_roots",
           "k_dbscan_label", "k_grid_clean")


def to_xyzi(p):
    return torch.from_numpy(np.concatenate([p, np.zeros((p.shape[0], 1), np.float32)], 1)).cuda()


def measure(ctx, p, eps, min_points):
    xyzi = to_xyzi(p)
    labels, n_cl, counts = ctx.cluster_dbscan(xyzi, eps, min_points, want_counts=True)   # warm-up, and the result
    ctx.check()
    got = (labels.cpu().numpy(), int(n_cl.item()), counts.cpu().numpy())
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(RUNS):
        ctx.cluster_dbscan(xyzi, eps, min_points)
    b.record()
    torch.cuda.synchronize()
    call_us = a.elapsed_time(b) / RUNS * 1e3
    ctx.profile(True)
    for _ in range(RUNS):
        ctx.cluster_dbscan(xyzi, eps, min_points)
    rep = ctx.profile_report()
    ctx.profile(False)
    ctx.check()
    per = {k: round(ms / n * 1e3, 1) for k, (ms, n) in rep.items() if k in KERNELS}
    t = time.perf_counter()
    ref, n_ref, cnt_ref, tests = odb.dbscan(p, eps, min_points)
    host_ms = (time.perf_counter() - t) * 1e3
    equal = bool(np.array_equal(got[0], ref) and got[1] == n_ref and np.array_equal(got[2], cnt_ref.astype(np.int32)))
    return dict(points=int(p.shape[0]), eps=eps, min_points=min_points, kernels_us=per,
                kernels_sum_us=round(sum(per.values()), 1), call_us=round(call_us, 1), neighbour_tests=tests,
                neighbours_mean=round(tests / p.shape[0], 1), neighbours_max=int(cnt_ref.max()), clusters=n_ref,
                noise=int((ref == -1).sum()), equal_to_oracle=equal, oracle_cpu_ms=round(host_ms, 1))


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "dbscan.json")
    res = dict(gpu_info(), runs_per_config=RUNS, inputs=[])
    scan = synth.lidar_scan(seed=3, n_beams=128, n_az=2048, nan_frac=0.0)["positions"].astype(np.float32)
    ctx = engine.Context(max_points=scan.shape[0])
    pcd = o3d.PointCloud(o3d.Device("CUDA:0"))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(voxel.voxel_down_sample(scan, 0.1, None, fixed=True)["positions"]).cuda())
    _, inliers = pcd.segment_plane(distance_threshold=0.2, ransac_n=3, num_iterations=200, seed=3)
    objects = np.ascontiguousarray(pcd.select_by_index(inliers, invert=True).point.positions.cpu().numpy(), np.float32)
    cases = [("a: C2 voxels 0.1 m, ground removed", objects, eps, mp) for eps in (0.3, 0.5, 1.0) for mp in (5, 10)]
    cases.append(("b: raw C2 scan", scan, 0.5, 10))
    cases.append(("c: dense_patch", dense_patch(), 0.45, 10))
    for name, p, eps, mp in cases:
        r = dict(input=name, **measure(ctx, p, eps, mp))
        print(json.dumps(r), flush=True)
        res["inputs"].append(r)
    ctx.close()
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()

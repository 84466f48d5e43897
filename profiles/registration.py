"""Cost of ICP (apc_icp) and evaluate_registration on one GPU: the time of every kernel of the call (CUDA events,
``ctx.profile(True)``) and of the whole call (CUDA events around RUNS calls, profiler off), with the GPU's name and
power limit read in the same run.

Inputs:
  (a) the recovery pair of tests/test_oracle_registration.py: a C2-shaped scan voxelised at 0.1 m as the target,
      another noise draw of the same scene voxelised on a shifted grid and moved by 0.5 m / 3 degrees as the
      source; max_correspondence_distance 1.0 m;
  (b) a C2-shaped scan voxelised at 0.01 m (about 260 k points) as the target and a copy moved by 0.1 m / 1 degree
      as the source; max_correspondence_distance 0.5 m.
Both estimations, the point-to-plane one with the target's radius normals (0.5 m) computed on the GPU.  Next to
each time: the iterations run, whether the loop agrees with ``oracle.registration.icp`` (iterations, convergence,
correspondences; T within 1e-9), and:
  * ``early_exit_us``: the call with max_iteration = 30 minus the call with max_iteration = the iterations the
    loop needed - the cost of the (match, solve) pairs launched after the loop stopped, which return at once;
  * ``dbscan_core_us``: k_dbscan_core on the target at the same radius (one pass over the same 27 cells).
Usage: python profiles/registration.py [out.json]   (default profiles/registration.json)"""
import json, os, sys, time
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from wide_neighbors import gpu_info
from test_oracle_registration import recovery_pair
from autodriver_pointcloud_preprocessor_b200 import engine, synth
from oracle import registration as reg
from oracle import voxel

RUNS = 20
KERNELS = ("k_grid_insert", "k_grid_assign", "k_grid_scatter", "k_icp_init", "k_icp_match", "k_icp_solve",
           "k_grid_clean")


def to_xyzi(p):
    return torch.from_numpy(np.concatenate([p, np.zeros((p.shape[0], 1), np.float32)], 1)).cuda()


def call_us(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(RUNS):
        fn()
    b.record()
    torch.cuda.synchronize()
    return round(a.elapsed_time(b) / RUNS * 1e3, 1)


def profiled(ctx, fn):
    ctx.profile(True)
    for _ in range(RUNS):
        fn()
    rep = ctx.profile_report()
    ctx.profile(False)
    ctx.check()
    # per call: total time of each kernel over its launches in one call
    return {k: round(ms / RUNS * 1e3, 1) for k, (ms, n) in rep.items()}, {k: n // RUNS for k, (ms, n) in rep.items()}


def measure(ctx, src, tgt, r, method, normals):
    xs, xt = to_xyzi(src), to_xyzi(tgt)
    nrm = torch.from_numpy(normals).cuda() if method == reg.POINT_TO_PLANE else None
    run = lambda it=30: ctx.icp(xs, xt, r, method=method, tgt_normals=nrm, max_iteration=it)
    T, stats, info, corr = run()                                         # warm-up, and the result
    ctx.check()
    T, stats, info, corr = T.cpu().numpy(), stats.cpu().numpy(), info.cpu().numpy(), corr.cpu().numpy()
    iters = int(info[0])
    full = call_us(run)
    exact = call_us(lambda: run(iters))
    per, launches = profiled(ctx, run)
    per = {k: v for k, v in per.items() if k in KERNELS}
    ev = call_us(lambda: ctx.evaluate_registration(xs, xt, r, T))
    ev_per, _ = profiled(ctx, lambda: ctx.evaluate_registration(xs, xt, r, T))
    _, _, db_counts = ctx.cluster_dbscan(xt, r, 10, want_counts=True)
    db_per, _ = profiled(ctx, lambda: ctx.cluster_dbscan(xt, r, 10, want_counts=True))
    t0 = time.perf_counter()
    ref = reg.icp(src, tgt, r, method=method, target_normals=normals if method == reg.POINT_TO_PLANE else None)
    host_s = time.perf_counter() - t0
    agree = bool(iters == ref["iterations"] and bool(info[1]) == ref["converged"] and info[2] == ref["status"]
                 and np.array_equal(corr, ref["correspondences"])
                 and np.abs(T - ref["transformation"]).max() < 1e-9)
    return dict(source_points=int(src.shape[0]), target_points=int(tgt.shape[0]), r=r,
                method="point_to_plane" if method == reg.POINT_TO_PLANE else "point_to_point",
                iterations=iters, converged=bool(info[1]), fitness=float(stats[0]), inlier_rmse=float(stats[1]),
                kernels_us=per, match_us_per_iteration=round(per.get("k_icp_match", 0.0) / max(iters, 1), 1),
                solve_us_per_iteration=round(per.get("k_icp_solve", 0.0) / max(iters, 1), 1),
                launches_per_call=launches.get("k_icp_match", 0), call_us=full, call_us_exact_iterations=exact,
                early_exit_us=round(full - exact, 1), early_exit_launches=2 * (30 - iters),
                evaluate_call_us=ev, evaluate_kernels_us={k: v for k, v in ev_per.items() if k in KERNELS},
                dbscan_core_us=db_per.get("k_dbscan_core"),
                target_neighbours_mean=round(float(db_counts.float().mean()), 1),
                equal_to_oracle=agree, max_abs_T_diff=float(np.abs(T - ref["transformation"]).max()),
                oracle_cpu_s=round(host_s, 1))


def dense_pair():
    scan = synth.lidar_scan(seed=3, n_beams=128, n_az=2048, nan_frac=0.0)["positions"].astype(np.float32)
    tgt = np.ascontiguousarray(voxel.voxel_down_sample(scan, 0.01, None, fixed=True)["positions"])
    T = reg.pose_to_transformation([0.0, 0.0, np.deg2rad(1.0), 0.08, -0.05, 0.02])
    return np.ascontiguousarray(reg.transform_points(tgt, np.linalg.inv(T))), tgt


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "registration.json")
    res = dict(gpu_info(), runs_per_config=RUNS, inputs=[])
    src_a, tgt_a, _ = recovery_pair()
    src_b, tgt_b = dense_pair()
    ctx = engine.Context(max_points=max(src_b.shape[0], tgt_b.shape[0], src_a.shape[0], tgt_a.shape[0]))
    for name, src, tgt, r in (("a: recovery pair (0.1 m voxels)", src_a, tgt_a, 1.0),
                              ("b: 0.01 m voxels against a moved copy", src_b, tgt_b, 0.5)):
        normals, _, _ = ctx.estimate_normals_radius(to_xyzi(tgt), 0.5)
        normals = normals.cpu().numpy()
        for method in (reg.POINT_TO_POINT, reg.POINT_TO_PLANE):
            r_ = dict(input=name, **measure(ctx, src, tgt, r, method, normals))
            print(json.dumps(r_), flush=True)
            res["inputs"].append(r_)
    ctx.close()
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()

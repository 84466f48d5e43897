"""Cost of generalized ICP (apc_icp_generalized) next to point-to-plane ICP (apc_icp) on one GPU: the time of every
kernel of the call (CUDA events, ``ctx.profile(True)``) and of the whole call (CUDA events around RUNS calls,
profiler off), with the GPU's name and power limit read in the same run.

Inputs (a) and (b) of profiles/registration.py.  Generalized ICP takes the KNN-20 covariances of both clouds
(``PointCloud.estimate_covariances()`` defaults), point-to-plane the target's radius normals (0.5 m), both computed
on the GPU.  For each input and estimation: the iterations run, the kernel and call times, the match kernel's time
per iteration, the pose error against the known motion, and whether the loop agrees with
``oracle.gicp.icp`` / ``oracle.registration.icp`` (iterations, convergence, status, correspondences; T within 1e-9),
generalized ICP fed the regularisation axes the GPU used.  ``estimate_covariances_us``: ``estimate_covariances()``
of both clouds on the carrier (CUDA clouds), once per call.
Usage: python profiles/gicp.py [out.json]   (default profiles/gicp.json)"""
import json, os, sys, time
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
from wide_neighbors import gpu_info
from registration import call_us, dense_pair, profiled, to_xyzi, RUNS
from test_oracle_registration import pose_error, recovery_pair
from autodriver_pointcloud_preprocessor_b200 import engine
from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
from oracle import gicp
from oracle import registration as reg

KERNELS = ("k_grid_insert", "k_grid_assign", "k_grid_scatter", "k_icp_init", "k_gicp_prep", "k_icp_match",
           "k_icp_match_gicp", "k_icp_solve", "k_grid_clean")


def cloud(p):
    pcd = o3d.PointCloud(o3d.Device("CUDA:0"))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(np.ascontiguousarray(p)).cuda())
    return pcd


def measure(ctx, src, tgt, r, T_true, generalized, normals, cs, ct):
    xs, xt = to_xyzi(src), to_xyzi(tgt)
    if generalized:
        run = lambda: ctx.icp_generalized(xs, cs, xt, ct, r)
        T, stats, info, corr, ax_s, ax_t = ctx.icp_generalized(xs, cs, xt, ct, r, want_axes=True)
        match = "k_icp_match_gicp"
    else:
        nrm = torch.from_numpy(normals).cuda()
        run = lambda: ctx.icp(xs, xt, r, method=reg.POINT_TO_PLANE, tgt_normals=nrm)
        T, stats, info, corr = run()
        match = "k_icp_match"
    ctx.check()
    T, stats, info, corr = T.cpu().numpy(), stats.cpu().numpy(), info.cpu().numpy(), corr.cpu().numpy()
    iters = int(info[0])
    call = call_us(run)
    per, _ = profiled(ctx, run)
    per = {k: v for k, v in per.items() if k in KERNELS}
    t0 = time.perf_counter()
    if generalized:
        ref = gicp.icp(src, tgt, r, source_axes=ax_s.cpu().numpy(),
                      target_axes=ax_t.cpu().numpy())
    else:
        ref = reg.icp(src, tgt, r, method=reg.POINT_TO_PLANE, target_normals=normals)
    host_s = time.perf_counter() - t0
    agree = bool(iters == ref["iterations"] and bool(info[1]) == ref["converged"] and info[2] == ref["status"]
                 and np.array_equal(corr, ref["correspondences"])
                 and np.abs(T - ref["transformation"]).max() < 1e-9)
    dt, angle = pose_error(T, T_true)
    return dict(method="generalized" if generalized else "point_to_plane", iterations=iters,
                converged=bool(info[1]), status=int(info[2]), fitness=float(stats[0]), inlier_rmse=float(stats[1]),
                kernels_us=per, match_us_per_iteration=round(per.get(match, 0.0) / max(iters, 1), 1),
                solve_us_per_iteration=round(per.get("k_icp_solve", 0.0) / max(iters, 1), 1), call_us=call,
                translation_error_m=float(dt), rotation_error_deg=float(angle), equal_to_oracle=agree,
                max_abs_T_diff=float(np.abs(T - ref["transformation"]).max()), oracle_cpu_s=round(host_s, 1))


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "gicp.json")
    res = dict(gpu_info(), runs_per_config=RUNS, inputs=[])
    src_a, tgt_a, T_a = recovery_pair()
    src_b, tgt_b = dense_pair()
    T_b = reg.pose_to_transformation([0.0, 0.0, np.deg2rad(1.0), 0.08, -0.05, 0.02])
    ctx = engine.Context(max_points=max(src_b.shape[0], tgt_b.shape[0], src_a.shape[0], tgt_a.shape[0]))
    for name, src, tgt, r, T_true in (("a: recovery pair (0.1 m voxels)", src_a, tgt_a, 1.0, T_a),
                                      ("b: 0.01 m voxels against a moved copy", src_b, tgt_b, 0.5, T_b)):
        normals, _, _ = ctx.estimate_normals_radius(to_xyzi(tgt), 0.5)
        normals = normals.cpu().numpy()
        cs_cloud, ct_cloud = cloud(src).estimate_covariances(), cloud(tgt).estimate_covariances()   # and warm-up
        cs = cs_cloud.point["covariances"].t.contiguous()
        ct = ct_cloud.point["covariances"].t.contiguous()
        cov_us = call_us(lambda: (cs_cloud.estimate_covariances(), ct_cloud.estimate_covariances()))
        out = dict(input=name, source_points=int(src.shape[0]), target_points=int(tgt.shape[0]), r=r,
                   estimate_covariances_us=cov_us,
                   results=[measure(ctx, src, tgt, r, T_true, g, normals, cs, ct) for g in (True, False)])
        g, p = out["results"]
        out["match_per_iteration_ratio_gicp_over_p2l"] = round(g["match_us_per_iteration"] /
                                                               max(p["match_us_per_iteration"], 1e-9), 2)
        print(json.dumps(out), flush=True)
        res["inputs"].append(out)
    ctx.close()
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()

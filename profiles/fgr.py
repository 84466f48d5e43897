"""Cost of Fast Global Registration (apc_fgr_from_features) on one GPU: the time of every kernel of a call (CUDA
events, ``ctx.profile(True)``) and of the whole call (CUDA events around RUNS calls, profiler off), with and without
the tuple test, the launches per call, and the GPU's name and power limit read in the same run.

Inputs: the recovery pair of tests/test_oracle_registration.py (profiles/registration.py's inputs): the target and
the source moved by a further 130 degrees of yaw, both voxelised at 0.3 m and 0.5 m (the sizes a user feeds a global
registration).  Normals: hybrid (30 within 0.8 m), oriented to the vertical; FPFH: hybrid (100 within 1.5 m), both
on the GPU.  ``matching_us`` is the two k_feat_nn searches (O(n_src * n_tgt * 33) each); ``fgr_us`` every other kernel
of the call.  Next to each: the pairs in and used, the tuple trials, and the pose error against the known motion.
Usage: python profiles/fgr.py [out.json]   (default profiles/fgr.json)"""
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
from registration import call_us, profiled, RUNS
from test_oracle_fgr import motion, pose_error
from test_oracle_registration import recovery_pair
from autodriver_pointcloud_preprocessor_b200 import geometry as o3d
from autodriver_pointcloud_preprocessor_b200 import registration as o3dreg
from oracle import registration as reg


def cloud(p):
    pcd = o3d.PointCloud(o3d.Device("CUDA:0"))
    pcd.point["positions"] = o3d.Tensor(torch.from_numpy(np.ascontiguousarray(p)).cuda())
    return pcd


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "fgr.json")
    res = dict(gpu_info(), runs_per_config=RUNS, cases=[])
    src0, tgt0, T_rec = recovery_pair()
    M = motion(130.0, 2.0, -1.0, (4.0, -3.0, 0.2))
    T_true = np.linalg.inv(M)
    for voxel in (0.3, 0.5):
        s = cloud(reg.transform_points(src0, M @ T_rec)).voxel_down_sample(voxel)
        t = cloud(tgt0).voxel_down_sample(voxel)
        for c, up in ((s, M[:3, :3] @ np.array([0.0, 0.0, 1.0])), (t, np.array([0.0, 0.0, 1.0]))):
            c.estimate_normals(30, 0.8)
            n = c.point["normals"].t                   # oriented to the vertical, as a user does before FPFH
            sign = torch.where(n.double() @ torch.from_numpy(up).cuda() < 0, -1.0, 1.0).to(n.dtype)[:, None]
            c.point["normals"] = o3d.Tensor((n * sign).contiguous())
        fs, ft = o3dreg.compute_fpfh_feature(s, 100, 1.5), o3dreg.compute_fpfh_feature(t, 100, 1.5)
        ctx = o3d.get_context(max(s._n(), t._n()))
        xs, xt = s._xyzi(), t._xyzi()
        fs, ft = fs.t.contiguous(), ft.t.contiguous()
        for tuple_test in (True, False):
            run = lambda: ctx.fgr_from_features(xs, xt, fs, ft, tuple_test=tuple_test)
            T, info, _ = run()
            ctx.check()
            info = info.cpu().numpy()
            dt, ang = pose_error(T.cpu().numpy(), T_true)
            per, launches = profiled(ctx, run)
            us = call_us(run)
            match = per.get("k_feat_nn", 0.0)
            res["cases"].append(dict(voxel=voxel, n_src=s._n(), n_tgt=t._n(), tuple_test=tuple_test,
                                     pairs_in=int(info[1]), pairs_used=int(info[2]), trials=int(info[4]),
                                     iterations=int(info[0]), status=int(info[3]), error_m=round(dt, 4),
                                     error_deg=round(ang, 3), call_us=us, matching_us=match,
                                     fgr_us=round(sum(v for k, v in per.items() if k != "k_feat_nn"), 1),
                                     kernels_us=per, launches=launches, launches_per_call=sum(launches.values())))
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

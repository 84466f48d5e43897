"""Cost of the large neighbourhood sizes (the *_wide kernels: k > 64, max_nn > 32) next to the sizes below, on one GPU:
eager pipeline runs with every kernel bracketed by CUDA events (``ctx.profile(True)``).

* statistical outlier removal on the C4 scan (1.5 M points, 0.05 m voxels), k in {20, 33, 48, 64, 65, 100, 256, 1024};
* normal estimation on the reference's default configuration (262 144-point scan, duplicate removal,
  non-finite filter, ROI crop, 0.01 m voxels, radius 0.1 m), max_nn in {30, 33, 48, 64, 65, 100, 256}.

Per configuration: one warm-up run, then RUNS profiled runs; the JSON holds the mean time per launch of
every kernel of the stage and the stage total, with the GPU's name and power limit.
Usage: python profiles/wide_neighbors.py [out.json]   (default profiles/wide_neighbors.json)"""
import json, os, subprocess, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from autodriver_pointcloud_preprocessor_b200 import _capi, engine, synth

RUNS = 10
STAT_KERNELS = ("k_grid_insert", "k_grid_assign", "k_grid_scatter", "k_knn_query", "k_knn_stragglers", "k_knn_query_wide",
                "k_knn_stragglers_wide", "k_grid_clean", "stat_reduce_mask")
NRM_KERNELS = ("k_normals_cov", "k_normals_wide", "k_normals_eigen")


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "not available"
    return dict(gpu=name, power_limit_and_max_sm_clock=q)


def profile_stage(ctx, desc, pcfg, kernels):
    ctx.pipeline_run_maps([desc], pcfg)                                  # warm-up (allocations, module load)
    ctx.check()
    ctx.profile(True)
    for _ in range(RUNS):
        _, counts, _, _ = ctx.pipeline_run_maps([desc], pcfg)          # (maps: the normals' destination)
    rep = ctx.profile_report()
    ctx.profile(False)
    ctx.check()
    per = {k: round(ms / n * 1e3, 1) for k, (ms, n) in rep.items() if k in kernels}
    c = counts.cpu().numpy()
    return dict(kernels_us=per, stage_us=round(sum(per.values()), 1), counts={
        "input": int(c[_capi.CNT_INPUT]), "voxels": int(c[_capi.CNT_VOXELS]), "after_stat": int(c[_capi.CNT_AFTER_STAT]),
        "output": int(c[_capi.CNT_OUTPUT])})


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "wide_neighbors.json")
    res = dict(gpu_info(), runs_per_config=RUNS, statistical=[], normals=[])
    # C4, as bench.py builds it
    m = synth.pack_cloud(synth.lidar_scan(seed=500, n_beams=128, n_az=2048, n_points=1_500_000), "xyzi16")
    ctx = engine.Context(max_points=m.width)
    desc = engine.make_cloud_desc(m.fields, m.point_step, m.width, torch.frombuffer(bytearray(m.data), dtype=torch.uint8).cuda())
    for k in (20, 33, 48, 64, 65, 100, 256, 1024):
        pcfg = engine.make_pipeline_cfg(engine.make_filter_cfg(skip_nans=True, remove_nan=True, remove_inf=True), voxel_size=0.05,
                                        statistical=dict(nb_neighbors=k, std_ratio=2.0))
        r = dict(k=k, **profile_stage(ctx, desc, pcfg, STAT_KERNELS))
        print("statistical", json.dumps(r), flush=True)
        res["statistical"].append(r)
    ctx.close()
    # the reference's default parameter set (profiles/default_cfg.py)
    m = bench.make_frames(1, seed0=3)[0]
    ctx = engine.Context(max_points=m.width)
    desc = engine.make_cloud_desc(m.fields, m.point_step, m.width, torch.frombuffer(bytearray(m.data), dtype=torch.uint8).cuda())
    fcfg = engine.make_filter_cfg(skip_nans=True, dedup_mode=_capi.DEDUP_OPEN3D, remove_nan=True, remove_inf=True, crop=bench.CROP)
    for nn in (30, 33, 48, 64, 65, 100, 256):
        pcfg = engine.make_pipeline_cfg(fcfg, voxel_size=0.01, normals=dict(radius=0.1, max_nn=nn))
        r = dict(max_nn=nn, **profile_stage(ctx, desc, pcfg, NRM_KERNELS))
        print("normals", json.dumps(r), flush=True)
        res["normals"].append(r)
    ctx.close()
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()

"""``open3d.t.pipelines.registration`` look-alike: single-scale ICP and ``evaluate_registration`` on the GPU.

The whole ICP loop runs on the device (``apc_icp``): the call synchronises once, at the end.  Definitions, and
where they differ from Open3D, are in ``oracle/registration.py``; in short:

* every iteration transforms the original source by the float64 transform accumulated so far and rounds to
  float32 (Open3D re-transforms its float32 cloud in place);
* a source point's correspondence is the nearest target point by the float32 squared distance with ties to the
  lower index, kept when ``d2 <= float32(max_correspondence_distance)^2`` (Open3D: ``d2 < r^2``);
* point-to-plane stops with ``RuntimeError`` when its 6x6 system is not positive definite (every normal parallel,
  for example), where Open3D would solve it anyway.

Not modelled: multi-scale ICP, colored / generalized ICP, robust kernels and per-iteration callbacks.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _capi
from .geometry import PointCloud, Tensor, get_context

_NO_CORRESPONDENCE = ("0 correspondence present between the pointclouds. Try increasing the "
                      "max_correspondence_distance parameter.")


class TransformationEstimationPointToPoint:
    """Kabsch (no scaling) over the correspondences."""
    method = _capi.APC_ICP_POINT_TO_POINT

    def __repr__(self):
        return "TransformationEstimationPointToPoint"


class TransformationEstimationPointToPlane:
    """One Gauss-Newton step of ``sum ((s' - t) . n_t)^2`` per iteration; needs the target's ``normals``."""
    method = _capi.APC_ICP_POINT_TO_PLANE

    def __repr__(self):
        return "TransformationEstimationPointToPlane"


class ICPConvergenceCriteria:
    def __init__(self, relative_fitness=1e-6, relative_rmse=1e-6, max_iteration=30):
        self.relative_fitness = float(relative_fitness)
        self.relative_rmse = float(relative_rmse)
        self.max_iteration = int(max_iteration)

    def __repr__(self):
        return (f"ICPConvergenceCriteria(relative_fitness={self.relative_fitness}, "
                f"relative_rmse={self.relative_rmse}, max_iteration={self.max_iteration})")


class RegistrationResult:
    """``transformation``: float64 4x4 ``Tensor`` on the CPU (as Open3D returns it); ``correspondences_``: int64
    ``Tensor`` [n_source] on the source's device, -1 where a source point has no correspondence."""

    def __init__(self, transformation, correspondences, fitness, inlier_rmse, converged=False, num_iterations=0):
        self.transformation = transformation
        self.correspondences_ = correspondences
        self.fitness = fitness
        self.inlier_rmse = inlier_rmse
        self.converged = converged
        self.num_iterations = num_iterations

    def __repr__(self):
        return (f"RegistrationResult[fitness={self.fitness:.6e}, inlier_rmse={self.inlier_rmse:.6e}, "
                f"converged={self.converged}, num_iterations={self.num_iterations}]")


def _transform(T) -> np.ndarray:
    if T is None:
        return np.eye(4)
    if isinstance(T, Tensor):
        T = T.t
    if isinstance(T, torch.Tensor):
        T = T.detach().cpu().numpy()
    T = np.asarray(T, dtype=np.float64)
    if T.shape != (4, 4):
        raise ValueError(f"the transformation must be 4x4, got {T.shape}")
    return T


def _check_distance(r):
    if not (math.isfinite(r) and r > 0):
        raise ValueError("max_correspondence_distance must be finite and > 0")


def _result(source: PointCloud, T, stats, corr, info=None) -> RegistrationResult:
    stats = stats.cpu().numpy()
    return RegistrationResult(Tensor(torch.from_numpy(np.array(T, np.float64))), source._home(corr.to(torch.int64)),
                              float(stats[0]), float(stats[1]),
                              bool(info[1]) if info is not None else False, int(info[0]) if info is not None else 0)


def evaluate_registration(source: PointCloud, target: PointCloud, max_correspondence_distance,
                          transformation=None) -> RegistrationResult:
    """Open3D ``evaluate_registration``: fitness, inlier rmse and correspondences of ``source`` moved by
    ``transformation`` (identity by default) against ``target``."""
    _check_distance(max_correspondence_distance)
    T = _transform(transformation)
    n_src, n_tgt = source._n(), target._n()
    if n_src == 0 or n_tgt == 0:
        corr = torch.full((n_src,), -1, dtype=torch.int64, device="cuda")
        return RegistrationResult(Tensor(torch.from_numpy(T.copy())), source._home(corr), 0.0, 0.0)
    ctx = get_context(max(n_src, n_tgt), source.device.index if source.device.kind == "CUDA" else None)
    stats, corr, _ = ctx.evaluate_registration(source._xyzi(), target._xyzi(), float(max_correspondence_distance), T)
    ctx.check()
    return _result(source, T, stats, corr)


def icp(source: PointCloud, target: PointCloud, max_correspondence_distance, init_source_to_target=None,
        estimation_method=None, criteria=None, voxel_size=-1.0, callback_after_iteration=None) -> RegistrationResult:
    """Open3D ``icp`` (single scale).  ``voxel_size > 0`` downsamples both clouds first, as Open3D does.  Raises
    ``RuntimeError`` when an iteration finds no correspondence, when point-to-plane runs on a target without
    ``normals`` or its system is degenerate, and ``NotImplementedError`` for ``callback_after_iteration`` (the
    loop never returns to the host)."""
    if callback_after_iteration is not None:
        raise NotImplementedError("callback_after_iteration: the ICP loop runs on the GPU without visiting the host")
    _check_distance(max_correspondence_distance)
    estimation = estimation_method if estimation_method is not None else TransformationEstimationPointToPoint()
    crit = criteria if criteria is not None else ICPConvergenceCriteria()
    if crit.max_iteration < 0:
        raise ValueError("max_iteration must be >= 0")
    T0 = _transform(init_source_to_target)
    if voxel_size > 0:
        source, target = source.voxel_down_sample(voxel_size), target.voxel_down_sample(voxel_size)
    point_to_plane = estimation.method == _capi.APC_ICP_POINT_TO_PLANE
    if point_to_plane and "normals" not in target.point:
        raise RuntimeError("TransformationEstimationPointToPlane requires pre-computed normals for the target "
                           "PointCloud")
    n_src, n_tgt = source._n(), target._n()
    if n_src == 0 or n_tgt == 0:
        raise RuntimeError("Source and/or Target pointcloud is empty.")
    ctx = get_context(max(n_src, n_tgt), source.device.index if source.device.kind == "CUDA" else None)
    normals = None
    if point_to_plane:
        normals = PointCloud._gpu(target.point["normals"]).to(torch.float32).contiguous()
    T, stats, info, corr = ctx.icp(source._xyzi(), target._xyzi(), float(max_correspondence_distance), T0,
                                   estimation.method, normals, crit.max_iteration, crit.relative_fitness,
                                   crit.relative_rmse)
    ctx.check()                                   # the one synchronisation of the call
    info = info.cpu().numpy()
    if info[2] == _capi.APC_ICP_NO_CORRESPONDENCE:
        raise RuntimeError(_NO_CORRESPONDENCE)
    if info[2] == _capi.APC_ICP_DEGENERATE:
        raise RuntimeError("point-to-plane ICP: the linear system is not positive definite (degenerate geometry, "
                           "e.g. all target normals parallel)")
    return _result(source, T.cpu().numpy(), stats, corr, info)

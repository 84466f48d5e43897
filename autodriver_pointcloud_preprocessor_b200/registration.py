"""``open3d.t.pipelines.registration`` look-alike: single-scale ICP (point-to-point, point-to-plane, generalized),
``evaluate_registration``, FPFH features (``compute_fpfh_feature``), matching in feature space
(``correspondences_from_features``) and Fast Global Registration (``registration_fgr_based_on_feature_matching``,
``registration_fgr_based_on_correspondence``) on the GPU.

The whole ICP loop runs on the device (``apc_icp``): the call synchronises once, at the end.  Definitions, and
where they differ from Open3D, are in ``oracle/registration.py`` and ``oracle/gicp.py``; in short:

* every iteration transforms the original source by the float64 transform accumulated so far and rounds to
  float32 (Open3D re-transforms its float32 cloud in place);
* a source point's correspondence is the nearest target point by the float32 squared distance with ties to the
  lower index, kept when ``d2 <= float32(max_correspondence_distance)^2`` (Open3D: ``d2 < r^2``);
* point-to-plane and generalized ICP stop with ``RuntimeError`` when their 6x6 system is not positive definite (every
  normal parallel, for example), where Open3D would solve it anyway;
* generalized ICP takes only each covariance's axis of least variance, and regularises it as Segal et al. do
  (``I - (1 - epsilon) a a^T``).  An isotropic covariance has no such axis: the identity that neighbourhoods of
  fewer than 3 points get is treated as a horizontal plane.

FPFH and feature matching (``oracle/features.py``):

* the neighbourhoods are those of ``estimate_normals``: hybrid (``max_nn`` and ``radius``) or KNN (``max_nn``
  only); radius-only search and ``indices=`` are not modelled.  Open3D's pair features and 3 x 11 bins; a pair
  whose feature is not finite (a NaN normal) adds to no bin.  The swap test of the pair feature compares ``|a1| <
  |a2|`` where Open3D compares their ``acos``; the SPFH multiplies each count by ``100 / (m - 1)`` once, and the
  FPFH sums in a fixed order, so results can differ from Open3D's in the last float32 bits;
* a feature row's match is the other set's row with the smallest float32 squared distance, ties to the lower
  index; rows whose distances are all NaN have no match and no pair.  The search is brute force,
  O(n_source * n_target * 33).

Fast Global Registration (``oracle/fgr.py``, Zhou, Park and Koltun 2016):

* the feature entry starts from the mutual set of the feature matching, with no ratio fallback;
* the tuple test draws its triples from a counter-based stream seeded with ``option.seed`` (0 when None), where
  Open3D uses its own random generator: results are reproducible but not Open3D's draws;
* the transform accumulates and the original target is transformed every iteration (Open3D moves its copy of the
  target in place); fewer than 10 pairs after the tuple test warn and return the identity.

Not modelled: multi-scale ICP, colored ICP, robust kernels, per-iteration callbacks and RANSAC global registration.
"""
from __future__ import annotations

import math
import warnings

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


class TransformationEstimationForGeneralizedICP:
    """Generalized ICP (Segal et al. 2009, plane-to-plane): one Gauss-Newton step of ``sum e^T W e`` per iteration,
    ``W = (R C_s R^T + C_t)^-1`` from the regularised covariances of both clouds (``point['covariances']``, or
    estimated with :meth:`PointCloud.estimate_covariances` defaults when a cloud has none).  ``epsilon`` is the
    variance kept along each covariance's axis of least variance."""
    method = _capi.APC_ICP_GENERALIZED

    def __init__(self, epsilon=1e-3, kernel=None):
        if kernel is not None:
            raise NotImplementedError("robust kernels are not modelled")
        epsilon = float(epsilon)
        if not (math.isfinite(epsilon) and epsilon > 0):
            raise ValueError("epsilon must be finite and > 0")
        self.epsilon = epsilon
        self.kernel = None

    def __repr__(self):
        return f"TransformationEstimationForGeneralizedICP(epsilon={self.epsilon})"


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


def _covariances(cloud: PointCloud) -> torch.Tensor:
    """float32 ``[n, 3, 3]`` on the GPU: the cloud's ``covariances``, or ``estimate_covariances()`` of its positions
    (the cloud itself is not modified)."""
    if "covariances" not in cloud.point:
        cov = cloud._like({"positions": cloud.point["positions"]}).estimate_covariances().point["covariances"]
    else:
        cov = cloud.point["covariances"]
    cov = PointCloud._gpu(cov).to(torch.float32).contiguous()
    if tuple(cov.shape) != (cloud._n(), 3, 3):
        raise ValueError(f"covariances must be [{cloud._n()}, 3, 3], got {tuple(cov.shape)}")
    return cov


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
    ``normals`` or its system (or generalized ICP's) is degenerate, and ``NotImplementedError`` for
    ``callback_after_iteration`` (the loop never returns to the host).

    Generalized ICP uses each cloud's ``covariances`` when present and otherwise estimates them with
    ``estimate_covariances()`` defaults; the caller's clouds are not modified.  With ``voxel_size > 0`` they are
    always estimated on the downsampled clouds: a voxel mean of covariances keeps at most 20 fractional bits
    (about 1e-6), the size of a planar neighbourhood's smallest eigenvalue, so averaged covariances lose their
    planes."""
    if callback_after_iteration is not None:
        raise NotImplementedError("callback_after_iteration: the ICP loop runs on the GPU without visiting the host")
    _check_distance(max_correspondence_distance)
    estimation = estimation_method if estimation_method is not None else TransformationEstimationPointToPoint()
    crit = criteria if criteria is not None else ICPConvergenceCriteria()
    if crit.max_iteration < 0:
        raise ValueError("max_iteration must be >= 0")
    T0 = _transform(init_source_to_target)
    generalized = estimation.method == _capi.APC_ICP_GENERALIZED
    if voxel_size > 0:
        if generalized:                          # not carried: estimated on the downsampled clouds below
            source, target = (c._like({k: v for k, v in c.point.items() if k != "covariances"}) for c in (source, target))
        source, target = source.voxel_down_sample(voxel_size), target.voxel_down_sample(voxel_size)
    point_to_plane = estimation.method == _capi.APC_ICP_POINT_TO_PLANE
    if point_to_plane and "normals" not in target.point:
        raise RuntimeError("TransformationEstimationPointToPlane requires pre-computed normals for the target "
                           "PointCloud")
    n_src, n_tgt = source._n(), target._n()
    if n_src == 0 or n_tgt == 0:
        raise RuntimeError("Source and/or Target pointcloud is empty.")
    ctx = get_context(max(n_src, n_tgt), source.device.index if source.device.kind == "CUDA" else None)
    if generalized:
        src_cov, tgt_cov = _covariances(source), _covariances(target)
        T, stats, info, corr = ctx.icp_generalized(source._xyzi(), src_cov, target._xyzi(), tgt_cov,
                                                   float(max_correspondence_distance), T0, estimation.epsilon,
                                                   crit.max_iteration, crit.relative_fitness, crit.relative_rmse)
    else:
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
        raise RuntimeError(f"{'generalized' if generalized else 'point-to-plane'} ICP: the linear system is not "
                           "positive definite (degenerate geometry, e.g. all target normals parallel)")
    return _result(source, T.cpu().numpy(), stats, corr, info)


def compute_fpfh_feature(input: PointCloud, max_nn=100, radius=None, indices=None) -> Tensor:
    """Open3D ``compute_fpfh_feature``: float32 ``Tensor [N, 33]`` on the cloud's device.  ``max_nn`` with ``radius``
    is the hybrid search (the ``max_nn`` nearest within ``radius``), ``max_nn`` alone the KNN search; the cloud needs
    ``normals``.  Raises ``RuntimeError`` without normals and ``NotImplementedError`` for a radius-only search or
    ``indices``."""
    if indices is not None:
        raise NotImplementedError("compute_fpfh_feature: indices= is not modelled")
    if max_nn is None:
        raise NotImplementedError("compute_fpfh_feature: the radius-only search is not modelled; pass max_nn")
    if "normals" not in input.point:
        raise RuntimeError("compute_fpfh_feature requires normals: call estimate_normals() first")
    n = input._n()
    if n == 0:
        return input._home(torch.zeros((0, 33), dtype=torch.float32, device="cuda"))
    normals = PointCloud._gpu(input.point["normals"]).to(torch.float32).contiguous()
    if tuple(normals.shape) != (n, 3):
        raise ValueError(f"normals must be [{n}, 3], got {tuple(normals.shape)}")
    feat, _, _ = input._ctx().compute_fpfh(input._xyzi(), normals, int(max_nn),
                                           None if radius is None else float(radius))
    return input._home(feat.contiguous())


def correspondences_from_features(source_features, target_features, mutual_filter=False,
                                  mutual_consistency_ratio=0.1) -> Tensor:
    """Open3D ``correspondences_from_features``: int64 ``Tensor [K, 2]`` of ``(source row, target row)`` pairs in
    ascending source row, each source row with its nearest target row in feature space.  With ``mutual_filter``
    only the pairs whose target row's nearest source row is the source row itself are kept, unless there are no
    more than ``mutual_consistency_ratio * n_source`` of them: then the unfiltered pairs are returned with a
    warning, as Open3D does.  Source rows without a finite distance (NaN features) have no pair."""
    src = source_features.t if isinstance(source_features, Tensor) else torch.as_tensor(source_features)
    tgt = target_features.t if isinstance(target_features, Tensor) else torch.as_tensor(target_features)
    if src.dim() != 2 or tgt.dim() != 2 or src.shape[1] != tgt.shape[1]:
        raise ValueError(f"features must be [n, dim] with the same dim, got {tuple(src.shape)} and {tuple(tgt.shape)}")
    ratio = float(mutual_consistency_ratio)
    if not (math.isfinite(ratio) and ratio >= 0):
        raise ValueError("mutual_consistency_ratio must be finite and >= 0")
    on_cuda = src.is_cuda
    dev = src.device.index if on_cuda else None
    home = (lambda t: Tensor(t)) if on_cuda else (lambda t: Tensor(t.cpu()))
    if src.shape[0] == 0 or tgt.shape[0] == 0:
        return home(torch.zeros((0, 2), dtype=torch.int64, device="cuda"))
    ctx = get_context(max(src.shape[0], tgt.shape[0]), dev)
    src = (src if src.is_cuda else src.cuda(ctx.device)).to(torch.float32).contiguous()
    tgt = (tgt if tgt.is_cuda else tgt.cuda(ctx.device)).to(torch.float32).contiguous()
    pairs, info, _ = ctx.correspondences_from_features(src, tgt, bool(mutual_filter), ratio)
    count, fell_back = (int(v) for v in info.cpu().tolist())      # the one synchronisation of the call
    if fell_back:
        warnings.warn("Too few correspondences after mutual filter, fall back to original correspondences.",
                      RuntimeWarning, stacklevel=2)
    return home(pairs[:count].to(torch.int64))


class FastGlobalRegistrationOption:
    """Open3D's ``FastGlobalRegistrationOption``.  ``seed`` (None means 0) seeds the tuple test's draws."""

    def __init__(self, division_factor=1.4, use_absolute_scale=False, decrease_mu=True,
                 maximum_correspondence_distance=0.025, iteration_number=64, tuple_scale=0.95,
                 maximum_tuple_count=1000, tuple_test=True, seed=None):
        self.division_factor = float(division_factor)
        self.use_absolute_scale = bool(use_absolute_scale)
        self.decrease_mu = bool(decrease_mu)
        self.maximum_correspondence_distance = float(maximum_correspondence_distance)
        self.iteration_number = int(iteration_number)
        self.tuple_scale = float(tuple_scale)
        self.maximum_tuple_count = int(maximum_tuple_count)
        self.tuple_test = bool(tuple_test)
        self.seed = None if seed is None else int(seed)
        if not (math.isfinite(self.division_factor) and self.division_factor > 1):
            raise ValueError("division_factor must be finite and > 1")
        if not (math.isfinite(self.maximum_correspondence_distance) and self.maximum_correspondence_distance > 0):
            raise ValueError("maximum_correspondence_distance must be finite and > 0")
        if self.iteration_number < 0:
            raise ValueError("iteration_number must be >= 0")
        if not (0 < self.tuple_scale <= 1):
            raise ValueError("tuple_scale must be in (0, 1]")
        if self.maximum_tuple_count < 1:
            raise ValueError("maximum_tuple_count must be >= 1")

    def __repr__(self):
        return (f"FastGlobalRegistrationOption(division_factor={self.division_factor}, "
                f"use_absolute_scale={self.use_absolute_scale}, decrease_mu={self.decrease_mu}, "
                f"maximum_correspondence_distance={self.maximum_correspondence_distance}, "
                f"iteration_number={self.iteration_number}, tuple_scale={self.tuple_scale}, "
                f"maximum_tuple_count={self.maximum_tuple_count}, tuple_test={self.tuple_test}, seed={self.seed})")


def _fgr_result(source: PointCloud, T, info) -> RegistrationResult:
    """The one synchronisation of an FGR call: status, warning or error, and the result."""
    info = info.cpu().numpy()
    if info[3] == _capi.APC_FGR_TOO_FEW:
        warnings.warn(f"Fast Global Registration: only {int(info[2])} correspondences (fewer than 10), returning the "
                      "identity.", RuntimeWarning, stacklevel=3)
    if info[3] == _capi.APC_FGR_DEGENERATE:
        raise RuntimeError("Fast Global Registration: the linear system is not positive definite (degenerate or "
                           "non-finite correspondences)")
    corr = torch.full((source._n(),), -1, dtype=torch.int64, device="cuda")
    return RegistrationResult(Tensor(T.cpu()), source._home(corr), 0.0, 0.0, False, int(info[0]))


def _fgr_clouds(source: PointCloud, target: PointCloud):
    n_src, n_tgt = source._n(), target._n()
    ctx = get_context(max(n_src, n_tgt, 1), source.device.index if source.device.kind == "CUDA" else None)
    return ctx, source._xyzi(), target._xyzi()


def registration_fgr_based_on_feature_matching(source: PointCloud, target: PointCloud, source_feature, target_feature,
                                               option=None) -> RegistrationResult:
    """Open3D ``registration_fgr_based_on_feature_matching``: Fast Global Registration (Zhou, Park and Koltun 2016)
    of ``source`` onto ``target`` from their features (``[n, dim]``, as :func:`compute_fpfh_feature` returns them).
    The pairs are the mutual nearest neighbours in feature space, filtered by the tuple test.  The result carries
    only the transformation (float64, CPU) and ``num_iterations``: ``fitness = inlier_rmse = 0`` and every
    correspondence is -1, as in Open3D.  Warns and returns the identity with fewer than 10 pairs; raises
    ``RuntimeError`` when the linear system is degenerate."""
    opt = option if option is not None else FastGlobalRegistrationOption()
    fs = source_feature.t if isinstance(source_feature, Tensor) else torch.as_tensor(source_feature)
    ft = target_feature.t if isinstance(target_feature, Tensor) else torch.as_tensor(target_feature)
    if fs.dim() != 2 or ft.dim() != 2 or fs.shape[1] != ft.shape[1]:
        raise ValueError(f"features must be [n, dim] with the same dim, got {tuple(fs.shape)} and {tuple(ft.shape)}")
    if fs.shape[0] != source._n() or ft.shape[0] != target._n():
        raise ValueError(f"features have {fs.shape[0]} and {ft.shape[0]} rows for clouds of {source._n()} and "
                         f"{target._n()} points")
    ctx, src, tgt = _fgr_clouds(source, target)
    fs = (fs if fs.is_cuda else fs.cuda(ctx.device)).to(torch.float32).contiguous()
    ft = (ft if ft.is_cuda else ft.cuda(ctx.device)).to(torch.float32).contiguous()
    T, info, _ = ctx.fgr_from_features(src, tgt, fs, ft, opt.division_factor, opt.use_absolute_scale, opt.decrease_mu,
                                       opt.maximum_correspondence_distance, opt.iteration_number, opt.tuple_scale,
                                       opt.maximum_tuple_count, opt.tuple_test, 0 if opt.seed is None else opt.seed)
    ctx.check()
    return _fgr_result(source, T, info)


def registration_fgr_based_on_correspondence(source: PointCloud, target: PointCloud, corres,
                                             option=None) -> RegistrationResult:
    """Open3D ``registration_fgr_based_on_correspondence``: Fast Global Registration on the given ``(source index,
    target index)`` pairs (int64 ``[K, 2]``, as :func:`correspondences_from_features` returns them), without the
    tuple test.  Raises ``ValueError`` for an index outside its cloud; otherwise as
    :func:`registration_fgr_based_on_feature_matching`."""
    opt = option if option is not None else FastGlobalRegistrationOption()
    c = corres.t if isinstance(corres, Tensor) else torch.as_tensor(corres)
    if c.dim() != 2 or c.shape[1] != 2:
        raise ValueError(f"corres must be [K, 2], got {tuple(c.shape)}")
    c = c.to(torch.int64)
    if c.shape[0] and (bool((c < 0).any()) or int(c[:, 0].max()) >= source._n() or int(c[:, 1].max()) >= target._n()):
        raise ValueError("corres holds an index outside its point cloud")
    ctx, src, tgt = _fgr_clouds(source, target)
    pairs = c.to(device=ctx.device, dtype=torch.int32).contiguous()
    T, info, _ = ctx.fgr(src, tgt, pairs, opt.division_factor, opt.use_absolute_scale, opt.decrease_mu,
                         opt.maximum_correspondence_distance, opt.iteration_number)
    ctx.check()
    return _fgr_result(source, T, info)

"""Host-side driver of the C-ABI library: contexts, descriptors and stage calls.

torch is used only as the carrier of device memory and streams; every computation goes
through ``libapc.so`` (``_capi``).  Functions here take/return torch CUDA tensors.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _capi
from ._capi import (ApcError, CloudDesc, Field, FilterCfg, OutField, PipelineCfg, lib)

VENDOR_INTENSITY = ["I", "intensity"]   # utils.py:42
_DT_SIZE = {1: 1, 2: 1, 3: 2, 4: 2, 5: 4, 6: 4, 7: 4, 8: 8}
_TORCH_TO_APC = {torch.int8: 1, torch.uint8: 2, torch.int16: 3, torch.uint16: 4, torch.int32: 5,
                 torch.uint32: 6, torch.float32: 7, torch.float64: 8}


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _t16(T):
    """A 4x4 transform as the ``double[16]`` (row-major) of the C ABI; identity when None."""
    v = np.eye(4) if T is None else np.asarray(T.cpu() if isinstance(T, torch.Tensor) else T, np.float64)
    if v.shape != (4, 4):
        raise ValueError("the transformation must be 4x4")
    return (C.c_double * 16)(*v.reshape(16).tolist())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def make_cloud_desc(fields, point_step: int, n_points: int, data_dev: torch.Tensor | None,
                    field_names=None, transform=None) -> CloudDesc:
    """Descriptor of one PointCloud2 buffer.

    ``fields``: iterable of objects with ``name/offset/datatype/count`` (PointField).
    ``field_names``: optional subset passed to ``read_points`` (utils.py:208) - it restricts
    the fields the NaN skip looks at.  The intensity field is resolved with the reference's
    vendor aliases (utils.py:41-48, last matching alias wins, utils.py:434-438).
    """
    by_name = {f.name: f for f in fields}
    selected = [f for f in fields if field_names is None or f.name in field_names]
    lower = [f.name.lower() for f in selected]
    d = CloudDesc()
    d.data_dev = data_dev.data_ptr() if data_dev is not None else None
    d.n_points = n_points
    d.point_step = point_step
    for axis in "xyz":
        if axis not in by_name:
            raise ValueError("Incoming PointCloud does not have x, y, z fields.")   # pp.py:413-415
        f = by_name[axis]
        setattr(d, axis, Field(f.offset, f.datatype))
    d.intensity = Field(0, 0)
    name = None
    for option in VENDOR_INTENSITY:
        if option.lower() in lower:
            name = option
    if name is not None and name in by_name:
        f = by_name[name]
        d.intensity = Field(f.offset, f.datatype)
    nan_fields = []
    for f in selected:
        for a in range(max(1, f.count)):
            nan_fields.append(Field(f.offset + a * _DT_SIZE[f.datatype], f.datatype))
    nan_fields = [f for f in nan_fields if f.datatype in (7, 8)]     # integer fields are never NaN
    if len(nan_fields) > _capi.APC_MAX_FIELDS:
        raise ValueError("too many floating-point fields")
    d.n_nan_fields = len(nan_fields)
    for i, f in enumerate(nan_fields):
        d.nan_fields[i] = f
    if transform is not None:
        d.has_transform = 1
        T = np.asarray(transform, dtype=np.float32).reshape(16)
        for i in range(16):
            d.transform[i] = float(T[i])
    d._keep_alive = data_dev            # the struct holds a raw device pointer: keep the tensor alive with it
    return d


def make_filter_cfg(skip_nans=False, dedup_mode=_capi.DEDUP_OFF, remove_nan=False, remove_inf=False,
                    transforms=(), crop=None) -> FilterCfg:
    cfg = FilterCfg()
    cfg.skip_nans, cfg.dedup_mode = int(bool(skip_nans)), int(dedup_mode)
    cfg.remove_nan, cfg.remove_inf = int(bool(remove_nan)), int(bool(remove_inf))
    transforms = list(transforms)
    if len(transforms) > _capi.APC_MAX_TRANSFORMS:
        raise ValueError("at most 3 transforms")
    cfg.n_transforms = len(transforms)
    for k, T in enumerate(transforms):
        T = np.asarray(T, dtype=np.float32).reshape(16)      # float64 -> float32 like pp.py:757
        for i in range(16):
            cfg.transforms[k][i] = float(T[i])
    if crop is not None:
        cfg.crop_enable = 1
        cfg.crop_mode = int(crop.get("mode", _capi.CROP_OPEN3D))
        cfg.crop_invert = int(bool(crop.get("invert", False)))
        for i in range(3):
            cfg.roi_min[i] = float(crop["min"][i])
            cfg.roi_max[i] = float(crop["max"][i])
    return cfg


class Context:
    """One device context (scratch + hash tables) bound to a GPU; not thread-safe."""

    def __init__(self, max_points: int, device: int | None = None):
        if not torch.cuda.is_available():
            raise RuntimeError("CUDA device required: this package has no CPU path")
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.max_points = int(max_points)
        h = C.c_void_p()
        rc = lib.apc_ctx_create(self.device_index, self.max_points, C.byref(h))
        if rc != 0:
            raise ApcError(rc, (lib.apc_last_error(None) or b"apc_ctx_create failed").decode())
        self.h = h
        self._graphs = []

    def close(self):
        if getattr(self, "h", None):
            for g in self._graphs:
                lib.apc_graph_destroy(g)
            self._graphs = []
            lib.apc_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ok(self, rc):
        _capi.check(self.h, rc)

    def set_low_latency(self, on: bool = True):
        """One scan in flight at a time: launch the per-scan kernels as programmatic dependents
        (``apc_ctx_set_low_latency``)."""
        self._ok(lib.apc_ctx_set_low_latency(self.h, int(bool(on))))

    def check(self):
        """Synchronise and raise on data-dependent device errors (key range / capacity)."""
        self._ok(lib.apc_check(self.h, _stream()))

    def profile(self, on: bool):
        """Bracket every eagerly launched kernel with CUDA events (see apc_profile_enable)."""
        self._ok(lib.apc_profile_enable(self.h, int(bool(on))))

    def profile_report(self) -> dict:
        """``{kernel: (total_ms, launches)}`` since the last report; synchronises the device."""
        buf = C.create_string_buffer(16384)
        n = lib.apc_profile_report(self.h, buf, len(buf))
        if n < 0:
            self._ok(n)
        out = {}
        for line in buf.value.decode().splitlines():
            name, ms, cnt = line.split()
            out[name] = (float(ms), int(cnt))
        return out

    def _empty(self, shape, dtype):
        return torch.empty(shape, dtype=dtype, device=self.device)

    # ---- front end ---------------------------------------------------------------------------
    def frontend(self, clouds, cfg: FilterCfg, want_src=True, want_stage=False):
        """Returns ``(xyzi[N,4], src_idx[N] | None, stage[N] | None, count[1])`` (device)."""
        n_total = sum(c.n_points for c in clouds)
        arr = (CloudDesc * len(clouds))(*clouds)
        xyzi = self._empty((max(n_total, 1), 4), torch.float32)
        src = self._empty((max(n_total, 1),), torch.int32) if want_src else None
        stage = torch.zeros((max(n_total, 1),), dtype=torch.uint8, device=self.device) if want_stage else None
        cnt = torch.zeros((1,), dtype=torch.int32, device=self.device)
        self._ok(lib.apc_frontend(self.h, arr, len(clouds), C.byref(cfg), _ptr(xyzi), _ptr(src), _ptr(stage),
                                  _ptr(cnt), _stream()))
        return xyzi, src, stage, cnt

    def unpack(self, cloud: CloudDesc):
        xyzi = self._empty((max(cloud.n_points, 1), 4), torch.float32)
        self._ok(lib.apc_unpack(self.h, C.byref(cloud), _ptr(xyzi), _stream()))
        return xyzi[:cloud.n_points]

    def transform(self, xyzi, T, out=None, n_dev=None):
        out = torch.empty_like(xyzi) if out is None else out
        T16 = (C.c_float * 16)(*np.asarray(T, dtype=np.float32).reshape(16).tolist())
        self._ok(lib.apc_transform(self.h, _ptr(xyzi), xyzi.shape[0], _ptr(n_dev), T16, _ptr(out), _stream()))
        return out

    def crop_mask(self, xyzi, min_bound, max_bound, mode=_capi.CROP_OPEN3D, invert=False):
        mask = self._empty((xyzi.shape[0],), torch.uint8)
        lo = (C.c_double * 3)(*[float(v) for v in min_bound])
        hi = (C.c_double * 3)(*[float(v) for v in max_bound])
        self._ok(lib.apc_crop_mask(self.h, _ptr(xyzi), xyzi.shape[0], None, lo, hi, int(mode), int(bool(invert)),
                                   _ptr(mask), _stream()))
        return mask

    def non_finite_mask(self, xyzi, remove_nan=True, remove_infinite=True):
        mask = self._empty((xyzi.shape[0],), torch.uint8)
        self._ok(lib.apc_non_finite_mask(self.h, _ptr(xyzi), xyzi.shape[0], None, int(bool(remove_nan)),
                                         int(bool(remove_infinite)), _ptr(mask), _stream()))
        return mask

    def duplicate_mask(self, xyzi):
        mask = self._empty((xyzi.shape[0],), torch.uint8)
        self._ok(lib.apc_duplicate_mask(self.h, _ptr(xyzi), xyzi.shape[0], None, _ptr(mask), _stream()))
        return mask

    def unique_rows(self, xyzi, want_first=True, want_inverse=False, n_dev=None):
        """``np.unique(positions, axis=0, return_index=True, return_inverse=True)`` on the device.
        Returns ``(first_idx int32[n] | None, inverse int32[n] | None, count[1])``; the first
        ``int(count)`` entries of ``first_idx`` are valid."""
        n = xyzi.shape[0]
        first = self._empty((max(n, 1),), torch.int32) if want_first else None
        inverse = self._empty((max(n, 1),), torch.int32) if want_inverse else None
        cnt = torch.zeros((1,), dtype=torch.int32, device=self.device)
        self._ok(lib.apc_unique_rows(self.h, _ptr(xyzi), n, _ptr(n_dev), _ptr(first), _ptr(inverse), _ptr(cnt),
                                     _stream()))
        return first, inverse, cnt

    def select_by_mask(self, xyzi, mask, invert=False, want_idx=True):
        """Order-preserving compaction.  Returns ``(xyzi_out, idx, count)`` with full-size
        buffers; slice with ``int(count)``."""
        n = mask.shape[0]
        out = self._empty((max(n, 1), 4), torch.float32) if xyzi is not None else None
        idx = self._empty((max(n, 1),), torch.int32) if want_idx else None
        cnt = torch.zeros((1,), dtype=torch.int32, device=self.device)
        self._ok(lib.apc_select_by_mask(self.h, _ptr(xyzi), n, None, _ptr(mask), int(bool(invert)), _ptr(out),
                                        _ptr(idx), _ptr(cnt), _stream()))
        return out, idx, cnt

    def gather(self, src, idx, n=None):
        n = idx.shape[0] if n is None else n
        src = src.contiguous()
        elem = src.element_size() * (int(np.prod(src.shape[1:])) if src.dim() > 1 else 1)
        out = torch.empty((n,) + tuple(src.shape[1:]), dtype=src.dtype, device=self.device)
        self._ok(lib.apc_gather(self.h, _ptr(src), elem, _ptr(idx), n, None, _ptr(out), _stream()))
        return out

    def pack_xyzi(self, pos3, intensity=None):
        """positions float32[N,3] (+ float32[N] intensity) -> SoA float4[N]."""
        n = pos3.shape[0]
        out = self._empty((max(n, 1), 4), torch.float32)
        self._ok(lib.apc_pack_xyzi(self.h, _ptr(pos3), _ptr(intensity), n, _ptr(out), _stream()))
        return out[:n]

    def split_xyzi(self, xyzi, n=None, want_intensity=True):
        """SoA float4 -> (positions float32[n,3], intensity float32[n] | None)."""
        n = xyzi.shape[0] if n is None else int(n)
        pos = self._empty((max(n, 1), 3), torch.float32)
        inten = self._empty((max(n, 1),), torch.float32) if want_intensity else None
        self._ok(lib.apc_split_xyzi(self.h, _ptr(xyzi), n, None, _ptr(pos), _ptr(inten), _stream()))
        return pos[:n], (inten[:n] if inten is not None else None)

    # ---- voxel ---------------------------------------------------------------------------------
    def voxel_downsample(self, xyzi, voxel_size, want_p2v=False, want_counts=False, n_dev=None):
        n = xyzi.shape[0]
        out = self._empty((max(n, 1), 4), torch.float32)
        p2v = self._empty((max(n, 1),), torch.int32) if want_p2v else None
        vc = self._empty((max(n, 1),), torch.int32) if want_counts else None
        cnt = torch.zeros((1,), dtype=torch.int32, device=self.device)
        self._ok(lib.apc_voxel_downsample(self.h, _ptr(xyzi), n, _ptr(n_dev), float(voxel_size), _ptr(out),
                                          _ptr(p2v), _ptr(vc), _ptr(cnt), _stream()))
        return out, p2v, vc, cnt

    def voxel_downsample_sorted(self, xyzi, voxel_size, want_counts=False, n_dev=None):
        """The sort-based voxel grid (``apc_voxel_downsample_sorted``): same voxels / counts / centroids as
        :meth:`voxel_downsample`, rows in ascending (ix, iy, iz) order."""
        n = xyzi.shape[0]
        out = self._empty((max(n, 1), 4), torch.float32)
        vc = self._empty((max(n, 1),), torch.int32) if want_counts else None
        cnt = torch.zeros((1,), dtype=torch.int32, device=self.device)
        self._ok(lib.apc_voxel_downsample_sorted(self.h, _ptr(xyzi), n, _ptr(n_dev), float(voxel_size), _ptr(out),
                                                 _ptr(vc), _ptr(cnt), _stream()))
        return out, vc, cnt

    def voxel_mean_attr(self, attr_f32, p2v, n_voxels_dev, n_vox_max, frac_bits: int = 20):
        """Order-independent voxel mean of one float32 attribute column (``apc_voxel_mean_attr``);
        ``frac_bits`` from :func:`attr_frac_bits` of the attribute's own dtype."""
        out = self._empty((max(n_vox_max, 1),), torch.float32)
        self._ok(lib.apc_voxel_mean_attr(self.h, _ptr(attr_f32), _ptr(p2v), attr_f32.shape[0], None,
                                         _ptr(n_voxels_dev), int(frac_bits), _ptr(out), _stream()))
        return out

    # ---- outliers --------------------------------------------------------------------------------
    def radius_outliers(self, xyzi, nb_points, radius, want_counts=False, n_dev=None):
        n = xyzi.shape[0]
        mask = self._empty((max(n, 1),), torch.uint8)
        counts = self._empty((max(n, 1),), torch.int32) if want_counts else None
        self._ok(lib.apc_radius_outliers(self.h, _ptr(xyzi), n, _ptr(n_dev), int(nb_points), float(radius),
                                         _ptr(mask), _ptr(counts), _stream()))
        return mask[:n], (counts[:n] if counts is not None else None)

    def statistical_outliers(self, xyzi, nb_neighbors, std_ratio, n_dev=None):
        n = xyzi.shape[0]
        mask = self._empty((max(n, 1),), torch.uint8)
        avg = self._empty((max(n, 1),), torch.float32)
        stats = torch.zeros((3,), dtype=torch.float64, device=self.device)
        self._ok(lib.apc_statistical_outliers(self.h, _ptr(xyzi), n, _ptr(n_dev), int(nb_neighbors),
                                              float(std_ratio), _ptr(mask), _ptr(avg), _ptr(stats), _stream()))
        return mask[:n], avg[:n], stats

    def estimate_normals(self, xyzi, max_nn, radius, want_counts=False, want_cov=False, n_dev=None):
        """Returns ``(normals float32[n,3], counts int32[n] | None, covariances float64[n,3,3] | None)``."""
        n = xyzi.shape[0]
        normals = self._empty((max(n, 1), 3), torch.float32)
        counts = self._empty((max(n, 1),), torch.int32) if want_counts else None
        cov = self._empty((max(n, 1), 3, 3), torch.float64) if want_cov else None
        self._ok(lib.apc_estimate_normals(self.h, _ptr(xyzi), n, _ptr(n_dev), int(max_nn), float(radius),
                                          _ptr(normals), _ptr(counts), _ptr(cov), _stream()))
        return normals[:n], (counts[:n] if counts is not None else None), (cov[:n] if cov is not None else None)

    def estimate_normals_knn(self, xyzi, max_nn, want_counts=False, want_cov=False, n_dev=None):
        """KNN search (``apc_estimate_normals_knn``): the ``max_nn`` nearest points, no distance bound.
        Returns the same tuple as :meth:`estimate_normals`."""
        return self._normals_search(lib.apc_estimate_normals_knn, xyzi, int(max_nn), want_counts, want_cov, n_dev)

    def estimate_normals_radius(self, xyzi, radius, want_counts=False, want_cov=False, n_dev=None):
        """Radius search (``apc_estimate_normals_radius``): every point within ``radius``, no cap on the count.
        Returns the same tuple as :meth:`estimate_normals`."""
        return self._normals_search(lib.apc_estimate_normals_radius, xyzi, float(radius), want_counts, want_cov, n_dev)

    def _normals_search(self, fn, xyzi, bound, want_counts, want_cov, n_dev):
        n = xyzi.shape[0]
        normals = self._empty((max(n, 1), 3), torch.float32)
        counts = self._empty((max(n, 1),), torch.int32) if want_counts else None
        cov = self._empty((max(n, 1), 3, 3), torch.float64) if want_cov else None
        self._ok(fn(self.h, _ptr(xyzi), n, _ptr(n_dev), bound, _ptr(normals), _ptr(counts), _ptr(cov), _stream()))
        return normals[:n], (counts[:n] if counts is not None else None), (cov[:n] if cov is not None else None)

    # ---- clustering ----------------------------------------------------------------------------------
    def cluster_dbscan(self, xyzi, eps, min_points, want_counts=False, n_dev=None):
        """DBSCAN (``apc_cluster_dbscan``).  Returns ``(labels int32[n], n_clusters int32[1] (device),
        counts int32[n] | None)``; label -1 = noise."""
        n = xyzi.shape[0]
        labels = self._empty((max(n, 1),), torch.int32)
        n_clusters = torch.zeros((1,), dtype=torch.int32, device=self.device)
        counts = self._empty((max(n, 1),), torch.int32) if want_counts else None
        self._ok(lib.apc_cluster_dbscan(self.h, _ptr(xyzi), n, _ptr(n_dev), float(eps), int(min_points), _ptr(labels),
                                        _ptr(n_clusters), _ptr(counts), _stream()))
        return labels[:n], n_clusters, (counts[:n] if counts is not None else None)

    # ---- registration ---------------------------------------------------------------------------------
    def evaluate_registration(self, src_xyzi, tgt_xyzi, max_correspondence_distance, T=None, n_src_dev=None,
                              n_tgt_dev=None):
        """``apc_evaluate_registration`` at ``T`` (float64 4x4, identity by default).  Returns ``(stats float64[2]
        {fitness, inlier_rmse}, correspondences int32[n_src] (-1: none), d2 float32[n_src])`` on the device."""
        n_src, n_tgt = src_xyzi.shape[0], tgt_xyzi.shape[0]
        corr = self._empty((max(n_src, 1),), torch.int32)
        d2 = self._empty((max(n_src, 1),), torch.float32)
        stats = self._empty((2,), torch.float64)
        self._ok(lib.apc_evaluate_registration(self.h, _ptr(src_xyzi), n_src, _ptr(n_src_dev), _ptr(tgt_xyzi), n_tgt,
                                               _ptr(n_tgt_dev), float(max_correspondence_distance), _t16(T),
                                               _ptr(corr), _ptr(d2), _ptr(stats), _stream()))
        return stats, corr[:n_src], d2[:n_src]

    def icp(self, src_xyzi, tgt_xyzi, max_correspondence_distance, init=None, method=_capi.APC_ICP_POINT_TO_POINT,
            tgt_normals=None, max_iteration=30, relative_fitness=1e-6, relative_rmse=1e-6, n_src_dev=None,
            n_tgt_dev=None):
        """``apc_icp``.  Returns ``(T float64[4,4], stats float64[2] {fitness, inlier_rmse}, info int32[4]
        {iterations, converged, APC_ICP_* status, 0}, correspondences int32[n_src])`` on the device, with no host
        synchronisation."""
        n_src, n_tgt = src_xyzi.shape[0], tgt_xyzi.shape[0]
        T = self._empty((4, 4), torch.float64)
        stats = self._empty((2,), torch.float64)
        info = self._empty((4,), torch.int32)
        corr = self._empty((max(n_src, 1),), torch.int32)
        self._ok(lib.apc_icp(self.h, _ptr(src_xyzi), n_src, _ptr(n_src_dev), _ptr(tgt_xyzi), _ptr(tgt_normals), n_tgt,
                             _ptr(n_tgt_dev), float(max_correspondence_distance), _t16(init), int(method),
                             int(max_iteration), float(relative_fitness), float(relative_rmse), _ptr(T), _ptr(stats),
                             _ptr(info), _ptr(corr), _stream()))
        return T, stats, info, corr[:n_src]

    def icp_generalized(self, src_xyzi, src_cov, tgt_xyzi, tgt_cov, max_correspondence_distance, init=None,
                        epsilon=1e-3, max_iteration=30, relative_fitness=1e-6, relative_rmse=1e-6, want_axes=False,
                        n_src_dev=None, n_tgt_dev=None):
        """``apc_icp_generalized`` with float32 covariances ``[n, 3, 3]`` (contiguous, on the device).  Returns the
        tuple of :meth:`icp`, plus the regularisation axes ``(float64[n_src, 3], float64[n_tgt, 3])`` when
        ``want_axes``; no host synchronisation."""
        n_src, n_tgt = src_xyzi.shape[0], tgt_xyzi.shape[0]
        T = self._empty((4, 4), torch.float64)
        stats = self._empty((2,), torch.float64)
        info = self._empty((4,), torch.int32)
        corr = self._empty((max(n_src, 1),), torch.int32)
        axes_s = self._empty((max(n_src, 1), 3), torch.float64) if want_axes else None
        axes_t = self._empty((max(n_tgt, 1), 3), torch.float64) if want_axes else None
        self._ok(lib.apc_icp_generalized(self.h, _ptr(src_xyzi), _ptr(src_cov), n_src, _ptr(n_src_dev), _ptr(tgt_xyzi),
                                         _ptr(tgt_cov), n_tgt, _ptr(n_tgt_dev), float(max_correspondence_distance),
                                         _t16(init), float(epsilon), int(max_iteration), float(relative_fitness),
                                         float(relative_rmse), _ptr(T), _ptr(stats), _ptr(info), _ptr(corr),
                                         _ptr(axes_s), _ptr(axes_t), _stream()))
        out = (T, stats, info, corr[:n_src])
        return out + (axes_s[:n_src], axes_t[:n_tgt]) if want_axes else out

    # ---- features --------------------------------------------------------------------------------------
    def compute_fpfh(self, xyzi, normals, max_nn, radius=None, want_spfh=False, want_counts=False, n_dev=None):
        """FPFH of every point (``apc_compute_fpfh``: hybrid search, or ``apc_compute_fpfh_knn`` when ``radius`` is
        None).  ``normals`` float32 ``[n, 3]`` contiguous on the device.  Returns ``(features float32[n, 33],
        spfh float32[n, 33] | None, counts int32[n] | None)``; no host synchronisation."""
        n = xyzi.shape[0]
        feat = self._empty((max(n, 1), 33), torch.float32)
        spfh = self._empty((max(n, 1), 33), torch.float32) if want_spfh else None
        counts = self._empty((max(n, 1),), torch.int32) if want_counts else None
        if radius is None:
            rc = lib.apc_compute_fpfh_knn(self.h, _ptr(xyzi), _ptr(normals), n, _ptr(n_dev), int(max_nn), _ptr(feat),
                                          _ptr(spfh), _ptr(counts), _stream())
        else:
            rc = lib.apc_compute_fpfh(self.h, _ptr(xyzi), _ptr(normals), n, _ptr(n_dev), int(max_nn), float(radius),
                                      _ptr(feat), _ptr(spfh), _ptr(counts), _stream())
        self._ok(rc)
        return feat[:n], (spfh[:n] if spfh is not None else None), (counts[:n] if counts is not None else None)

    def correspondences_from_features(self, src, tgt, mutual_filter=False, mutual_consistency_ratio=0.1,
                                      want_nearest=False, n_src_dev=None, n_tgt_dev=None):
        """``apc_correspondences_from_features`` on float32 ``[n, dim]`` rows (contiguous, on the device).  Returns
        ``(pairs int32[n_src, 2], info int32[2] {count, fell_back}, nearest int32[n_src] | None)`` on the device;
        the first ``count`` rows of ``pairs`` are valid.  No host synchronisation."""
        n_src, n_tgt = src.shape[0], tgt.shape[0]
        dim = src.shape[1] if src.dim() == 2 else 0
        pairs = self._empty((max(n_src, 1), 2), torch.int32)
        info = self._empty((2,), torch.int32)
        nearest = self._empty((max(n_src, 1),), torch.int32) if want_nearest else None
        self._ok(lib.apc_correspondences_from_features(self.h, _ptr(src), n_src, _ptr(n_src_dev), _ptr(tgt), n_tgt,
                                                       _ptr(n_tgt_dev), int(dim), int(bool(mutual_filter)),
                                                       float(mutual_consistency_ratio), _ptr(pairs), _ptr(nearest),
                                                       _ptr(info), _stream()))
        return pairs[:n_src], info, (nearest[:n_src] if nearest is not None else None)

    def fgr_from_features(self, src_xyzi, tgt_xyzi, src_feat, tgt_feat, division_factor=1.4, use_absolute_scale=False,
                          decrease_mu=True, maximum_correspondence_distance=0.025, iteration_number=64,
                          tuple_scale=0.95, maximum_tuple_count=1000, tuple_test=True, seed=0, n_src_dev=None,
                          n_tgt_dev=None):
        """``apc_fgr_from_features`` on xyzi clouds and float32 ``[n, dim]`` feature rows (contiguous, on the device).
        Returns ``(T float64[4,4], info int32[6] {iterations, pairs in, pairs used, APC_FGR_* status, trials, pairs
        dropped}, pairs_used int32[cap, 2])`` on the device, with no host synchronisation; the first ``pairs used``
        rows of ``pairs_used`` are valid."""
        n_src, n_tgt = src_xyzi.shape[0], tgt_xyzi.shape[0]
        dim = src_feat.shape[1] if src_feat.dim() == 2 else 0
        T = self._empty((4, 4), torch.float64)
        info = self._empty((6,), torch.int32)
        cap = 3 * min(max(int(maximum_tuple_count), 1), self.max_points) if tuple_test else n_src   # larger: rejected
        used = self._empty((max(cap, 1), 2), torch.int32)
        self._ok(lib.apc_fgr_from_features(self.h, _ptr(src_xyzi), n_src, _ptr(n_src_dev), _ptr(tgt_xyzi), n_tgt,
                                           _ptr(n_tgt_dev), _ptr(src_feat), _ptr(tgt_feat), int(dim),
                                           float(division_factor), int(bool(use_absolute_scale)),
                                           int(bool(decrease_mu)), float(maximum_correspondence_distance),
                                           int(iteration_number), float(tuple_scale), int(maximum_tuple_count),
                                           int(bool(tuple_test)), int(seed) & 0xFFFFFFFFFFFFFFFF, _ptr(T), _ptr(info),
                                           _ptr(used), _stream()))
        return T, info, used

    def fgr(self, src_xyzi, tgt_xyzi, pairs, division_factor=1.4, use_absolute_scale=False, decrease_mu=True,
            maximum_correspondence_distance=0.025, iteration_number=64, n_src_dev=None, n_tgt_dev=None,
            n_pairs_dev=None):
        """``apc_fgr`` on int32 ``[K, 2]`` pairs (contiguous, on the device).  Returns the tuple of
        :meth:`fgr_from_features` (``pairs_used`` int32[K, 2]); no host synchronisation."""
        n_src, n_tgt, n_pairs = src_xyzi.shape[0], tgt_xyzi.shape[0], pairs.shape[0]
        T = self._empty((4, 4), torch.float64)
        info = self._empty((6,), torch.int32)
        used = self._empty((max(n_pairs, 1), 2), torch.int32)
        self._ok(lib.apc_fgr(self.h, _ptr(src_xyzi), n_src, _ptr(n_src_dev), _ptr(tgt_xyzi), n_tgt, _ptr(n_tgt_dev),
                             _ptr(pairs), n_pairs, _ptr(n_pairs_dev), float(division_factor),
                             int(bool(use_absolute_scale)), int(bool(decrease_mu)),
                             float(maximum_correspondence_distance), int(iteration_number), _ptr(T), _ptr(info),
                             _ptr(used), _stream()))
        return T, info, used

    # ---- ransac ------------------------------------------------------------------------------------
    def segment_plane(self, xyzi, distance_threshold, ransac_n, num_iterations, probability, seed=0,
                      sample_table=None, n_dev=None):
        """Returns ``(plane8 float64[8], inlier_mask uint8[n], info int32[4])`` (device)."""
        n = xyzi.shape[0]
        plane = torch.zeros((8,), dtype=torch.float64, device=self.device)
        mask = torch.zeros((max(n, 1),), dtype=torch.uint8, device=self.device)
        info = torch.zeros((4,), dtype=torch.int32, device=self.device)
        tab = None
        if sample_table is not None:
            tab = torch.as_tensor(np.ascontiguousarray(sample_table, dtype=np.int32)).to(self.device)
        self._ok(lib.apc_segment_plane(self.h, _ptr(xyzi), n, _ptr(n_dev), float(distance_threshold), int(ransac_n),
                                       int(num_iterations), float(probability), C.c_uint64(int(seed)), _ptr(tab),
                                       _ptr(plane), _ptr(mask), _ptr(info), _stream()))
        return plane, mask[:n], info

    def segment_plane_scores(self, num_iterations):
        """``uint64[num_iterations, 2]`` = (inlier count, integer error sum) per hypothesis of the
        most recent ``segment_plane`` / pipeline call (device tensor, viewed as int64)."""
        out = torch.zeros((int(num_iterations), 2), dtype=torch.int64, device=self.device)
        self._ok(lib.apc_segment_plane_scores(self.h, _ptr(out), int(num_iterations), _stream()))
        return out

    # ---- repack --------------------------------------------------------------------------------------
    def repack(self, xyzi, out_fields, point_step, n_dev=None):
        """``out_fields``: list of ``(offset, datatype, source, attr_tensor | None)``."""
        n = xyzi.shape[0]
        arr = (OutField * len(out_fields))()
        keep = []
        for i, (off, dt, src, attr) in enumerate(out_fields):
            arr[i].offset, arr[i].datatype, arr[i].source = int(off), int(dt), int(src)
            if attr is not None:
                attr = attr.contiguous()
                keep.append(attr)
                arr[i].attr_dev = attr.data_ptr()
                arr[i].attr_datatype = _TORCH_TO_APC[attr.dtype]
        out = self._empty((max(n, 1) * point_step,), torch.uint8)
        self._ok(lib.apc_repack(self.h, _ptr(xyzi), n, _ptr(n_dev), arr, len(out_fields), int(point_step),
                                _ptr(out), _stream()))
        return out

    # ---- pipeline ------------------------------------------------------------------------------------
    def pipeline_run(self, clouds, pcfg: PipelineCfg, out_xyzi=None, out_counts=None, out_plane=None):
        n_total = sum(c.n_points for c in clouds)
        arr = (CloudDesc * len(clouds))(*clouds)
        out_xyzi = self._empty((max(n_total, 1), 4), torch.float32) if out_xyzi is None else out_xyzi
        out_counts = torch.zeros((8,), dtype=torch.int32, device=self.device) if out_counts is None else out_counts
        out_plane = torch.zeros((8,), dtype=torch.float64, device=self.device) if out_plane is None else out_plane
        self._ok(lib.apc_pipeline_run(self.h, arr, len(clouds), C.byref(pcfg), _ptr(out_xyzi), _ptr(out_counts),
                                      _ptr(out_plane), _stream()))
        return out_xyzi, out_counts, out_plane

    def pipeline_run_maps(self, clouds, pcfg: PipelineCfg):
        """preprocess() plus the index maps that let the caller carry any other attribute through it
        (``apc_pipeline_run_maps``).  Returns ``(out_xyzi, counts, plane, maps)`` with ``maps`` a dict
        of device tensors ``src_idx`` / ``p2v`` / ``voxel_counts`` / ``out_row`` (int32, full size;
        valid lengths are in ``counts``)."""
        n_total = sum(c.n_points for c in clouds)
        arr = (CloudDesc * len(clouds))(*clouds)
        out_xyzi = self._empty((max(n_total, 1), 4), torch.float32)
        out_counts = torch.zeros((8,), dtype=torch.int32, device=self.device)
        out_plane = torch.zeros((8,), dtype=torch.float64, device=self.device)
        maps = {k: self._empty((max(n_total, 1),), torch.int32) for k in ("src_idx", "p2v", "voxel_counts", "out_row")}
        if pcfg.normals_enable:
            maps["normals"] = self._empty((max(n_total, 1), 3), torch.float32)
        m = make_pipeline_maps(maps)
        self._ok(lib.apc_pipeline_run_maps(self.h, arr, len(clouds), C.byref(pcfg), _ptr(out_xyzi), _ptr(out_counts),
                                           _ptr(out_plane), C.byref(m), _stream()))
        return out_xyzi, out_counts, out_plane, maps

    def capture_pipeline(self, clouds, pcfg: PipelineCfg, out_xyzi, out_counts, out_plane, mirror=None, maps=None):
        """Capture the pipeline over fixed buffers into a CUDA graph; returns a handle for
        :meth:`launch_graph`.  ``mirror``: an ``OutMirror`` from :func:`make_out_mirror` - the final
        stage then also stores its rows / counters into the peers' buffers (``apc_out_mirror``).
        ``maps``: dict of device tensors (``src_idx`` / ``p2v`` / ``voxel_counts`` / ``out_row`` /
        ``normals``) the replay fills; ``normals`` is required when the config enables normals."""
        arr = (CloudDesc * len(clouds))(*clouds)
        g = C.c_void_p()
        m = make_pipeline_maps(maps) if maps is not None else None
        self._ok(lib.apc_graph_capture_pipeline_ex(self.h, arr, len(clouds), C.byref(pcfg), _ptr(out_xyzi),
                                                   _ptr(out_counts), _ptr(out_plane),
                                                   C.byref(m) if m is not None else None,
                                                   C.byref(mirror) if mirror is not None else None, C.byref(g)))
        self._graphs.append(g)
        return g

    def pipeline_run_mirrored(self, clouds, pcfg: PipelineCfg, out_xyzi, out_counts, out_plane, mirror):
        arr = (CloudDesc * len(clouds))(*clouds)
        self._ok(lib.apc_pipeline_run_mirrored(self.h, arr, len(clouds), C.byref(pcfg), _ptr(out_xyzi), _ptr(out_counts),
                                               _ptr(out_plane), C.byref(mirror), _stream()))
        return out_xyzi, out_counts, out_plane

    def launch_graph(self, g):
        self._ok(lib.apc_graph_launch(self.h, g, _stream()))


def attr_frac_bits(col: torch.Tensor) -> int:
    """Fractional bits of the fixed-point voxel mean for an attribute column of dtype ``col.dtype``:
    0 for integer attributes (exact sums), else as many as keep ``|v| * 2^bits`` below 2^39 (at most 20)."""
    if not col.dtype.is_floating_point:
        return 0
    big = float(col.abs().nan_to_num(0.0, 0.0, 0.0).max().item()) if col.numel() else 0.0
    bits = 20
    while bits > 0 and big * (1 << bits) >= 2.0 ** 39:
        bits -= 1
    return bits


def make_pipeline_maps(maps: dict) -> "_capi.PipelineMaps":
    """``apc_pipeline_maps`` from a dict of device tensors (missing keys = NULL)."""
    def p(k):
        t = maps.get(k)
        return t.data_ptr() if t is not None else None
    m = _capi.PipelineMaps(p("src_idx"), p("p2v"), p("voxel_counts"), p("out_row"), p("normals"))
    m._keep_alive = maps
    return m


def make_out_mirror(xyzi_ptrs=(), counts_ptrs=(), multicast: bool = False) -> "_capi.OutMirror":
    """``apc_out_mirror`` from raw device addresses (peer-mapped buffers of the other GPUs, or one NVLS
    multicast address with ``multicast=True``).  The caller keeps the mapped tensors alive."""
    m = _capi.OutMirror()
    xyzi_ptrs, counts_ptrs = list(xyzi_ptrs), list(counts_ptrs)
    if len(xyzi_ptrs) > _capi.APC_MAX_MIRRORS or len(counts_ptrs) > _capi.APC_MAX_MIRRORS:
        raise ValueError("at most 8 mirrors")
    m.n_xyzi, m.xyzi_multicast, m.n_counts = len(xyzi_ptrs), int(bool(multicast)), len(counts_ptrs)
    for i, p in enumerate(xyzi_ptrs):
        m.xyzi_dev[i] = int(p)
    for i, p in enumerate(counts_ptrs):
        m.counts_dev[i] = int(p)
    return m


def make_pipeline_cfg(filter_cfg: FilterCfg, voxel_size=0.0, statistical=None, radius=None, ground=None,
                      normals=None) -> PipelineCfg:
    p = PipelineCfg()
    p.filter = filter_cfg
    p.voxel_size = float(voxel_size or 0.0)
    if statistical:
        p.stat_enable, p.stat_nb_neighbors = 1, int(statistical["nb_neighbors"])
        p.stat_std_ratio = float(statistical["std_ratio"])
    if radius:
        p.radius_enable, p.radius_nb_points = 1, int(radius["nb_points"])
        p.radius_search_radius = float(radius["radius"])
    if ground:
        p.ground_enable = 1
        p.ground_distance_threshold = float(ground["distance_threshold"])
        p.ground_ransac_n = int(ground["ransac_n"])
        p.ground_num_iterations = int(ground["num_iterations"])
        p.ground_probability = float(ground["probability"])
        p.ground_seed = int(ground.get("seed", 0))
    if normals:
        p.normals_enable, p.normals_max_nn = 1, int(normals["max_nn"])
        p.normals_radius = float(normals["radius"])
    return p

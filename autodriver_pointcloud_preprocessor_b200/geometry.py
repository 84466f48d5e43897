"""Open3D-shaped carriers (``Tensor``, ``PointCloud``, ``AxisAlignedBoundingBox``) backed by
the CUDA library.

The reference drives everything through ``open3d.t.geometry.PointCloud`` and
``open3d.core.Tensor`` (``pp.py:309,421-443,466-543``, ``utils.py:135-137,255-299,521-544``).
These classes expose exactly the surface those call sites touch (SURVEY.md section 8b), so the
node and the ``utils`` functions read like the reference's, while every operation runs in
``libapc.so`` on the GPU.  torch tensors are the storage; torch itself is only used to move
or cast buffers.

A cloud whose ``device`` is ``CPU:0`` keeps its tensors on the host (as Open3D would) and
stages them through the GPU for each operation; there is no CPU implementation.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _capi, engine

# ---- devices / dtypes ----------------------------------------------------------------------------


class Device:
    """``o3d.core.Device`` look-alike: ``Device('CPU:0')`` / ``Device('CUDA:0')``."""

    def __init__(self, spec="CPU:0"):
        spec = str(spec)
        kind, _, idx = spec.partition(":")
        self.kind = "CUDA" if kind.upper() in ("CUDA", "GPU") else "CPU"
        self.index = int(idx) if idx else 0

    def __str__(self):
        return f"{self.kind}:{self.index}"

    __repr__ = __str__

    def __eq__(self, other):
        return str(self) == str(Device(other) if not isinstance(other, Device) else other)

    def __hash__(self):
        return hash(str(self))

    @property
    def torch(self) -> torch.device:
        return torch.device("cuda", self.index) if self.kind == "CUDA" else torch.device("cpu")


class Dtype:
    Float32, Float64 = torch.float32, torch.float64
    Int8, Int16, Int32, Int64 = torch.int8, torch.int16, torch.int32, torch.int64
    UInt8, UInt16, UInt32 = torch.uint8, torch.uint16, torch.uint32
    Bool = torch.bool


float32, float64, int32, int64, uint8, uint16, bool8 = (Dtype.Float32, Dtype.Float64, Dtype.Int32, Dtype.Int64,
                                                        Dtype.UInt8, Dtype.UInt16, Dtype.Bool)


class Tensor:
    """``o3c.Tensor`` look-alike over a torch tensor."""

    Dtype = Dtype

    def __init__(self, data, dtype=None, device=None):
        if isinstance(data, Tensor):
            t = data.t
        elif isinstance(data, torch.Tensor):
            t = data
        else:
            t = torch.as_tensor(np.asarray(data))
        if dtype is not None:
            t = t.to(dtype)
        if device is not None:
            t = t.to(Device(device).torch)
        self.t = t

    # -- construction (utils.py:234,271,294; pp.py:426-431,777-782)
    @staticmethod
    def from_numpy(a):
        return Tensor(torch.from_numpy(np.ascontiguousarray(a)) if not a.flags.writeable or not a.flags.c_contiguous
                      else torch.from_numpy(a))

    @staticmethod
    def from_dlpack(capsule):
        return Tensor(torch.utils.dlpack.from_dlpack(capsule))

    def to_dlpack(self):
        return torch.utils.dlpack.to_dlpack(self.t)

    # -- placement
    @property
    def is_cpu(self):
        return not self.t.is_cuda

    @property
    def is_cuda(self):
        return self.t.is_cuda

    @property
    def device(self):
        return Device(f"CUDA:{self.t.device.index or 0}") if self.t.is_cuda else Device("CPU:0")

    def cpu(self):
        return Tensor(self.t.cpu())

    def cuda(self, index=0):
        return Tensor(self.t.cuda(index))

    def to(self, target, copy=False):
        if isinstance(target, torch.dtype):
            return Tensor(self.t.to(target))
        if isinstance(target, (Device, str)):
            return Tensor(self.t.to(Device(target).torch))
        raise TypeError(f"cannot convert Tensor to {target!r}")

    def numpy(self):
        if self.t.is_cuda:
            raise RuntimeError("Tensor is on CUDA; call .cpu() first (same rule as Open3D)")
        return self.t.numpy()

    def clone(self):
        return Tensor(self.t.clone())

    # -- shape
    @property
    def shape(self):
        return tuple(self.t.shape)

    @property
    def dtype(self):
        return self.t.dtype

    def reshape(self, *shape):
        return Tensor(self.t.reshape(*shape))

    def __len__(self):
        return self.t.shape[0]

    def __getitem__(self, key):
        return Tensor(self.t[key.t if isinstance(key, Tensor) else key])

    def item(self):
        return self.t.item()

    def __repr__(self):
        return f"Tensor(shape={self.shape}, dtype={self.dtype}, device={self.device})"


class AxisAlignedBoundingBox:
    """``o3d.t.geometry.AxisAlignedBoundingBox`` (pp.py:311-313): float32 bounds."""

    def __init__(self, min_bound, max_bound):
        self.min_bound = Tensor(min_bound).to(Dtype.Float32)
        self.max_bound = Tensor(max_bound).to(Dtype.Float32)

    def to(self, device):
        return self


class TensorMap(dict):
    """``pcd.point``: dict of attribute tensors with attribute-style access."""

    def __setitem__(self, key, value):
        super().__setitem__(key, value if isinstance(value, Tensor) else Tensor(value))

    def __getattr__(self, key):
        try:
            return self[key]
        except KeyError as e:
            raise AttributeError(key) from e

    def __setattr__(self, key, value):
        self[key] = value


# ---- contexts ----------------------------------------------------------------------------------------

_CONTEXTS: dict = {}
MAX_CONTEXT_POINTS = 1 << 22         # apc_ctx_create's limit


def get_context(n_points: int, device_index: int | None = None) -> engine.Context:
    """Shared per-device apc context, grown (recreated) when a larger cloud arrives."""
    idx = torch.cuda.current_device() if device_index is None else device_index
    ctx = _CONTEXTS.get(idx)
    need = max(int(n_points), 1)
    if need > MAX_CONTEXT_POINTS:          # refuse before touching the shared context (INTEGRATION.md: parameter caps)
        raise ValueError(f"clouds of more than {MAX_CONTEXT_POINTS} points are not supported ({need} requested)")
    if ctx is None or ctx.max_points < need:
        cap = 1 << 16
        while cap < need:
            cap <<= 1
        if ctx is not None:
            ctx.close()
        ctx = engine.Context(max_points=min(cap, MAX_CONTEXT_POINTS), device=idx)
        ctx.set_low_latency(True)          # the node and the utils functions run one call at a time (pp.py:1056)
        _CONTEXTS[idx] = ctx
    return ctx


class PointCloud:
    """``o3d.t.geometry.PointCloud`` look-alike (the surface listed in SURVEY.md section 8b)."""

    def __init__(self, arg=None):
        self.point = TensorMap()
        self.device = Device("CPU:0")
        if isinstance(arg, (Device, str)):
            self.device = Device(arg)
        elif isinstance(arg, dict):                       # utils.py:136 t.PointCloud(dict)
            for k, v in arg.items():
                if v is None or k == "header":
                    continue
                self.point[k] = v
            if "positions" in self.point:
                self.device = self.point["positions"].device
        elif arg is not None:
            raise TypeError("PointCloud(arg): arg must be a device, a dict of tensors or None")

    # -- housekeeping
    def clear(self):                                      # pp.py:421
        self.point.clear()
        return self

    def is_empty(self):
        return "positions" not in self.point or len(self.point["positions"]) == 0

    def to(self, device):                                 # utils.py:136
        out = PointCloud(Device(device))
        for k, v in self.point.items():
            out.point[k] = v.to(Device(device))
        return out

    def cpu(self):
        return self.to("CPU:0")

    def cuda(self, index=0):
        return self.to(f"CUDA:{index}")

    def clone(self):
        out = PointCloud(self.device)
        for k, v in self.point.items():
            out.point[k] = v.clone()
        return out

    def to_legacy(self):                                  # pp.py:367 (visualiser only)
        raise NotImplementedError("legacy Open3D geometry (visualisation) is outside the CUDA hot path")

    def estimate_normals(self, max_nn=30, radius=None):   # pp.py:523
        """Open3D ``estimate_normals``: neighbourhood search -> covariance -> eigenvector of the
        smallest eigenvalue; sets ``point['normals']`` (float32 N x 3), not oriented.  The search
        follows the arguments, as in Open3D:

        * both given (the reference's call, pp.py:523-526): hybrid, the ``max_nn`` nearest within ``radius``;
        * ``max_nn`` only (the default call ``estimate_normals()``): KNN, the ``max_nn`` nearest;
        * ``radius`` only (``max_nn=None``): every point within ``radius``, no cap on the count;
        * neither: ``ValueError``.

        ``max_nn`` in 1..``APC_MAX_NEIGHBORS`` (1024) and ``radius`` finite and > 0; otherwise the call
        raises ``ApcError``."""
        if radius is None and max_nn is None:
            raise ValueError("estimate_normals needs max_nn, radius or both")
        if self._n() == 0:
            self.point["normals"] = self._home(torch.zeros((0, 3), dtype=torch.float32, device="cuda"))
            return self
        if radius is None:
            normals, _, _ = self._ctx().estimate_normals_knn(self._xyzi(), int(max_nn))
        elif max_nn is None:
            normals, _, _ = self._ctx().estimate_normals_radius(self._xyzi(), float(radius))
        else:
            normals, _, _ = self._ctx().estimate_normals(self._xyzi(), int(max_nn), float(radius))
        self.point["normals"] = self._home(normals.contiguous())
        return self

    def __repr__(self):
        n = 0 if self.is_empty() else len(self.point["positions"])
        return f"PointCloud on {self.device} [{n} points] attributes: {sorted(k for k in self.point if k != 'positions')}"

    # -- internals
    def _n(self):
        return 0 if "positions" not in self.point else len(self.point["positions"])

    def _ctx(self) -> engine.Context:
        return get_context(self._n(), self.device.index if self.device.kind == "CUDA" else None)

    @staticmethod
    def _gpu(t: Tensor) -> torch.Tensor:
        x = t.t
        return (x if x.is_cuda else x.cuda()).contiguous()

    def _xyzi(self):
        """SoA float4 view of positions (+ intensity when present) on the GPU."""
        pos = self._gpu(self.point["positions"]).to(torch.float32)
        inten = None
        if "intensity" in self.point:
            inten = self._gpu(self.point["intensity"]).reshape(-1).to(torch.float32)
        return self._ctx().pack_xyzi(pos, inten)

    def _home(self, t: torch.Tensor) -> Tensor:
        return Tensor(t if self.device.kind == "CUDA" else t.cpu())

    def _like(self, attrs: dict):
        out = PointCloud(self.device)
        for k, v in attrs.items():
            out.point[k] = v
        return out

    def _gather_all(self, idx32: torch.Tensor, n: int):
        ctx = self._ctx()
        out = {}
        for k, v in self.point.items():
            src = self._gpu(v)
            out[k] = self._home(ctx.gather(src, idx32, n))
        return self._like(out)

    # -- selection (utils.py:271,297,534,541; pp.py:542)
    def select_by_mask(self, mask, invert=False):
        m = mask.t if isinstance(mask, Tensor) else torch.as_tensor(np.asarray(mask))
        if m.shape[0] != self._n():
            raise ValueError("mask length does not match the number of points")
        m8 = (m if m.is_cuda else m.cuda()).to(torch.uint8).contiguous()
        ctx = self._ctx()
        _, idx, cnt = ctx.select_by_mask(None, m8, invert=invert, want_idx=True)
        n = int(cnt.item())
        return self._gather_all(idx[:n].contiguous(), n)

    def select_by_index(self, indices, invert=False, remove_duplicates=False):
        idx = indices.t if isinstance(indices, Tensor) else torch.as_tensor(np.asarray(indices))
        idx = (idx if idx.is_cuda else idx.cuda()).reshape(-1)
        if invert:
            mask = torch.ones(self._n(), dtype=torch.uint8, device=idx.device)
            mask[idx.long()] = 0
            return self.select_by_mask(Tensor(mask))
        idx32 = idx.to(torch.int32).contiguous()
        return self._gather_all(idx32, idx32.shape[0])

    # -- filters
    def remove_non_finite_points(self, remove_nan=True, remove_infinite=True):      # pp.py:469
        mask = self._ctx().non_finite_mask(self._xyzi(), remove_nan, remove_infinite)
        return self.select_by_mask(Tensor(mask)), self._home(mask.to(torch.bool))

    def remove_duplicated_points(self):                                             # utils.py:544
        mask = self._ctx().duplicate_mask(self._xyzi())
        return self.select_by_mask(Tensor(mask)), self._home(mask.to(torch.bool))

    def unique_rows_index(self) -> "Tensor":                                        # utils.py:532-533
        """``np.unique(positions, axis=0, return_index=True)[1]``: lowest input index of every
        unique row, in lexicographic row order (device sort)."""
        first, _, cnt = self._ctx().unique_rows(self._xyzi(), want_first=True, want_inverse=False)
        return Tensor(first[:int(cnt.item())])

    def unique_rows_inverse(self) -> "Tensor":                                      # utils.py:538-540
        """``torch.unique(positions, dim=0, return_inverse=True)[1]``: unique-row number of every
        input row (NaN-free input; NaN rows are ordered like numpy orders them)."""
        _, inverse, _ = self._ctx().unique_rows(self._xyzi(), want_first=False, want_inverse=True)
        return Tensor(inverse[:self._n()])

    def transform(self, T):                                                         # pp.py:482,487,490
        T = T.t.cpu().numpy() if isinstance(T, Tensor) else np.asarray(T)
        ctx = self._ctx()
        xyzi = ctx.transform(self._xyzi(), T.astype(np.float32))
        pos, _ = ctx.split_xyzi(xyzi, want_intensity=False)
        self.point["positions"] = self._home(pos)
        if "normals" in self.point:
            # Open3D rotates the normals by the upper-left 3x3 block (no translation, no divide)
            R = np.eye(4, dtype=np.float32)
            R[:3, :3] = T.astype(np.float32)[:3, :3]
            nrm = ctx.pack_xyzi(self._gpu(self.point["normals"]).to(torch.float32), None)
            rot, _ = ctx.split_xyzi(ctx.transform(nrm, R), want_intensity=False)
            self.point["normals"] = self._home(rot)
        return self

    def crop_mask(self, min_bound, max_bound, mode=_capi.CROP_OPEN3D, invert=False) -> Tensor:
        return Tensor(self._ctx().crop_mask(self._xyzi(), min_bound, max_bound, mode=mode, invert=invert))

    def crop(self, aabb, invert=False):                                             # utils.py:299
        lo = aabb.min_bound.t.cpu().double().tolist()
        hi = aabb.max_bound.t.cpu().double().tolist()
        return self.select_by_mask(self.crop_mask(lo, hi, _capi.CROP_OPEN3D, invert))

    # -- voxel grid (pp.py:511)
    def voxel_down_sample(self, voxel_size, reduction="mean"):
        if reduction != "mean":
            raise NotImplementedError("only reduction='mean' is implemented")
        if voxel_size <= 0:
            raise ValueError("voxel_size must be positive")
        ctx = self._ctx()
        n = self._n()
        out, p2v, _, cnt = ctx.voxel_downsample(self._xyzi(), voxel_size, want_p2v=True)
        ctx.check()
        v = int(cnt.item())
        pos, inten = ctx.split_xyzi(out, v, want_intensity="intensity" in self.point)
        attrs = {"positions": self._home(pos)}
        for k, val in self.point.items():
            if k == "positions":
                continue
            src = self._gpu(val)
            if k == "intensity":
                res = inten.reshape((v,) + tuple(src.shape[1:])).to(src.dtype)
            else:
                # Open3D: attr.to(float32) -> index_add mean -> cast back to the attribute dtype
                cols = src.reshape(n, -1)
                fb = engine.attr_frac_bits(cols)
                outs = [ctx.voxel_mean_attr(cols[:, c].to(torch.float32).contiguous(), p2v, cnt, n, fb)[:v]
                        for c in range(cols.shape[1])]
                res = torch.stack(outs, 1).reshape((v,) + tuple(src.shape[1:])).to(src.dtype)
            attrs[k] = self._home(res)
        return self._like(attrs)

    # -- outliers (pp.py:516; TODO pp.py:37)
    def remove_statistical_outliers(self, nb_neighbors, std_ratio):
        """Open3D ``remove_statistical_outliers``: keep the points whose mean distance to their
        ``nb_neighbors`` nearest (self included) is at most mu + std_ratio * sigma.  ``nb_neighbors`` in
        1..``APC_MAX_NEIGHBORS`` (1024; beyond it the call raises ``ApcError``)."""
        if nb_neighbors < 1 or std_ratio <= 0:
            raise ValueError("Illegal input parameters, the number of neighbors and standard deviation ratio must be positive")
        ctx = self._ctx()
        mask, _, _ = ctx.statistical_outliers(self._xyzi(), nb_neighbors, std_ratio)
        ctx.check()
        return self.select_by_mask(Tensor(mask)), self._home(mask.to(torch.bool))

    def remove_radius_outliers(self, nb_points, search_radius):
        if nb_points < 1 or search_radius <= 0:
            raise ValueError("Illegal input parameters, number of points and radius must be positive")
        ctx = self._ctx()
        mask, _ = ctx.radius_outliers(self._xyzi(), nb_points, search_radius)
        ctx.check()
        return self.select_by_mask(Tensor(mask)), self._home(mask.to(torch.bool))

    # -- clustering
    def cluster_dbscan(self, eps, min_points, print_progress=False):
        """Open3D ``cluster_dbscan``: int32 label of every point (``Tensor`` [N] on the cloud's device), -1 for
        noise.  Neighbours are the points within ``eps`` (self included, the float32 distance of
        ``remove_radius_outliers``); a point with at least ``min_points`` neighbours is a core point; clusters are
        the connected components of the core points, numbered in the order of their lowest point index; a
        non-core point joins the lowest-numbered cluster among its core neighbours.  ``print_progress`` is
        accepted and ignored."""
        if not (math.isfinite(eps) and eps > 0) or min_points < 0:
            raise ValueError("Illegal input parameters, eps must be positive and finite and min_points >= 0")
        n = self._n()
        if n == 0:
            return self._home(torch.zeros((0,), dtype=torch.int32, device="cuda"))
        ctx = self._ctx()
        labels, _, _ = ctx.cluster_dbscan(self._xyzi(), float(eps), min(int(min_points), n + 1))
        ctx.check()
        return self._home(labels.contiguous())

    # -- RANSAC plane (pp.py:535)
    def segment_plane(self, distance_threshold=0.01, ransac_n=3, num_iterations=100, probability=0.99999999,
                      seed=0):
        """Returns ``(plane_model Tensor float64[4], inliers Tensor int64[K])``.  ``seed`` selects
        the hypothesis stream (the reference never seeds Open3D's RNG, pp.py:535-540)."""
        if self._n() < ransac_n:
            raise RuntimeError("There must be at least 'ransac_n' points.")
        ctx = self._ctx()
        plane8, mask, _ = ctx.segment_plane(self._xyzi(), distance_threshold, ransac_n, num_iterations, probability,
                                            seed=seed)
        _, idx, cnt = ctx.select_by_mask(None, mask.contiguous(), invert=False, want_idx=True)
        k = int(cnt.item())
        return self._home(plane8[:4].clone()), self._home(idx[:k].to(torch.int64))

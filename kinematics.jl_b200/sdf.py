"""BoxSDF / UnionSDF (sdf.jl:1-119) on the B200 backend.  An SDF object is a description (box poses
and widths); evaluating it at points or against a robot's collision spheres runs in libkin_b200.

SphereSDF / CylinderSDF are an EXTENSION (SURVEY 8 f4): the reference supports boxes only
(load_urdf.jl:10-15, sdf.jl:92-94).  They honour the same AbstractSDF contract -- ``sdf(p)``, the generic
forward-difference ``gradient!`` (sdf.jl:34-41), membership in a UnionSDF with first-minimum argmin.  So does
GridSDF, a sampled signed-distance grid (extension; the formula is stated at KinGrid in include/kin_b200.h)."""
from __future__ import annotations

import ctypes as C
import itertools
import uuid

import numpy as np

from . import lib as _lib
from .mechanism import BoxMetaData, CylinderMetaData, Link, Mechanism, SphereMetaData, add_new_link
from .transform import Transform


class AbstractSDF:
    def world_boxes(self):
        """-> (poses (B, 4, 4), widths (B, 3)) in UnionSDF.sdfs order."""
        raise NotImplementedError

    def world_primitives(self):
        """-> (poses (B, 4, 4), sizes (B, 3), kinds (B,) int32: lib.PRIM_BOX / PRIM_SPHERE / PRIM_CYLINDER)."""
        poses, widths = self.world_boxes()
        return poses, widths, np.zeros(len(poses), dtype=np.int32)

    def world_scene(self):
        """-> world_primitives() + grids: a list with the GridSDF of every lib.PRIM_GRID row, None on the others."""
        poses, sizes, kinds = self.world_primitives()
        return poses, sizes, kinds, [None] * len(poses)

    # ---- sdf(p) and gradient!(sdf, p, out) -------------------------------------------------------
    def __call__(self, p, return_argmin=False):
        """sdf.jl:67-74 / 108-114.  ``p``: 3-vector -> float, or points (N, 3) -> tensor (N,)."""
        vals, _, am = self._points(p, want_grad=False, want_argmin=return_argmin)
        return (vals, am) if return_argmin else vals

    def gradient(self, p, grad_mode=_lib.GRAD_FD):
        """``gradient!`` (sdf.jl:34-41, 116-119): forward difference (eps 1e-7) on the argmin box."""
        return self._points(p, want_grad=True, grad_mode=grad_mode)[1]

    def _points(self, p, want_grad, want_argmin=False, grad_mode=_lib.GRAD_FD):
        import torch
        if not torch.cuda.is_available():
            raise _lib.KinError("no CUDA device: the kinematics.jl_b200 operators have no CPU fallback")
        single = not isinstance(p, torch.Tensor) and np.ndim(p) == 1
        P = p if isinstance(p, torch.Tensor) else torch.as_tensor(np.atleast_2d(np.asarray(p, dtype=np.float64)))
        P = P.cuda()
        if P.dtype not in (torch.float32, torch.float64):
            P = P.double()
        P = P.contiguous()
        N = P.shape[0]
        poses, widths, kinds, grids = self.world_scene()
        poses_cm = np.ascontiguousarray(poses.transpose(0, 2, 1)).reshape(-1, 16)
        widths = np.ascontiguousarray(widths, dtype=np.float64)
        kinds = np.ascontiguousarray(kinds, dtype=np.int32)
        vals = torch.empty(N, dtype=P.dtype, device=P.device)
        grads = torch.empty((N, 3), dtype=P.dtype, device=P.device) if want_grad else None
        am = torch.empty(N, dtype=torch.int32, device=P.device) if want_argmin else None
        dp = C.POINTER(C.c_double)
        head = (len(poses_cm), kinds.ctypes.data_as(C.POINTER(C.c_int32)), poses_cm.ctypes.data_as(dp), widths.ctypes.data_as(dp))
        tail = (_lib.F32 if P.dtype == torch.float32 else _lib.F64, _lib.AOS, P.data_ptr(), N, grad_mode,
                vals.data_ptr(), grads.data_ptr() if want_grad else None, am.data_ptr() if want_argmin else None,
                torch.cuda.current_stream(P.device).cuda_stream)
        if any(g is not None for g in grids):
            _lib.check(_lib.lib().kin_sdf_points_scene(*head, grid_handles(grids), *tail))
        else:
            _lib.check(_lib.lib().kin_sdf_points_prims(*head, *tail))
        if single:
            return (float(vals[0]), grads[0].double().cpu().numpy() if want_grad else None,
                    int(am[0]) if want_argmin else None)
        return vals, grads, am


class BoxSDF(AbstractSDF):
    """sdf.jl:48-65: ``BoxSDF(pose, width)`` stand-alone, or attached to a link of a mechanism."""

    def __init__(self, pose, width=None, attach=None):
        if isinstance(pose, BoxMetaData):
            pose, width = pose.origin, pose.extents
        self.pose = pose if isinstance(pose, Transform) else Transform(pose)
        self.width = np.asarray(width, dtype=np.float64)
        self.attach = attach               # (mech, link) for IsAttached (sdf.jl:3-6)

    def world_pose(self):
        if self.attach is None:
            return self.pose.mat
        from .algorithm import get_transform
        mech, link = self.attach           # sdf.jl:14-32: pose of the SDF link in the obstacle mechanism
        return _obstacle_transform(mech, link)

    def world_boxes(self):
        return self.world_pose()[None], self.width[None]


class SphereSDF(BoxSDF):
    """Extension: ``SphereSDF(pose, radius)``; d = |p - c| - r."""
    kind = _lib.PRIM_SPHERE

    def __init__(self, pose, radius=None, attach=None):
        if isinstance(pose, SphereMetaData):
            pose, radius = pose.origin, pose.radius
        BoxSDF.__init__(self, pose, [radius, 0.0, 0.0], attach)
        self.radius = float(radius)

    def world_boxes(self):
        raise _lib.KinError("a SphereSDF is not a box: use world_primitives()")

    def world_primitives(self):
        return self.world_pose()[None], self.width[None], np.array([self.kind], dtype=np.int32)


class CylinderSDF(SphereSDF):
    """Extension: ``CylinderSDF(pose, radius, length)``, axis = local z, centred on the pose (URDF <cylinder>)."""
    kind = _lib.PRIM_CYLINDER

    def __init__(self, pose, radius=None, length=None, attach=None):
        if isinstance(pose, CylinderMetaData):
            pose, radius, length = pose.origin, pose.radius, pose.length
        BoxSDF.__init__(self, pose, [radius, length, 0.0], attach)
        self.radius, self.length = float(radius), float(length)


_grid_serial = itertools.count(1)


class GridSDF(BoxSDF):
    """Extension: a sampled signed-distance grid.  ``values`` is an (nx, ny, nz) array or CUDA tensor indexed [i, j, k]
    (x first), ``spacing`` the distance between samples; the grid is centred on ``pose``.  The samples are stored as
    float32 on the device (``kin_grid_create``); between samples the distance is interpolated trilinearly, outside the
    grid box the distance to the box is added (include/kin_b200.h, KinGrid)."""
    kind = _lib.PRIM_GRID

    def __init__(self, values, spacing, pose=None, attach=None):
        BoxSDF.__init__(self, Transform() if pose is None else pose, [0.0, 0.0, 0.0], attach)
        self.h = None
        self.shape = tuple(int(n) for n in values.shape)
        if len(self.shape) != 3:
            raise ValueError("GridSDF: values must be an (nx, ny, nz) array, got shape %s" % (self.shape,))
        self.spacing = float(spacing)
        self.serial = next(_grid_serial)      # identity of the device storage (DeviceModel.set_boxes compares it)
        buf, keep = self._storage(values)
        if hasattr(keep, "is_cuda"):
            import torch
            torch.cuda.current_stream(keep.device).synchronize()  # kin_grid_create copies on the legacy default stream
        h = C.c_void_p()
        _lib.check(_lib.lib().kin_grid_create(*self.shape, self.spacing, buf, C.byref(h)))
        self.h = h

    def __del__(self):
        try:
            if self.h:
                _lib.lib().kin_grid_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def _storage(self, values):
        """values -> (address of the samples with x fastest, float32, keep-alive)."""
        if tuple(values.shape) != self.shape:
            raise ValueError("GridSDF: values of shape %s, the grid is %s" % (tuple(values.shape), self.shape))
        if hasattr(values, "is_cuda") and values.is_cuda:
            import torch
            t = values.detach().permute(2, 1, 0).contiguous().to(torch.float32)
            return t.data_ptr(), t
        if hasattr(values, "detach"):
            values = values.detach().numpy()
        a = np.ascontiguousarray(np.asarray(values, dtype=np.float32).transpose(2, 1, 0))
        return a.ctypes.data, a

    def update(self, values):
        """Rewrites the samples in place (``kin_grid_set_values``, ordered on the current stream); the shape stays.
        Every model and union that holds this grid sees the new values at its next launch; nothing recompiles."""
        import torch
        buf, keep = self._storage(values)      # a temporary tensor is freed in the order of the current stream
        _lib.check(_lib.lib().kin_grid_set_values(self.h, buf, torch.cuda.current_stream().cuda_stream))

    @classmethod
    def from_sdf(cls, sdf, pose, shape, spacing, attach=None):
        """Samples any AbstractSDF on the device at the points of a grid of ``shape`` = (nx, ny, nz) samples at
        ``spacing``, centred on ``pose`` (e.g. rasterises a UnionSDF of boxes)."""
        import torch
        if not torch.cuda.is_available():
            raise _lib.KinError("no CUDA device: the kinematics.jl_b200 operators have no CPU fallback")
        nx, ny, nz = (int(n) for n in shape)
        pose = pose if isinstance(pose, Transform) else Transform(pose if pose is not None else np.eye(4))
        axes = [(torch.arange(n, dtype=torch.float64, device="cuda") - (n - 1) / 2.0) * float(spacing) for n in (nx, ny, nz)]
        gx, gy, gz = torch.meshgrid(*axes, indexing="ij")                       # (nx, ny, nz), [i, j, k]
        local = torch.stack([gx.reshape(-1), gy.reshape(-1), gz.reshape(-1)], dim=1)
        M = torch.as_tensor(pose.mat, dtype=torch.float64, device="cuda")
        world = (local @ M[:3, :3].T + M[:3, 3]).contiguous()
        vals = sdf(world).reshape(nx, ny, nz)
        return cls(vals, spacing, pose, attach)

    def world_boxes(self):
        raise _lib.KinError("a GridSDF is not a box: use world_scene()")

    def world_primitives(self):
        raise _lib.KinError("a GridSDF needs its grid handle: use world_scene()")

    def world_scene(self):
        return self.world_pose()[None], self.width[None], np.array([self.kind], dtype=np.int32), [self]


def grid_handles(grids):
    """[GridSDF or None] -> the KinGrid* array of kin_model_set_scene / kin_sdf_points_scene."""
    return (C.c_void_p * len(grids))(*[g.h.value if g is not None else None for g in grids])


def _obstacle_transform(mech: Mechanism, link: Link):
    """World pose of an attached SDF link at the obstacle mechanism's current state (FK runs on the GPU,
    N = 1), memoised on the mechanism per state version like the reference memoises inv_pose (sdf.jl:14-20)."""
    from .algorithm import get_transform
    version = (mech._state_version, mech._structure_version)
    cache = getattr(mech, "_sdf_pose_cache", None)
    if cache is None or cache[0] != version:
        cache = mech._sdf_pose_cache = (version, {})
    if link.id not in cache[1]:
        assert mech._single, "an obstacle mechanism must hold a single configuration"
        cache[1][link.id] = get_transform(mech, link).mat
    return cache[1][link.id]


class UnionSDF(AbstractSDF):
    """sdf.jl:76-114.  ``UnionSDF(mech)`` makes one box per link of ``mech`` that carries box collision
    metadata, in ``mech.links`` order, attached through a new link placed at the collision origin
    (sdf.jl:82-97); ``UnionSDF([sdf, ...])`` unions existing SDFs."""

    def __init__(self, arg, primitives=False):
        """``primitives=True`` (extension) also turns the URDF's <sphere> / <cylinder> collision geometry into
        SphereSDF / CylinderSDF members; the default skips them as the reference does (sdf.jl:92-94)."""
        if isinstance(arg, Mechanism):
            mech, sdfs = arg, []
            for link in list(mech.links):
                meta = link.geometric_meta_data
                cls = BoxSDF if isinstance(meta, BoxMetaData) else None
                if primitives and link.link_type == "URDF":
                    cls = SphereSDF if isinstance(meta, SphereMetaData) else CylinderSDF if isinstance(meta, CylinderMetaData) else cls
                if cls is not None:
                    new_link = Link("boxsdf_" + str(uuid.uuid1()), link_type="SdfLinkType")
                    add_new_link(mech, new_link, link, meta.origin)
                    sdfs.append(cls(meta, attach=(mech, new_link)))
            self.sdfs = sdfs
        else:
            self.sdfs = list(arg)

    def world_boxes(self):
        parts = [s.world_boxes() for s in self.sdfs]
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])

    def world_primitives(self):
        parts = [s.world_primitives() for s in self.sdfs]
        return tuple(np.concatenate([p[i] for p in parts]) for i in range(3))

    def world_scene(self):
        parts = [s.world_scene() for s in self.sdfs]
        return tuple(np.concatenate([p[i] for p in parts]) for i in range(3)) + ([g for p in parts for g in p[3]],)

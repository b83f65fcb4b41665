"""Device models: flattens a ``Mechanism`` (+ control joints, frozen joint angles, sphere and box
tables) into the ``KinModelDesc`` of include/kin_b200.h, keeps the resulting handles cached on the
mechanism, and issues ``kin_eval`` calls on torch CUDA tensors.  torch is used for device memory and
streams only."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import lib as _lib
from .mechanism import Mechanism

_MAX_CACHED = 8


def _dptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _iptr(a):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


def make_desc(m: Mechanism, ctrl_ids, spheres=None, boxes=None):
    """Mechanism (+ optional (links, centers, radii) and (poses, widths)) -> (KinModelDesc, keep-alive).
    Pure host code: also used by the CPU tests through ``kin_program_dump``."""
    L = len(m.links)
    parent = np.full(L, -1, dtype=np.int32)
    jtype = np.zeros(L, dtype=np.int32)
    pose = np.tile(np.eye(4).reshape(-1), (L, 1))
    axis = np.zeros((L, 3))
    qidx = np.full(L, -1, dtype=np.int32)
    defang = np.zeros(L)
    col = {jid: c for c, jid in enumerate(ctrl_ids)}
    for l in m.links:
        i = l.id - 1
        if l.plink_id == -1:
            continue
        j = m.joints[l.pjoint_id - 1]
        parent[i] = l.plink_id
        jtype[i] = j.type
        pose[i] = j.pose.mat.T.reshape(-1)          # column-major, like Transform.mat in Julia
        axis[i] = j.axis
        qidx[i] = col.get(j.id, -1)
        defang[i] = m.angles[j.id - 1]
    keep = [parent, jtype, np.ascontiguousarray(pose), np.ascontiguousarray(axis), qidx, defang]
    d = _lib.KinModelDesc()
    d.n_links = L
    d.parent_link, d.joint_type, d.joint_pose = _iptr(parent), _iptr(jtype), _dptr(keep[2])
    d.joint_axis, d.q_index, d.default_angle = _dptr(keep[3]), _iptr(qidx), _dptr(defang)
    d.n_joints = len(ctrl_ids)
    d.with_base = int(m.with_base)
    d.n_spheres = d.n_boxes = 0
    if spheres is not None:
        sl = np.ascontiguousarray(spheres[0], dtype=np.int32)
        sc = np.ascontiguousarray(spheres[1], dtype=np.float64).reshape(-1, 3)
        sr = np.ascontiguousarray(spheres[2], dtype=np.float64)
        keep += [sl, sc, sr]
        d.n_spheres, d.sphere_link, d.sphere_center, d.sphere_radius = len(sl), _iptr(sl), _dptr(sc), _dptr(sr)
    if boxes is not None:
        bp = np.ascontiguousarray(np.asarray(boxes[0], dtype=np.float64).reshape(-1, 4, 4).transpose(0, 2, 1)).reshape(-1, 16)
        bw = np.ascontiguousarray(boxes[1], dtype=np.float64).reshape(-1, 3)
        keep += [bp, bw]
        d.n_boxes, d.box_pose, d.box_width = len(bp), _dptr(bp), _dptr(bw)
    return d, keep


class DeviceModel:
    """Owns one ``KinModel*``."""

    def __init__(self, m: Mechanism, ctrl_ids):
        d, self._keep = make_desc(m, ctrl_ids)
        h = C.c_void_p()
        _lib.check(_lib.lib().kin_model_create(C.byref(d), C.byref(h)))
        self.h = h
        self.n_dof = len(ctrl_ids) + (3 if m.with_base else 0)
        self.n_links = len(m.links)
        self._sph_sig = self._box_sig = self._pair_sig = None
        self.n_spheres = self.n_boxes = self.n_self_pairs = 0

    def __del__(self):
        try:
            if self.h:
                _lib.lib().kin_model_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def set_spheres(self, links, centers, radii):
        links = np.ascontiguousarray(links, dtype=np.int32)
        centers = np.ascontiguousarray(centers, dtype=np.float64).reshape(-1, 3)
        radii = np.ascontiguousarray(radii, dtype=np.float64)
        sig = (links.tobytes(), centers.tobytes(), radii.tobytes())
        if sig != self._sph_sig:
            _lib.check(_lib.lib().kin_model_set_spheres(self.h, len(links), _iptr(links), _dptr(centers), _dptr(radii)))
            self._sph_sig, self.n_spheres = sig, len(links)
            self._pair_sig, self.n_self_pairs = None, 0         # the library dropped the pair table with the old spheres

    def set_self_pairs(self, pairs):
        """Self-collision pair table: (P, 2) 1-based sphere ids (``kin_model_set_self_pairs``)."""
        pairs = np.ascontiguousarray(np.asarray(pairs, dtype=np.int32).reshape(-1, 2))
        sig = pairs.tobytes()
        if sig != self._pair_sig:
            _lib.check(_lib.lib().kin_model_set_self_pairs(self.h, len(pairs), _iptr(pairs)))
            self._pair_sig, self.n_self_pairs = sig, len(pairs)

    def set_boxes(self, poses, widths, kinds=None, grids=None):
        """The SDF table (``kin_model_set_boxes`` / ``_primitives``; with a GridSDF in ``grids``, ``kin_model_set_scene``).
        A grid enters the signature by identity only: its samples live in the grid's own device storage, which the
        model shares, so ``GridSDF.update`` needs no new call here."""
        poses = np.ascontiguousarray(np.asarray(poses, dtype=np.float64).reshape(-1, 4, 4).transpose(0, 2, 1)).reshape(-1, 16)
        widths = np.ascontiguousarray(widths, dtype=np.float64).reshape(-1, 3)
        kinds = np.zeros(len(poses), dtype=np.int32) if kinds is None else np.ascontiguousarray(kinds, dtype=np.int32)
        has_grid = grids is not None and any(g is not None for g in grids)
        sig = (poses.tobytes(), widths.tobytes(), kinds.tobytes())
        if has_grid:
            sig += (tuple(g.serial if g is not None else 0 for g in grids),)
        if sig != self._box_sig:
            if has_grid:
                from .sdf import grid_handles
                _lib.check(_lib.lib().kin_model_set_scene(self.h, len(poses), _iptr(kinds), _dptr(poses), _dptr(widths),
                                                          grid_handles(grids)))
            elif kinds.any():       # sphere / cylinder rows (extension)
                _lib.check(_lib.lib().kin_model_set_primitives(self.h, len(poses), _iptr(kinds), _dptr(poses), _dptr(widths)))
            else:
                _lib.check(_lib.lib().kin_model_set_boxes(self.h, len(poses), _dptr(poses), _dptr(widths)))
            self._box_sig, self.n_boxes = sig, len(poses)


def device_model(m: Mechanism, ctrl_ids=None) -> DeviceModel:
    """Cached per (structure, control joints, angles of the joints that are not controlled)."""
    ctrl_ids = tuple(m._ctrl if ctrl_ids is None else ctrl_ids)
    frozen = m.angles.copy()
    for jid in ctrl_ids:
        frozen[jid - 1] = 0.0
    key = (m._structure_version, ctrl_ids, frozen.tobytes())
    dm = m._models.get(key)
    if dm is None:
        if len(m._models) >= _MAX_CACHED:
            m._models.pop(next(iter(m._models)))
        dm = m._models[key] = DeviceModel(m, ctrl_ids)
    return dm


def current_q(m: Mechanism, dtype=None):
    """The configuration batch as a CUDA tensor + its layout.  Returns (tensor, layout, N)."""
    import torch
    if not torch.cuda.is_available():
        raise _lib.KinError("no CUDA device: the kinematics.jl_b200 operators have no CPU fallback")
    n_dof = len(m._ctrl) + (3 if m.with_base else 0)
    if m._Q is None:
        a = [m.angles[jid - 1] for jid in m._ctrl] + (list(m.base_pose) if m.with_base else [])
        q = torch.tensor([a if a else [0.0]], dtype=dtype or torch.float64, device="cuda")
        return q, _lib.AOS, 1
    Q = m._Q
    if not isinstance(Q, torch.Tensor):
        Q = torch.as_tensor(np.ascontiguousarray(Q))
    if not Q.is_cuda:
        Q = Q.cuda()
    if dtype is not None and Q.dtype != dtype:
        Q = Q.to(dtype)
    if Q.dtype not in (torch.float64, torch.float32):
        Q = Q.double()
    N = Q.shape[0]
    if n_dof == 0:
        return torch.zeros(1, dtype=Q.dtype, device="cuda"), _lib.AOS, N
    if Q.is_contiguous():
        return Q, _lib.AOS, N
    if Q.t().is_contiguous():
        return Q, _lib.SOA, N
    return Q.contiguous(), _lib.AOS, N


def tile32(x):
    """(N, rec) batch-first tensor -> tiled storage (ceil(N/32), rec, 32) (KIN_LAYOUT_TILED32), zero padded."""
    import torch
    N, rec = x.shape
    NT = (N + 31) // 32
    out = torch.zeros((NT * 32, rec), dtype=x.dtype, device=x.device)
    out[:N] = x
    return out.reshape(NT, 32, rec).permute(0, 2, 1).contiguous()


def untile32(x, N):
    """tiled storage (NT, ..., 32) -> batch-first (N, ...) copy."""
    nd = x.dim()
    return x.permute(0, nd - 1, *range(1, nd - 1)).reshape((x.shape[0] * 32,) + tuple(x.shape[1:-1]))[:N]


def _relayout(Q, q_layout, layout):
    """Q (batch-first (N, n_dof) in ``q_layout``) brought to the layout of a call: one layout per call."""
    if layout == _lib.TILED32:
        return tile32(Q.contiguous() if q_layout == _lib.AOS else Q)
    if layout != q_layout:
        return Q.t().contiguous().t() if layout == _lib.SOA else Q.contiguous()
    return Q


def _alloc(layout, N, shape_soa, shape_aos, dtype, dev):
    """Output storage of a call: SoA / AoS shapes as given; tiled: (NT, components..., 32), the SoA component order
    inside each tile."""
    import torch
    if layout == _lib.TILED32:
        return torch.empty(((N + 31) // 32,) + tuple(shape_soa[:-1]) + (32,), dtype=dtype, device=dev)
    return torch.empty(shape_soa if layout == _lib.SOA else shape_aos, dtype=dtype, device=dev)


def _view(x, layout, N, perm_soa, perm_aos):
    """Batch-first view of an output storage; tiled: a batch-first COPY (N, c1, ..., ck), then the SoA reordering of
    the component axes (indices shifted by one)."""
    if layout == _lib.TILED32:
        return untile32(x, N).permute(0, *[p + 1 for p in perm_soa[1:]])
    return x.permute(*perm_soa) if layout == _lib.SOA else x.permute(*perm_aos)


def _into(buf, shape, dtype, dev):
    """Caller-provided output storage (SoA / AoS only): must be a contiguous tensor of exactly the storage shape."""
    if tuple(buf.shape) != tuple(shape) or buf.dtype != dtype or buf.device != dev or not buf.is_contiguous():
        raise ValueError("output storage must be a contiguous %s tensor of shape %s on %s" % (dtype, tuple(shape), dev))
    return buf


def evaluate(dm: DeviceModel, Q, q_layout, N, *, layout=None, fk_links=None, jac_links=None, with_rot=True,
             rpy_jac=False, keep_irrelevant=False, J_into=None, collision=False, with_grads=True,
             truncation_dist=np.inf, grad_mode=_lib.GRAD_FD, scratch_mode=_lib.SCRATCH_REFERENCE,
             want_argmin=False, vals_offset=0.0, stream=None, launch_info=False, vals_into=None, grads_into=None):
    """One ``kin_eval``.  Outputs are allocated in the layout of the call (default: the layout of Q) and
    returned as batch-first VIEWS: T (N, n_fk, 3, 4), J (N, n_jac, rows, cols), vals (N, S),
    grads (N, n_dof, S), argmin (N, S)."""
    import torch
    layout = q_layout if layout is None else layout
    Q = _relayout(Q, q_layout, layout)
    dt = Q.dtype
    dev = Q.device
    c = _lib.KinCall()
    c.precision = _lib.F32 if dt == torch.float32 else _lib.F64
    c.layout = layout
    c.n = N
    c.batch_stride = 0
    c.q = Q.data_ptr()
    c.truncation_dist = float(truncation_dist)
    c.grad_mode, c.scratch_mode = grad_mode, scratch_mode
    c.vals_offset = float(vals_offset)
    c.stream = torch.cuda.current_stream(dev).cuda_stream if stream is None else stream
    nd = dm.n_dof
    out = {}
    keep = []
    pending = []                             # (key, storage, perm_soa, perm_aos): views are built after the launch
    if fk_links is not None and len(fk_links):
        ids = np.ascontiguousarray(fk_links, dtype=np.int32)
        keep.append(ids)
        n = len(ids)
        T = _alloc(layout, N, (n, 4, 3, N), (N, n, 4, 3), dt, dev)
        c.n_fk_links, c.fk_links, c.T_out = n, _iptr(ids), T.data_ptr()
        pending.append(("T", T, (3, 0, 2, 1), (0, 1, 3, 2)))
    if jac_links is not None and len(jac_links):
        ids = np.ascontiguousarray(jac_links, dtype=np.int32)
        keep.append(ids)
        n, rows = len(ids), (6 if with_rot else 3)
        if J_into is not None:
            J = J_into                       # storage tensor in the call's layout (get_jacobian! semantics)
            if J.dtype != dt or J.device != dev or J.numel() != n * nd * rows * N:
                raise ValueError("get_jacobian!: mat_out must be a %s tensor on %s holding %d x %d x %d values per "
                                 "configuration (got %s, %s, %d values)" % (dt, dev, n, rows, nd, J.dtype, J.device, J.numel()))
        else:
            J = _alloc(layout, N, (n, nd, rows, N), (N, n, nd, rows), dt, dev)
        c.n_jac_links, c.jac_links, c.J_out = n, _iptr(ids), J.data_ptr()
        c.with_rot, c.rpy_jac, c.keep_irrelevant = int(with_rot), int(rpy_jac), int(keep_irrelevant)
        pending.append(("J", J, (3, 0, 2, 1), (0, 1, 3, 2)))
    if collision:
        if dm.n_spheres == 0 or dm.n_boxes == 0:
            raise _lib.KinError("collision requested but the device model has no spheres / no boxes "
                                "(add_coll_links and pass an SDF first)")
        S = dm.n_spheres
        V = _alloc(layout, N, (S, N), (N, S), dt, dev) if vals_into is None else \
            _into(vals_into, (S, N) if layout == _lib.SOA else (N, S), dt, dev)
        c.vals_out = V.data_ptr()
        pending.append(("vals", V, (1, 0), (0, 1)))
        if with_grads:
            G = _alloc(layout, N, (S, nd, N), (N, S, nd), dt, dev) if grads_into is None else \
                _into(grads_into, (S, nd, N) if layout == _lib.SOA else (N, S, nd), dt, dev)
            c.grads_out = G.data_ptr()
            pending.append(("grads", G, (2, 1, 0), (0, 2, 1)))
        if want_argmin:
            Am = _alloc(layout, N, (S, N), (N, S), torch.int32, dev)
            c.argmin_out = Am.data_ptr()
            pending.append(("argmin", Am, (1, 0), (0, 1)))
    _lib.check(_lib.lib().kin_eval(dm.h, C.byref(c)))
    for key, store, perm_soa, perm_aos in pending:
        out[key] = _view(store, layout, N, perm_soa, perm_aos)
    if launch_info:                          # which kernel configuration this call maps to (kin_query_launch)
        regs, smem, block, grid = C.c_int32(), C.c_int32(), C.c_int32(), C.c_int32()
        _lib.check(_lib.lib().kin_query_launch(dm.h, C.byref(c), C.byref(regs), C.byref(smem), C.byref(block), C.byref(grid)))
        out["launch"] = {"regs": regs.value, "smem_bytes": smem.value, "block": block.value, "grid": grid.value}
    return out


def evaluate_self(dm: DeviceModel, Q, q_layout, N, *, layout=None, with_vals=True, with_grads=False,
                  truncation_dist=np.inf, vals_offset=0.0, want_summary=False, stream=None):
    """One ``kin_self_collision`` over the model's pair table.  vals / grads are allocated in the layout of the call
    (default: the layout of Q) and returned as batch-first views vals (N, P), grads (N, n_dof, P); dmin (N,) and
    amin (N,) int32 are plain arrays."""
    import torch
    layout = q_layout if layout is None else layout
    Q = _relayout(Q, q_layout, layout)
    dt, dev, nd, P = Q.dtype, Q.device, dm.n_dof, dm.n_self_pairs
    V = _alloc(layout, N, (P, N), (N, P), dt, dev) if with_vals else None
    G = _alloc(layout, N, (P, nd, N), (N, P, nd), dt, dev) if with_grads else None
    dmin = torch.empty(N, dtype=dt, device=dev) if want_summary else None
    amin = torch.empty(N, dtype=torch.int32, device=dev) if want_summary else None
    ptr = lambda t: None if t is None else t.data_ptr()
    _lib.check(_lib.lib().kin_self_collision(dm.h, _lib.F32 if dt == torch.float32 else _lib.F64, layout, Q.data_ptr(), N,
                                             float(truncation_dist), float(vals_offset), ptr(V), ptr(G), ptr(dmin), ptr(amin),
                                             torch.cuda.current_stream(dev).cuda_stream if stream is None else stream))
    out = {}
    if V is not None:
        out["vals"] = _view(V, layout, N, (1, 0), (0, 1))
    if G is not None:
        out["grads"] = _view(G, layout, N, (2, 1, 0), (0, 2, 1))
    if want_summary:
        out["dmin"], out["amin"] = dmin, amin
    return out

"""Grasp scoring on the GPU: penetration volume, penetration depth and contact of a batch of hands against one object mesh,
the metrics the reference scripts compute per grasp on the CPU (``intersection_eval`` in ``gen_diverse_grasp_obman.py``:
trimesh voxelisation and containment, igl distances).

- ``winding_number(points, verts, faces)``: generalised winding numbers (``w >= 0.5`` is "inside").
- ``point_mesh_distance(points, verts, faces, differentiable=False)``: squared distance to the mesh and the closest face.
- ``penetration_depth(points, verts, faces)``: the squared distance of the points inside the mesh (0 outside) and their
  closest face, in one fused launch; differentiable.
- ``GraspQuality(obj_verts, obj_faces, hand_faces, pitch, contact_tol)``: ``forward(hand_verts) -> (volume, depth,
  contact)``.

The contract (winding number, box rule, distance, tie rule, voxel centres, metrics) is stated once in
``csrc/mesh_exact.cuh`` and restated in float64 in ``oracle/mesh_oracle.py``.  CUDA fp32 only.  ``GraspQuality`` and
``winding_number`` have no autograd (the metrics are step functions and maxima used for scoring, so inputs that require
grad are detached); ``penetration_depth`` and ``point_mesh_distance(differentiable=True)`` carry the gradient of the
squared distance to the points and the mesh vertices, with the closest point's barycentrics held fixed (the envelope
theorem, as pytorch3d's ``point_mesh_face_distance``), for refinement losses.

The voxelisation is filled and centre-sampled: a cell counts when its centre is inside the object, and a cell of the
object counts for hand b when its centre is inside hand b.  trimesh's ``voxelized()`` marks the cells the surface passes
through (then fills), so its volume differs by up to about one layer of cells on the boundary; the two agree as the pitch
shrinks.

One object per module.  A caller whose object is rotated per grasp (the FHAB / GRAB / HO3D scripts) maps the hands into
the object's frame first: ``hand_obj = (hand - t) @ R`` for an object placed as ``R @ x + t``.
"""
from __future__ import annotations

import math

import numpy as np
import torch
from torch import nn
from torch.autograd.function import once_differentiable

from . import _cabi
from .quantizer import _stream_ptr

MAX_CELLS = 1 << 24         # voxel grid cap: above it the pitch is almost certainly a unit mistake (mm vs m)


def _points(x, name, what, detach=True):
    if not isinstance(x, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if x.dtype != torch.float32:
        raise TypeError("%s must be fp32; got %s" % (name, x.dtype))
    if not x.is_cuda:
        raise ValueError("%s has no CPU path: %s must be a CUDA tensor" % (what, name))
    if x.dim() != 3 or x.shape[2] != 3:
        raise ValueError("%s must be [B, n, 3]; got %s" % (name, tuple(x.shape)))
    return (x.detach() if detach else x).contiguous()


def check_faces(faces, num_verts=None, name="faces"):
    """Host-side validation of a triangle list: integer ``[F, 3]``, ids in ``[0, num_verts)`` -> int32 numpy array."""
    f = np.asarray(faces.detach().cpu() if isinstance(faces, torch.Tensor) else faces)
    if f.dtype.kind not in "iu":
        raise TypeError("%s must be an integer array; got %s" % (name, f.dtype))
    if f.ndim != 2 or f.shape[1] != 3:
        raise ValueError("%s must be [F, 3]; got %s" % (name, f.shape))
    if f.size and (f.min() < 0 or f.max() >= (num_verts if num_verts is not None else 2 ** 31 - 1)):
        raise ValueError("%s: vertex ids must be in [0, V)%s" % (name, "" if num_verts is None else " (V = %d)" % num_verts))
    return np.ascontiguousarray(f.astype(np.int32))


def _broadcast(Bm, Bp):
    if Bm != Bp and 1 not in (Bm, Bp):
        raise ValueError("points and verts batch sizes must be equal or 1; got %d and %d" % (Bp, Bm))
    return Bp if Bm == 1 else Bm


def _prepare(points, verts, faces, what, detach=True):
    points, verts = _points(points, "points", what, detach), _points(verts, "verts", what, detach)
    if points.device != verts.device:
        raise ValueError("points are on %s, verts on %s" % (points.device, verts.device))
    if verts.shape[1] == 0:
        raise ValueError("verts must hold at least one vertex per batch item")
    f = torch.from_numpy(check_faces(faces, verts.shape[1])).to(verts.device)
    return points, verts, f, _broadcast(verts.shape[0], points.shape[0])


def _mesh_call(entry, points, verts, faces, *tensors):
    """Calls the C entry ``entry`` (one of the four ``dvq_mesh_*``) with the common mesh arguments (verts, Bm, V, faces, F,
    pts, Bp, Q), then ``tensors`` (None is NULL) and the current stream of the points' device."""
    with torch.cuda.device(points.device):
        _cabi.check(getattr(_cabi.lib, entry)(verts.data_ptr(), verts.shape[0], verts.shape[1], faces.data_ptr(), faces.shape[0],
                                              points.data_ptr(), points.shape[0], points.shape[1],
                                              *(t.data_ptr() if t is not None else None for t in tensors), _stream_ptr(points.device)),
                    entry)


def _winding(points, verts, faces, w=None, count=None):
    _mesh_call("dvq_mesh_winding", points, verts, faces, w, count)


def _distance(points, verts, faces, B, entry="dvq_mesh_distance"):
    dist2 = torch.empty(B, points.shape[1], device=points.device, dtype=torch.float32)
    face = torch.empty(B, points.shape[1], device=points.device, dtype=torch.int64)
    _mesh_call(entry, points, verts, faces, dist2, face)
    return dist2, face


def winding_number(points, verts, faces):
    """``points [Bp,Q,3]``, ``verts [Bm,V,3]`` (fp32 CUDA; Bm, Bp each 1 or B), ``faces [F,3]`` int -> ``w [B,Q]`` fp32: the
    generalised winding number of each point with respect to its batch item's mesh (1 inside and 0 outside an
    outward-oriented closed mesh; ``w >= 0.5`` is "inside").  A point outside the item's vertex box gets exactly 0.
    ``faces`` is validated on the host (a CUDA tensor is copied there)."""
    points, verts, faces, B = _prepare(points, verts, faces, "dvq.winding_number")
    w = torch.empty(B, points.shape[1], device=points.device, dtype=torch.float32)
    _winding(points, verts, faces, w=w)
    return w


def _penetration(points, verts, faces, B):
    return _distance(points, verts, faces, B, "dvq_mesh_penetration")


class _MeshDistance(torch.autograd.Function):
    """(points, verts, faces) -> (dist2, face) through ``dvq_mesh_distance`` or, with ``fused``, ``dvq_mesh_penetration``;
    the backward is ``dvq_mesh_distance_backward`` from the saved inputs and ``face``.  Its gradients are per broadcast
    item: an input given with a batch of 1 gets their sum over b, which the [B, ., 3] temporary exists for."""

    @staticmethod
    def forward(ctx, points, verts, faces, B, fused):
        dist2, face = (_penetration if fused else _distance)(points, verts, faces, B)
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(points, verts, faces, face)
        ctx.B = B
        ctx.mark_non_differentiable(face)
        return dist2, face

    @staticmethod
    @once_differentiable
    def backward(ctx, g_dist2, _g_face):
        points, verts, faces, face = ctx.saved_tensors
        want_pts, want_verts = ctx.needs_input_grad[:2]
        if g_dist2 is None or not (want_pts or want_verts):
            return None, None, None, None, None
        B, Q, V = ctx.B, points.shape[1], verts.shape[1]
        g = g_dist2.to(torch.float32).contiguous()
        g_pts = torch.empty(B, Q, 3, device=points.device, dtype=torch.float32) if want_pts else None
        g_verts = torch.empty(B, V, 3, device=verts.device, dtype=torch.float32) if want_verts else None
        _mesh_call("dvq_mesh_distance_backward", points, verts, faces, face, g, g_pts, g_verts)
        if g_pts is not None and points.shape[0] != B:
            g_pts = g_pts.sum(0, keepdim=True)
        if g_verts is not None and verts.shape[0] != B:
            g_verts = g_verts.sum(0, keepdim=True)
        return g_pts, g_verts, None, None, None


def point_mesh_distance(points, verts, faces, differentiable=False):
    """``points [Bp,Q,3]``, ``verts [Bm,V,3]`` (fp32 CUDA; Bm, Bp each 1 or B), ``faces [F,3]`` int, F > 0 -> ``(dist2 [B,Q]
    fp32, face [B,Q] int64)``: the squared distance from each point to the closest point of its batch item's mesh and the
    closest face (the lowest index among exact ties).  ``faces`` is validated on the host.

    By default the inputs are detached.  With ``differentiable=True``, ``dist2`` carries gradients to ``points`` and
    ``verts`` (the closest point's barycentrics held fixed; deterministic); ``face`` is not differentiable.  An input
    given with a batch of 1 gets the sum over b of the per-item gradients (the same bits autograd gives an explicit
    ``expand``)."""
    points, verts, faces, B = _prepare(points, verts, faces, "dvq.point_mesh_distance", detach=not differentiable)
    if faces.shape[0] == 0:
        raise ValueError("faces must hold at least one face")
    if not differentiable:
        return _distance(points, verts, faces, B)
    return _MeshDistance.apply(points, verts, faces, B, False)


def penetration_depth(points, verts, faces):
    """``points [Bp,Q,3]``, ``verts [Bm,V,3]`` (fp32 CUDA; Bm, Bp each 1 or B), ``faces [F,3]`` int, F > 0 -> ``(depth2
    [B,Q] fp32, face [B,Q] int64)``: for a point inside its batch item's mesh (winding number >= 0.5), the squared distance
    to the mesh and the closest face, exactly as ``point_mesh_distance`` gives them; 0 and -1 for any other point.  One
    launch: the distance sweep runs only for the inside points.

    ``depth2`` is differentiable with respect to ``points`` and ``verts`` like ``point_mesh_distance(...,
    differentiable=True)``; the inside test (a step function) has no gradient.  Hand vertices [B,778,3] against an object
    mesh [1,V,3] give ``sqrt(depth2).amax(1)`` = ``GraspQuality``'s depth; an object's points or ``GraspQuality.centres``
    [1,M,3] against the hand meshes [B,778,3] with ``ManoLayer.faces`` (open at the wrist: the winding rule handles it)
    give, summed over the points, a differentiable counterpart of the penetration volume."""
    points, verts, faces, B = _prepare(points, verts, faces, "dvq.penetration_depth", detach=False)
    if faces.shape[0] == 0:
        raise ValueError("faces must hold at least one face")
    return _MeshDistance.apply(points, verts, faces, B, True)


def voxel_grid(lo, hi, pitch):
    """Grid sizing rule: ``n = max(1, ceil((hi - lo) / pitch))`` cells per axis, from the fp32 box ``lo``, ``hi`` and the fp32
    pitch (the quotient taken in float64).  Raises ``ValueError`` above ``MAX_CELLS`` cells."""
    lo, hi, p = np.asarray(lo, np.float32), np.asarray(hi, np.float32), np.float32(pitch)
    if not (np.isfinite(p) and p > 0):
        raise ValueError("pitch must be a positive finite number; got %r" % (pitch,))
    if not (np.all(np.isfinite(lo)) and np.all(np.isfinite(hi))):
        raise ValueError("the object's vertices must be finite")
    n = [max(1, int(math.ceil((float(h) - float(l)) / float(p)))) for l, h in zip(lo, hi)]
    cells = n[0] * n[1] * n[2]
    if cells > MAX_CELLS:
        raise ValueError("pitch %g gives a %d x %d x %d grid (%d cells, above the cap of %d): is the pitch in the mesh's units?"
                         % (float(p), n[0], n[1], n[2], cells, MAX_CELLS))
    return n


class GraspQuality(nn.Module):
    """Penetration volume, penetration depth and contact of a batch of hands against one object mesh.

    ``obj_verts [V,3]`` fp32 CUDA and ``obj_faces [F,3]`` int: the object (an outward-oriented closed mesh, in the frame the
    hands are given in).  ``hand_faces [Fh,3]`` int: the hand's triangles (``dvq.ManoLayer.faces`` works).  ``pitch``: the
    voxel size, in mesh units; ``contact_tol``: the contact distance, in mesh units.

    At construction the object's voxel centres (see ``csrc/mesh_exact.cuh``) are built on the GPU with the winding kernel
    and kept, with the meshes, as buffers that move with ``.to()``.  ``forward(hand_verts [B,Vh,3]) -> (volume [B] fp32,
    depth [B] fp32, contact [B] bool)``:

    - ``volume[b]`` = (voxel centres of the object inside hand b) x pitch^3, in mesh units cubed;
    - ``depth[b]`` = the largest distance to the object's surface of a hand vertex inside the object (0 if none);
    - ``contact[b]`` = some hand vertex is inside the object or within ``contact_tol`` of its surface.

    The forward is three kernel launches and a few device-side reductions, with no host synchronisation (CUDA-graph
    capturable).  No autograd."""

    def __init__(self, obj_verts, obj_faces, hand_faces, pitch, contact_tol):
        super().__init__()
        if not isinstance(obj_verts, torch.Tensor):
            raise TypeError("obj_verts must be a torch.Tensor")
        if obj_verts.dtype != torch.float32:
            raise TypeError("obj_verts must be fp32; got %s" % obj_verts.dtype)
        if obj_verts.dim() != 2 or obj_verts.shape[1] != 3 or obj_verts.shape[0] == 0:
            raise ValueError("obj_verts must be [V, 3] with V > 0; got %s" % (tuple(obj_verts.shape),))
        of = check_faces(obj_faces, obj_verts.shape[0], "obj_faces")
        if of.shape[0] == 0:
            raise ValueError("obj_faces must hold at least one face")
        hf = check_faces(hand_faces, None, "hand_faces")
        if hf.shape[0] == 0:
            raise ValueError("hand_faces must hold at least one face")
        self.num_hand_verts = int(hf.max()) + 1              # a hand must have at least this many vertices
        tol = float(contact_tol)
        if not (math.isfinite(tol) and tol >= 0):
            raise ValueError("contact_tol must be a finite number >= 0; got %r" % (contact_tol,))
        self.pitch = float(np.float32(pitch))
        self.contact_tol = tol
        self.contact_tol2 = float(np.float32(np.float32(tol) * np.float32(tol)))
        host = obj_verts.detach().cpu().numpy()
        lo, hi = host.min(0), host.max(0)
        self.grid = voxel_grid(lo, hi, pitch)
        ov = _points(obj_verts[None], "obj_verts", "dvq.GraspQuality")
        dev = ov.device
        self.register_buffer("obj_verts", ov.clone(), persistent=False)
        self.register_buffer("obj_faces", torch.from_numpy(of).to(dev), persistent=False)
        self.register_buffer("hand_faces", torch.from_numpy(hf).to(dev), persistent=False)
        self.register_buffer("centres", self._voxel_centres(torch.from_numpy(lo).to(dev)), persistent=False)

    @torch.no_grad()
    def _voxel_centres(self, lo, chunk=1 << 22):
        """fp32 centres [1, M, 3] of the grid cells whose centre is inside the object, in (i, j, k) order, k fastest."""
        nx, ny, nz = self.grid
        p = torch.tensor(self.pitch, dtype=torch.float32, device=lo.device)
        half = torch.tensor(0.5, dtype=torch.float32, device=lo.device)
        kept = []
        for c0 in range(0, nx * ny * nz, chunk):
            cell = torch.arange(c0, min(c0 + chunk, nx * ny * nz), device=lo.device, dtype=torch.int64)
            ijk = torch.stack([cell // (ny * nz), cell // nz % ny, cell % nz], 1).to(torch.float32)   # exact: < 2^24
            c = (lo + (ijk + half) * p).contiguous()[None]        # fl(lo + fl((i + 0.5) pitch)): two rounded ops
            w = torch.empty(1, c.shape[1], device=lo.device, dtype=torch.float32)
            _winding(c, self.obj_verts, self.obj_faces, w=w)
            kept.append(c[0][w[0] >= 0.5])
        return torch.cat(kept)[None].contiguous()

    @property
    def num_voxels(self):
        return self.centres.shape[1]

    def forward(self, hand_verts):
        hand = _points(hand_verts, "hand_verts", "dvq.GraspQuality")
        if self.obj_verts.device != hand.device:
            raise ValueError("the module is on %s, hand_verts on %s: move it with .to(device)" % (self.obj_verts.device, hand.device))
        B, Vh = hand.shape[0], hand.shape[1]
        if Vh < self.num_hand_verts:
            raise ValueError("hand_faces reach vertex %d, the hands have Vh = %d" % (self.num_hand_verts - 1, Vh))
        dev = hand.device
        count = torch.zeros(B, device=dev, dtype=torch.int32)
        _winding(self.centres, hand, self.hand_faces, count=count)                     # object voxels inside each hand
        w = torch.empty(B, Vh, device=dev, dtype=torch.float32)
        _winding(hand, self.obj_verts, self.obj_faces, w=w)                             # hand vertices inside the object
        dist2, _ = _distance(hand, self.obj_verts, self.obj_faces, B)
        inside = w >= 0.5
        volume = (count.to(torch.float64) * self.pitch ** 3).to(torch.float32)
        depth = torch.where(inside, dist2.sqrt(), torch.zeros((), device=dev)).amax(1)
        contact = (inside | (dist2 <= self.contact_tol2)).any(1)
        return volume, depth, contact

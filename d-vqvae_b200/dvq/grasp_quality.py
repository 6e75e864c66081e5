"""Grasp scoring on the GPU: penetration volume, penetration depth and contact of a batch of hands against one object mesh,
the metrics the reference scripts compute per grasp on the CPU (``intersection_eval`` in ``gen_diverse_grasp_obman.py``:
trimesh voxelisation and containment, igl distances).

- ``winding_number(points, verts, faces)``: generalised winding numbers (``w >= 0.5`` is "inside").
- ``point_mesh_distance(points, verts, faces)``: squared distance to the mesh and the closest face.
- ``GraspQuality(obj_verts, obj_faces, hand_faces, pitch, contact_tol)``: ``forward(hand_verts) -> (volume, depth,
  contact)``.

The contract (winding number, box rule, distance, tie rule, voxel centres, metrics) is stated once in
``csrc/mesh_exact.cuh`` and restated in float64 in ``oracle/mesh_oracle.py``.  CUDA fp32 only, no autograd: the metrics are
step functions and maxima used for scoring, so inputs that require grad are detached.

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

from . import _cabi
from .quantizer import _stream_ptr

MAX_CELLS = 1 << 24         # voxel grid cap: above it the pitch is almost certainly a unit mistake (mm vs m)


def _points(x, name, what):
    if not isinstance(x, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if x.dtype != torch.float32:
        raise TypeError("%s must be fp32; got %s" % (name, x.dtype))
    if not x.is_cuda:
        raise ValueError("%s has no CPU path: %s must be a CUDA tensor" % (what, name))
    if x.dim() != 3 or x.shape[2] != 3:
        raise ValueError("%s must be [B, n, 3]; got %s" % (name, tuple(x.shape)))
    return x.detach().contiguous()


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


def _prepare(points, verts, faces, what):
    points, verts = _points(points, "points", what), _points(verts, "verts", what)
    if points.device != verts.device:
        raise ValueError("points are on %s, verts on %s" % (points.device, verts.device))
    if verts.shape[1] == 0:
        raise ValueError("verts must hold at least one vertex per batch item")
    f = torch.from_numpy(check_faces(faces, verts.shape[1])).to(verts.device)
    return points, verts, f, _broadcast(verts.shape[0], points.shape[0])


def _winding(points, verts, faces, w=None, count=None):
    with torch.cuda.device(points.device):
        _cabi.check(_cabi.lib.dvq_mesh_winding(verts.data_ptr(), verts.shape[0], verts.shape[1], faces.data_ptr(), faces.shape[0],
                                               points.data_ptr(), points.shape[0], points.shape[1],
                                               w.data_ptr() if w is not None else None, count.data_ptr() if count is not None else None,
                                               _stream_ptr(points.device)), "dvq_mesh_winding")


def _distance(points, verts, faces, B):
    dist2 = torch.empty(B, points.shape[1], device=points.device, dtype=torch.float32)
    face = torch.empty(B, points.shape[1], device=points.device, dtype=torch.int64)
    with torch.cuda.device(points.device):
        _cabi.check(_cabi.lib.dvq_mesh_distance(verts.data_ptr(), verts.shape[0], verts.shape[1], faces.data_ptr(), faces.shape[0],
                                                points.data_ptr(), points.shape[0], points.shape[1], dist2.data_ptr(), face.data_ptr(),
                                                _stream_ptr(points.device)), "dvq_mesh_distance")
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


def point_mesh_distance(points, verts, faces):
    """``points [Bp,Q,3]``, ``verts [Bm,V,3]`` (fp32 CUDA; Bm, Bp each 1 or B), ``faces [F,3]`` int, F > 0 -> ``(dist2 [B,Q]
    fp32, face [B,Q] int64)``: the squared distance from each point to the closest point of its batch item's mesh and the
    closest face (the lowest index among exact ties).  ``faces`` is validated on the host."""
    points, verts, faces, B = _prepare(points, verts, faces, "dvq.point_mesh_distance")
    if faces.shape[0] == 0:
        raise ValueError("faces must hold at least one face")
    return _distance(points, verts, faces, B)


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

"""Hand-object nearest-point search for grasp refinement (GraspTTA / ``TTT_loss``): the pytorch3d pieces the reference's
losses stand on, as CUDA kernels.

- ``nearest_points(src, trg)`` replaces ``get_NN`` (``utils/utils_loss.py:7-24``, ``knn_points(..., K=1)``): batched 1-NN
  with the squared distance, differentiable with respect to both point sets.
- ``HandObjectContact(faces)`` runs the object -> hand search together with the reference's interior test
  (``utils/loss.py:144-167``): the area-weighted vertex normals of ``Meshes.verts_normals_packed`` and "the offset from an
  object point to its nearest hand vertex points along that vertex's normal".

Nothing is materialised: the [B, N1, N2] distance tensor of a plain-torch search (38 GB per direction at the grasp batch of
4096) never exists, and the backward keeps only the inputs and ``idx``.  The exact FP32 arithmetic is stated once in
``csrc/contact_exact.cuh``.  CUDA fp32 only; one neighbour (K = 1), dense batches (no ragged ``lengths``), no gradient through
the normals, which the interior mask (a step function) does not need.
"""
from __future__ import annotations

import numpy as np
import torch
from torch import nn
from torch.autograd.function import once_differentiable

from . import _cabi
from .quantizer import _stream_ptr


def _points(x, name):
    if not isinstance(x, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor" % name)
    if x.dtype != torch.float32:
        raise TypeError("%s must be fp32; got %s" % (name, x.dtype))
    if not x.is_cuda:
        raise ValueError("dvq.nearest_points has no CPU path: %s must be a CUDA tensor" % name)
    if x.dim() != 3 or x.shape[2] != 3:
        raise ValueError("%s must be [B, n, 3]; got %s" % (name, tuple(x.shape)))
    return x.contiguous()


class _NearestPoints(torch.autograd.Function):
    """(src, trg[, trg_normals]) -> (dist, idx, interior or None) through ``dvq_nn_forward``; the backward is
    ``dvq_nn_backward`` from the saved src, trg and idx, with NULL for a gradient nobody needs."""

    @staticmethod
    def forward(ctx, src, trg, trg_normals):
        B, N1, N2 = src.shape[0], src.shape[1], trg.shape[1]
        dev = src.device
        dist = torch.empty(B, N1, device=dev, dtype=torch.float32)
        idx = torch.empty(B, N1, device=dev, dtype=torch.int64)
        interior = torch.empty(B, N1, device=dev, dtype=torch.bool) if trg_normals is not None else None
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib.dvq_nn_forward(src.data_ptr(), trg.data_ptr(), B, N1, N2,
                                                 trg_normals.data_ptr() if trg_normals is not None else None, dist.data_ptr(),
                                                 idx.data_ptr(), interior.data_ptr() if interior is not None else None,
                                                 _stream_ptr(dev)), "dvq_nn_forward")
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(src, trg, idx)
        ctx.mark_non_differentiable(idx, *([interior] if interior is not None else []))
        return dist, idx, interior

    @staticmethod
    @once_differentiable
    def backward(ctx, g_dist, _g_idx, _g_interior):
        src, trg, idx = ctx.saved_tensors
        want_src, want_trg, _ = ctx.needs_input_grad
        if g_dist is None or not (want_src or want_trg):
            return None, None, None
        g = g_dist.to(torch.float32).contiguous()
        g_src = torch.empty_like(src) if want_src else None
        g_trg = torch.empty_like(trg) if want_trg else None
        ptr = lambda t: t.data_ptr() if t is not None else None
        with torch.cuda.device(src.device):
            _cabi.check(_cabi.lib.dvq_nn_backward(src.data_ptr(), trg.data_ptr(), idx.data_ptr(), g.data_ptr(), src.shape[0],
                                                  src.shape[1], trg.shape[1], ptr(g_src), ptr(g_trg), _stream_ptr(src.device)),
                        "dvq_nn_backward")
        return g_src, g_trg, None


def _search(src, trg, trg_normals=None):
    src, trg = _points(src, "src"), _points(trg, "trg")
    if src.device != trg.device:
        raise ValueError("src is on %s, trg on %s" % (src.device, trg.device))
    if src.shape[0] != trg.shape[0]:
        raise ValueError("src and trg must have the same batch size; got %d and %d" % (src.shape[0], trg.shape[0]))
    if trg.shape[1] == 0:
        raise ValueError("trg must hold at least one point per batch item")
    return _NearestPoints.apply(src, trg, trg_normals)


def nearest_points(src, trg):
    """``src [B,N1,3]``, ``trg [B,N2,3]`` (fp32 CUDA) -> ``(dist [B,N1] fp32, idx [B,N1] int64)``: for every src point of
    batch item b, the squared Euclidean distance to the nearest trg point of item b and that point's index (the lowest index
    among exact ties), as ``knn_points(src, trg, K=1)`` returns them without the K axis.  ``dist`` is differentiable with
    respect to both inputs; the backward is deterministic.  Non-contiguous inputs are copied to contiguous ones."""
    dist, idx, _ = _search(src, trg)
    return dist, idx


class HandObjectContact(nn.Module):
    """Object -> hand nearest points with the penetration mask of GraspTTA's ``TTT_loss``.

    ``faces`` is the hand mesh's triangle list, int ``[F,3]`` (``dvq.ManoLayer.faces`` works).  It is validated on the host
    here; the vertex -> face lists of the normal computation are built once and kept with ``faces`` as int32 buffers, so
    ``.to(device)`` moves them.  ``forward(hand_verts [B,V,3], obj_pts [B,P,3])`` returns ``(dist [B,P], idx [B,P],
    interior [B,P] bool)``: the squared distance from each object point to its nearest hand vertex, that vertex's index,
    and whether the offset from the object point to that vertex points along the vertex's area-weighted normal (the
    object point is inside the hand).  ``dist`` is differentiable with respect to both inputs; the normals are taken of
    ``hand_verts.detach()``, since the mask is a step function without a gradient."""

    def __init__(self, faces):
        super().__init__()
        f = np.asarray(faces.detach().cpu() if isinstance(faces, torch.Tensor) else faces)
        if f.dtype.kind not in "iu":
            raise TypeError("faces must be an integer array; got %s" % f.dtype)
        if f.ndim != 2 or f.shape[1] != 3:
            raise ValueError("faces must be [F, 3]; got %s" % (f.shape,))
        if f.size and (f.min() < 0 or f.max() >= 2 ** 31 - 1):
            raise ValueError("face vertex ids must be in [0, V)")
        f = f.astype(np.int64)
        self.num_verts = int(f.max()) + 1 if f.size else 0     # the hand must have at least this many vertices
        offsets, vf_faces = vertex_face_csr(f, self.num_verts)
        self.register_buffer("faces", torch.from_numpy(f.astype(np.int32)), persistent=False)
        self.register_buffer("vf_offsets", torch.from_numpy(offsets), persistent=False)
        self.register_buffer("vf_faces", torch.from_numpy(vf_faces), persistent=False)

    def vertex_normals(self, verts):
        B, V = verts.shape[0], verts.shape[1]
        if V < self.num_verts:
            raise ValueError("face vertex ids must be in [0, V): faces reach vertex %d, the hand has V = %d" % (self.num_verts - 1, V))
        offsets = self.vf_offsets
        if V > self.num_verts:       # vertices past the last one a face lists have no faces
            offsets = torch.cat([offsets, offsets[-1:].expand(V - self.num_verts)])
        normals = torch.empty_like(verts)
        with torch.cuda.device(verts.device):
            _cabi.check(_cabi.lib.dvq_vertex_normals(verts.data_ptr(), B, V, self.faces.data_ptr(), self.faces.shape[0],
                                                     offsets.data_ptr(), self.vf_faces.data_ptr(), normals.data_ptr(),
                                                     _stream_ptr(verts.device)), "dvq_vertex_normals")
        return normals

    def forward(self, hand_verts, obj_pts):
        hand = _points(hand_verts, "hand_verts")
        if self.faces.device != hand.device:
            raise ValueError("the module is on %s, hand_verts on %s: move it with .to(device)" % (self.faces.device, hand.device))
        normals = self.vertex_normals(hand.detach())
        return _search(obj_pts, hand, normals)


def vertex_face_csr(faces, num_verts):
    """CSR of the faces that list each vertex: ``offsets [V+1]`` int32 and ``vf_faces`` int32, ascending face index per
    vertex, one entry per occurrence (a face that lists a vertex twice appears twice)."""
    flat = np.asarray(faces, dtype=np.int64).reshape(-1)
    order = np.argsort(flat, kind="stable")                    # occurrences are face-major, so each vertex's run ascends in f
    counts = np.bincount(flat, minlength=num_verts)
    offsets = np.zeros(num_verts + 1, dtype=np.int32)
    np.cumsum(counts, out=offsets[1:])
    return offsets, (order // 3).astype(np.int32)

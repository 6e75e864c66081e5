"""``dvq.ManoLayer`` — the MANO hand layer the reference calls at network/gen_net.py:116-118

    recon_mano = self.rh_mano(betas=recon[:, :10], global_orient=zero_params, hand_pose=recon[:, 10:55],
                              transl=zero_params).vertices                                   # [B, 778, 3]

(created at gen_diverse_grasp_obman.py:355-360 with the third-party package ``mano``: ``mano.load(model_path=
'./models/mano/MANO_RIGHT.pkl', model_type='mano', use_pca=True, num_pca_comps=45, batch_size=1, flat_hand_mean=True)``)
as one CUDA kernel behind the same call signature, so ``GenNet.set_rh_mano(dvq.ManoLayer.from_pkl(...))`` is the whole
change and the decoder's 55 parameters reach the 778-point PointNet without leaving the device.  The arithmetic is the
linear blend skinning of ``smplx/lbs.py`` (which ``mano`` wraps); ``oracle/mano_oracle.py`` restates it for the tests.
CUDA tensors only.  Gradients with respect to betas, global_orient, hand_pose and transl are opt-in
(``ManoLayer(..., differentiable=True)``): a second kernel, ``dvq_mano_backward``, computes the vector-Jacobian product.
"""
from __future__ import annotations

import ctypes as C
import pickle
import sys
import types
from types import SimpleNamespace

import numpy as np
import torch
from torch import nn
from torch.autograd.function import once_differentiable

from . import _cabi
from .quantizer import _stream_ptr

_TREE = (-1, 0, 1, 2, 0, 4, 5, 0, 7, 8, 0, 10, 11, 0, 13, 14)    # MANO's kinematic tree: five three-joint fingers off the wrist


def read_mano_pkl(path):
    """MANO_{LEFT,RIGHT}.pkl -> dict of numpy arrays.  The file pickles ``chumpy`` objects; they are read through stand-in
    classes, so the (unmaintained) package is not needed."""
    class Ch:
        def __setstate__(self, st):
            self.__dict__.update(st if isinstance(st, dict) else {"state": st})

    names = ("chumpy", "chumpy.ch", "chumpy.reordering", "chumpy.ch_ops", "chumpy.logic", "chumpy.utils")
    saved = {k: sys.modules.get(k) for k in names}
    try:
        for name in names:
            m = types.ModuleType(name)
            m.Ch = Ch
            m.__getattr__ = lambda n, _C=Ch: type(n, (_C,), {})
            sys.modules[name] = m
        with open(path, "rb") as f:
            d = pickle.load(f, encoding="latin1")
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v

    def arr(v):
        if isinstance(v, np.ndarray):
            return np.asarray(v, dtype=np.float64)
        if hasattr(v, "toarray"):
            return np.asarray(v.toarray(), dtype=np.float64)
        st = v.__dict__
        if "x" in st:
            return np.asarray(st["x"], dtype=np.float64)
        if "a" in st and "idxs" in st:
            return arr(st["a"]).ravel()[np.asarray(st["idxs"])]
        raise TypeError("unsupported object in the MANO pickle: %r" % (v,))

    return {"v_template": arr(d["v_template"]), "shapedirs": arr(d["shapedirs"]), "posedirs": arr(d["posedirs"]),
            "J_regressor": arr(d["J_regressor"]), "weights": arr(d["weights"]), "hands_components": arr(d["hands_components"]),
            "hands_mean": arr(d["hands_mean"]), "parents": np.asarray(d["kintree_table"])[0].astype(np.int64),
            "faces": np.asarray(d["f"]).astype(np.int64)}


class _ManoLBS(torch.autograd.Function):
    """(betas, global_orient, hand_pose, transl) -> (vertices, joints) through ``dvq_mano_forward``.  The backward is
    ``dvq_mano_backward``: it recomputes the forward intermediates from the saved inputs, so nothing else is kept.  The inputs
    arrive as contiguous fp32 tensors; global_orient and transl may be None."""

    @staticmethod
    def forward(ctx, layer, betas, global_orient, hand_pose, transl):
        ctx.layer = layer
        ctx.set_materialize_grads(False)          # an unused output gives None: the kernel reads NULL as zero
        ctx.save_for_backward(betas, global_orient, hand_pose)
        return layer._launch_forward(betas, global_orient, hand_pose, transl)

    @staticmethod
    @once_differentiable
    def backward(ctx, g_vertices, g_joints):
        betas, global_orient, hand_pose = ctx.saved_tensors
        layer = ctx.layer
        _, want_betas, want_orient, want_pose, want_transl = ctx.needs_input_grad
        B, dev = betas.shape[0], betas.device
        new = lambda cols, want: torch.empty(B, cols, device=dev, dtype=torch.float32) if want else None
        g_betas, g_orient, g_pose, g_transl = new(10, want_betas), new(3, want_orient), new(hand_pose.shape[1], want_pose), new(3, want_transl)
        gv = g_vertices.to(torch.float32).contiguous() if g_vertices is not None else None
        gj = g_joints.to(torch.float32).contiguous() if g_joints is not None else None
        ptr = lambda t: t.data_ptr() if t is not None else None
        m = layer._model_struct()
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib.dvq_mano_backward(C.byref(m), betas.data_ptr(), ptr(global_orient), hand_pose.data_ptr(), B,
                                                    ptr(gv), ptr(gj), ptr(g_betas), ptr(g_orient), ptr(g_pose), ptr(g_transl),
                                                    _stream_ptr(dev)), "dvq_mano_backward")
        return None, g_betas, g_orient, g_pose, g_transl


class ManoLayer(nn.Module):
    """MANO linear blend skinning: ``layer(betas=[B,10], global_orient=[B,3], hand_pose=[B,ncomps], transl=[B,3])`` returns an
    object with ``.vertices [B,778,3]`` and ``.joints [B,16,3]`` (the posed joints of the kinematic tree).

    ``differentiable=False`` (the default) detaches the inputs: the outputs never carry a ``grad_fn``.  That keeps the drop-in
    flow working where the hand parameters come out of a decoder that requires grad (``GenNet.gen`` outside ``no_grad``):
    the vertices feed ``dvq.PointNetEncoder``, which refuses an input that requires grad.  With ``differentiable=True``, a
    call in grad mode where some input requires grad returns vertices and joints with gradients to betas, global_orient,
    hand_pose and transl (fp32 arithmetic; each gradient comes back in its input's dtype), e.g. for test-time refinement of a
    grasp with Adam.  Every other call runs the same inference path as the default."""

    def __init__(self, model: dict, use_pca: bool = True, num_pca_comps: int = 45, flat_hand_mean: bool = True,
                 differentiable: bool = False):
        super().__init__()
        self.differentiable = bool(differentiable)
        nv = 778
        f32 = lambda a, shape: torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(shape), dtype=np.float32))
        parents = np.asarray(model["parents"]).astype(np.int64).copy()
        parents[0] = -1
        if tuple(int(p) for p in parents) != _TREE:
            raise ValueError("unexpected kinematic tree %s (the kernel walks MANO's five three-joint finger chains)" % (parents,))
        if not 1 <= num_pca_comps <= 45:
            raise ValueError("num_pca_comps must be in [1, 45]")
        self.use_pca, self.num_pca_comps, self.flat_hand_mean = bool(use_pca), int(num_pca_comps), bool(flat_hand_mean)
        self.register_buffer("v_template", f32(model["v_template"], (nv * 3,)), persistent=False)
        self.register_buffer("shapedirs", f32(np.asarray(model["shapedirs"]).reshape(nv * 3, 10).T, (10, nv * 3)), persistent=False)
        self.register_buffer("posedirs", f32(np.asarray(model["posedirs"]).reshape(nv * 3, 135).T, (135, nv * 3)), persistent=False)
        self.register_buffer("j_regressor", f32(model["J_regressor"], (16, nv)), persistent=False)
        self.register_buffer("weights", f32(model["weights"], (nv, 16)), persistent=False)
        self.register_buffer("hands_components", f32(np.asarray(model["hands_components"])[:num_pca_comps], (num_pca_comps, 45)), persistent=False)
        mean = np.zeros(48)
        if not flat_hand_mean:
            mean[3:] = np.asarray(model["hands_mean"], dtype=np.float64)
        self.register_buffer("pose_mean", f32(mean, (48,)), persistent=False)
        self.register_buffer("parents", torch.tensor([0] + list(_TREE[1:]), dtype=torch.int32), persistent=False)
        self.faces = np.asarray(model.get("faces", np.zeros((0, 3))), dtype=np.int64)

    @classmethod
    def from_pkl(cls, model_path, use_pca=True, num_pca_comps=45, flat_hand_mean=True, differentiable=False, **_ignored):
        """Same keyword arguments as ``mano.load`` (``model_type``, ``batch_size`` ... are accepted and ignored), plus
        ``differentiable``."""
        return cls(read_mano_pkl(model_path), use_pca=use_pca, num_pca_comps=num_pca_comps, flat_hand_mean=flat_hand_mean,
                   differentiable=differentiable)

    def _model_struct(self):
        return _cabi.ManoModel(self.v_template.data_ptr(), self.shapedirs.data_ptr(), self.posedirs.data_ptr(), self.j_regressor.data_ptr(),
                               self.weights.data_ptr(), self.hands_components.data_ptr(), self.pose_mean.data_ptr(), self.parents.data_ptr(),
                               self.num_pca_comps if self.use_pca else 0)

    def _launch_forward(self, betas, global_orient, hand_pose, transl):
        dev, B = betas.device, betas.shape[0]
        vertices = torch.empty(B, 778, 3, device=dev, dtype=torch.float32)
        joints = torch.empty(B, 16, 3, device=dev, dtype=torch.float32)
        m = self._model_struct()
        with torch.cuda.device(dev):
            _cabi.check(_cabi.lib.dvq_mano_forward(C.byref(m), betas.data_ptr(), global_orient.data_ptr() if global_orient is not None else None,
                                                   hand_pose.data_ptr(), transl.data_ptr() if transl is not None else None, B,
                                                   vertices.data_ptr(), joints.data_ptr(), _stream_ptr(dev)), "dvq_mano_forward")
        return vertices, joints

    def forward(self, betas=None, global_orient=None, hand_pose=None, transl=None, **_ignored):
        dev = self.v_template.device
        if dev.type != "cuda":
            raise ValueError("dvq.ManoLayer has no CPU path: move the layer and its inputs to a CUDA device")
        ncols = self.num_pca_comps if self.use_pca else 45
        if hand_pose is None and betas is None:
            raise ValueError("need betas or hand_pose to infer the batch size")
        B = int((betas if betas is not None else hand_pose).shape[0])
        grad = self.differentiable and torch.is_grad_enabled() and any(
            t is not None and t.requires_grad for t in (betas, global_orient, hand_pose, transl))

        def prep(t, cols, name):
            if t is None:
                return None
            if t.device != dev:
                raise ValueError("%s is on %s, the layer on %s" % (name, t.device, dev))
            if tuple(t.shape) != (B, cols):
                raise RuntimeError("%s must be [%d, %d], got %s" % (name, B, cols, tuple(t.shape)))
            # the differentiable path casts in the graph, so each gradient comes back in its input's dtype
            return (t if grad else t.detach()).to(torch.float32).contiguous()

        betas = prep(betas, 10, "betas") if betas is not None else torch.zeros(B, 10, device=dev)
        hand_pose = prep(hand_pose, ncols, "hand_pose") if hand_pose is not None else torch.zeros(B, ncols, device=dev)
        global_orient = prep(global_orient, 3, "global_orient")
        transl = prep(transl, 3, "transl")
        if grad:
            vertices, joints = _ManoLBS.apply(self, betas, global_orient, hand_pose, transl)
        else:
            vertices, joints = self._launch_forward(betas, global_orient, hand_pose, transl)
        return SimpleNamespace(vertices=vertices, joints=joints)

"""Torch restatement of the MANO forward (linear blend skinning) with the op sequence of ``smplx/lbs.py``, which the
third-party ``mano`` package wraps; differentiable through autograd.  Two roles: in float64 on the CPU its autograd gradients
are the reference of ``dvq.ManoLayer(differentiable=True)`` (tests/test_mano_grad.py); in float32 on the GPU it is what a
``mano`` / ``smplx`` layer launches, the baseline arm of scripts/bench_mano_grad.py.  tests/test_mano_grad.py pins it to the
float64 numpy oracle (``oracle/mano_oracle.py`` ``mano_forward``) to 1e-12."""
import numpy as np
import torch
import torch.nn.functional as F

from oracle.mano_oracle import N_BETAS, N_JOINTS, N_POSE, N_VERTS


def _torch_batch_rodrigues(rot_vecs):
    """smplx.lbs.batch_rodrigues, op for op: [n,3] -> [n,3,3]."""
    n = rot_vecs.shape[0]
    angle = torch.norm(rot_vecs + 1e-8, dim=1, keepdim=True)
    rot_dir = rot_vecs / angle
    cos = torch.unsqueeze(torch.cos(angle), dim=1)
    sin = torch.unsqueeze(torch.sin(angle), dim=1)
    rx, ry, rz = torch.split(rot_dir, 1, dim=1)
    zeros = torch.zeros((n, 1), dtype=rot_vecs.dtype, device=rot_vecs.device)
    K = torch.cat([zeros, -rz, ry, rz, zeros, -rx, -ry, rx, zeros], dim=1).view((n, 3, 3))
    ident = torch.eye(3, dtype=rot_vecs.dtype, device=rot_vecs.device).unsqueeze(dim=0)
    return ident + sin * K + (1 - cos) * torch.bmm(K, K)


def torch_model(model, dtype, device):
    """The model's tables as torch tensors in smplx's layouts (the buffers a `mano` / `smplx` layer keeps on its device)."""
    tab = lambda a, *shape: torch.as_tensor(np.asarray(a, dtype=np.float64).reshape(shape), dtype=dtype, device=device)
    return {"v_template": tab(model["v_template"], N_VERTS, 3), "shapedirs": tab(model["shapedirs"], N_VERTS, 3, N_BETAS),
            "posedirs": tab(np.asarray(model["posedirs"]).reshape(-1, 9 * (N_JOINTS - 1)).T, 9 * (N_JOINTS - 1), 3 * N_VERTS),
            "J_regressor": tab(model["J_regressor"], N_JOINTS, N_VERTS), "weights": tab(model["weights"], N_VERTS, N_JOINTS),
            "hands_components": tab(model["hands_components"], N_POSE, N_POSE), "hands_mean": tab(model["hands_mean"], N_POSE),
            "parents": [int(p) for p in model["parents"]]}


def mano_forward_torch(model, betas, global_orient=None, hand_pose=None, transl=None, use_pca=True, num_pca_comps=45,
                       flat_hand_mean=True):
    """`mano_forward` in torch (smplx/lbs.py's op sequence, differentiable).  betas [B,10] sets the dtype and device; `model`
    is a numpy model (converted on each call) or the output of `torch_model`.  -> (vertices [B,778,3], joints [B,16,3])."""
    dt, dev = betas.dtype, betas.device
    tm = model if torch.is_tensor(model["v_template"]) else torch_model(model, dt, dev)
    B = betas.shape[0]
    go = torch.zeros(B, 3, dtype=dt, device=dev) if global_orient is None else global_orient
    hp = torch.zeros(B, num_pca_comps if use_pca else N_POSE, dtype=dt, device=dev) if hand_pose is None else hand_pose
    if use_pca:
        hp = torch.einsum("bi,ij->bj", hp, tm["hands_components"][:num_pca_comps])
    full_pose = torch.cat([go, hp], dim=1)
    if not flat_hand_mean:
        full_pose = full_pose + torch.cat([torch.zeros(3, dtype=dt, device=dev), tm["hands_mean"]])
    # smplx.lbs.lbs
    v_shaped = tm["v_template"] + torch.einsum("bl,mkl->bmk", betas, tm["shapedirs"])
    J = torch.einsum("bik,ji->bjk", v_shaped, tm["J_regressor"])
    ident = torch.eye(3, dtype=dt, device=dev)
    rot_mats = _torch_batch_rodrigues(full_pose.reshape(-1, 3)).view(B, -1, 3, 3)
    pose_feature = (rot_mats[:, 1:, :, :] - ident).view(B, -1)
    v_posed = torch.matmul(pose_feature, tm["posedirs"]).view(B, -1, 3) + v_shaped
    # smplx.lbs.batch_rigid_transform
    parents = tm["parents"]
    joints = torch.unsqueeze(J, dim=-1)
    rel_joints = joints.clone()
    rel_joints[:, 1:] -= joints[:, parents[1:]]
    R = rot_mats.reshape(-1, 3, 3)
    t = rel_joints.reshape(-1, 3, 1)
    transforms_mat = torch.cat([F.pad(R, [0, 0, 0, 1]), F.pad(t, [0, 0, 0, 1], value=1)], dim=2).reshape(-1, N_JOINTS, 4, 4)
    chain = [transforms_mat[:, 0]]
    for i in range(1, N_JOINTS):
        chain.append(torch.matmul(chain[parents[i]], transforms_mat[:, i]))
    transforms = torch.stack(chain, dim=1)
    posed_joints = transforms[:, :, :3, 3]
    joints_homogen = F.pad(joints, [0, 0, 0, 1])
    A = transforms - F.pad(torch.matmul(transforms, joints_homogen), [3, 0, 0, 0, 0, 0, 0, 0])
    # skinning
    W = tm["weights"].unsqueeze(dim=0).expand([B, -1, -1])
    T = torch.matmul(W, A.view(B, N_JOINTS, 16)).view(B, -1, 4, 4)
    v_posed_homo = torch.cat([v_posed, torch.ones([B, v_posed.shape[1], 1], dtype=dt, device=dev)], dim=2)
    verts = torch.matmul(T, torch.unsqueeze(v_posed_homo, dim=-1))[:, :, :3, 0]
    if transl is not None:
        verts = verts + transl.unsqueeze(dim=1)
        posed_joints = posed_joints + transl.unsqueeze(dim=1)
    return verts, posed_joints

"""MANO hand layer (SURVEY §8 f4; reference call site network/gen_net.py:116-118, layer created at
gen_diverse_grasp_obman.py:355-360 by the un-vendored package `mano`).

CPU: the oracle (oracle/mano_oracle.py, a restatement of smplx/lbs.py's published algorithm) on a synthetic model.
GPU: the CUDA kernel behind `dvq.ManoLayer` against the oracle on a synthetic model of MANO's structure (the MANO asset is
licensed separately and not part of the repository), through the reference's call signature.  Bar: 2e-6 of the hand size
(FP32 kernel vs float64 oracle).
"""
import numpy as np
import pytest
import torch

from oracle import mano_oracle as mo

TOL = 2e-6


def test_oracle_synthetic_model_sanity():
    m = mo.synthetic_model(5)
    v, j = mo.mano_forward(m, np.zeros((1, 10)), None, np.zeros((1, 45)))
    assert np.abs(v[0] - m["v_template"]).max() < 1e-12
    R = mo.rodrigues(np.random.RandomState(0).randn(7, 3))
    assert np.abs(R @ R.transpose(0, 2, 1) - np.eye(3)).max() < 1e-6 and np.abs(np.linalg.det(R) - 1).max() < 1e-6


def test_mano_layer_refuses_cpu_and_bad_trees():
    import dvq
    layer = dvq.ManoLayer(mo.synthetic_model(1))
    with pytest.raises(ValueError, match="no CPU path"):
        layer(betas=torch.zeros(1, 10), hand_pose=torch.zeros(1, 45))
    bad = mo.synthetic_model(1)
    bad["parents"] = np.arange(-1, 15)
    with pytest.raises(ValueError, match="kinematic tree"):
        dvq.ManoLayer(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("use_pca,ncomps,flat", [(True, 45, True), (True, 12, False), (False, 45, False)])
def test_mano_kernel_matches_oracle(use_pca, ncomps, flat):
    import dvq
    m = mo.synthetic_model(7)
    rs = np.random.RandomState(8)
    B = 37
    betas, go, tr = rs.randn(B, 10), rs.randn(B, 3), 0.3 * rs.randn(B, 3)
    pose = 0.8 * rs.randn(B, ncomps if use_pca else 45)
    pose[3] = 0.0
    go[3] = 0.0                                                       # a zero rotation vector (the epsilon path of rodrigues)
    rv, rj = mo.mano_forward(m, betas, go, pose, tr, use_pca=use_pca, num_pca_comps=ncomps, flat_hand_mean=flat)
    layer = dvq.ManoLayer(m, use_pca=use_pca, num_pca_comps=ncomps, flat_hand_mean=flat).cuda()
    t = lambda a: torch.from_numpy(a.astype(np.float32)).cuda()
    out = layer(betas=t(betas), global_orient=t(go), hand_pose=t(pose), transl=t(tr))
    scale = float(np.abs(rv).max())
    assert np.abs(out.vertices.cpu().numpy() - rv).max() <= TOL * max(scale, 1.0)
    assert np.abs(out.joints.cpu().numpy() - rj).max() <= TOL * max(scale, 1.0)
    # the reference's call: zero global orientation and translation (gen_net.py:116-118), passed as tensors or omitted
    z3 = torch.zeros(B, 3, device="cuda")
    a = layer(betas=t(betas), global_orient=z3, hand_pose=t(pose), transl=z3).vertices
    b = layer(betas=t(betas), hand_pose=t(pose)).vertices
    assert torch.equal(a, b)
    rv0, _ = mo.mano_forward(m, betas, None, pose, None, use_pca=use_pca, num_pca_comps=ncomps, flat_hand_mean=flat)
    assert np.abs(a.cpu().numpy() - rv0).max() <= TOL * max(float(np.abs(rv0).max()), 1.0)


@pytest.mark.gpu
def test_grasp_generator_with_the_mano_layer():
    """GraspGenerator(hand_layer=dvq.ManoLayer): the decoder's 55 parameters go through the LBS kernel into the 778-point PointNet."""
    import dvq
    torch.manual_seed(0)
    g = dvq.GraspGenerator(hand_layer=dvq.ManoLayer(mo.synthetic_model(2))).cuda().eval()
    obj = 0.1 * torch.randn(5, 4, 600, device="cuda")
    obj[:, 3] = 0.2
    recon, pos = g.gen(obj)
    assert tuple(recon.shape) == (5, 55) and tuple(pos.shape) == (5, 6) and torch.isfinite(pos).all()
    rv, _ = mo.mano_forward(mo.synthetic_model(2), recon[:, :10].cpu().numpy().astype(np.float64), None,
                            recon[:, 10:55].cpu().numpy().astype(np.float64))
    assert np.abs(g.last["verts"].cpu().numpy() - rv).max() <= 1e-5

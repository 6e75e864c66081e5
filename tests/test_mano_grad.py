"""Gradients of the MANO hand layer: ``dvq.ManoLayer(differentiable=True)`` and ``dvq_mano_backward``.

CPU: the torch restatement of the forward (tests/_mano_torch.py ``mano_forward_torch``, smplx/lbs.py's op sequence) equals
the float64 oracle; the C ABI's argument checks; the differentiable layer still has no CPU path.
GPU: the fused backward kernel against ``torch.autograd.grad`` of the float64 restatement on a synthetic model of MANO's
structure.  Bar: max |g - g_ref| <= 1e-4 max |g_ref| per gradient tensor (FP32 kernel vs float64 autograd).
"""
import ctypes

import numpy as np
import pytest
import torch

from _mano_torch import mano_forward_torch
from oracle import mano_oracle as mo

CASES = [(True, 45, True), (True, 12, False), (False, 45, False)]
REL = 1e-4
B = 37


def _inputs(use_pca, ncomps, seed=8):
    """B hands; rows 3 carry zero rotation vectors (the epsilon path of rodrigues), row 5's global orientation is an angle
    near pi (and so is one finger joint of row 6 without PCA)."""
    rs = np.random.RandomState(seed)
    betas, go, tr = rs.randn(B, 10), rs.randn(B, 3), 0.3 * rs.randn(B, 3)
    pose = 0.8 * rs.randn(B, ncomps if use_pca else 45)
    pose[3] = 0.0
    go[3] = 0.0
    axis = np.array([0.48, -0.6, 0.64])
    go[5] = (np.pi - 1e-3) * axis
    if not use_pca:
        pose[6, 3:6] = (np.pi - 2e-3) * axis[::-1]
    return betas, go, pose, tr


def _reference_grads(model, arrays, gv, gj, use_pca, ncomps, flat):
    """torch.autograd.grad of the float64 restatement on the CPU: gradients of <vertices, gv> + <joints, gj>."""
    ts = [None if a is None else torch.from_numpy(np.asarray(a, dtype=np.float64)).requires_grad_(True) for a in arrays]
    v, j = mano_forward_torch(model, *ts, use_pca=use_pca, num_pca_comps=ncomps, flat_hand_mean=flat)
    loss = (v * torch.from_numpy(gv)).sum() + (j * torch.from_numpy(gj)).sum()
    live = [t for t in ts if t is not None]
    got = iter(torch.autograd.grad(loss, live))
    return [None if t is None else next(got).numpy() for t in ts]


def _layer(model, use_pca=True, ncomps=45, flat=True, differentiable=True):
    import dvq
    return dvq.ManoLayer(model, use_pca=use_pca, num_pca_comps=ncomps, flat_hand_mean=flat, differentiable=differentiable).cuda()


def _cuda(arrays, dtype=torch.float32):
    return [None if a is None else torch.from_numpy(np.asarray(a, dtype=np.float32)).cuda().to(dtype).requires_grad_(True) for a in arrays]


def _kernel_grads(layer, ts, gv, gj):
    out = layer(betas=ts[0], global_orient=ts[1], hand_pose=ts[2], transl=ts[3])
    outs, ups = [], []
    if gv is not None:
        outs.append(out.vertices)
        ups.append(torch.from_numpy(np.asarray(gv, dtype=np.float32)).cuda())
    if gj is not None:
        outs.append(out.joints)
        ups.append(torch.from_numpy(np.asarray(gj, dtype=np.float32)).cuda())
    live = [t for t in ts if t is not None]
    got = iter(torch.autograd.grad(outs, live, ups))
    return [None if t is None else next(got) for t in ts]


def _check(got, ref, names):
    errs = {}
    for g, r, n in zip(got, ref, names):
        if r is None:
            assert g is None
            continue
        scale = float(np.abs(r).max())
        err = float(np.abs(g.double().cpu().numpy() - r).max())
        errs[n] = err / scale
        assert err <= REL * scale, (n, err, scale)
    print("relative max errors:", {k: "%.2e" % v for k, v in errs.items()})


NAMES = ("betas", "global_orient", "hand_pose", "transl")


# ---------------------------------------------------------------- CPU

@pytest.mark.parametrize("use_pca,ncomps,flat", CASES)
def test_torch_restatement_matches_oracle(use_pca, ncomps, flat):
    m = mo.synthetic_model(7)
    betas, go, pose, tr = _inputs(use_pca, ncomps)
    t = lambda a: None if a is None else torch.from_numpy(a)
    for g, tl in ((go, tr), (None, None), (go, None)):
        rv, rj = mo.mano_forward(m, betas, g, pose, tl, use_pca=use_pca, num_pca_comps=ncomps, flat_hand_mean=flat)
        v, j = mano_forward_torch(m, t(betas), t(g), t(pose), t(tl), use_pca=use_pca, num_pca_comps=ncomps, flat_hand_mean=flat)
        assert v.dtype == torch.float64
        assert np.abs(v.numpy() - rv).max() <= 1e-12 and np.abs(j.numpy() - rj).max() <= 1e-12


def test_backward_argument_errors():
    from dvq import _cabi
    buf = (ctypes.c_float * 1024)()
    p = ctypes.addressof(buf)
    p = (p + 15) // 16 * 16
    m = _cabi.ManoModel(p, p, p, p, p, p, p, p, 45)
    call = lambda model, Bn: _cabi.lib.dvq_mano_backward(model, p, None, p, Bn, p, None, p, None, None, None, None)
    assert call(ctypes.byref(m), -1) == -1 and "B must be" in _cabi.last_error()
    assert call(None, 1) == -7
    m.ncomps = 46
    assert call(ctypes.byref(m), 1) == -1 and "ncomps" in _cabi.last_error()


def test_differentiable_layer_refuses_cpu():
    import dvq
    layer = dvq.ManoLayer(mo.synthetic_model(1), differentiable=True)
    with pytest.raises(ValueError, match="no CPU path"):
        layer(betas=torch.zeros(1, 10, requires_grad=True), hand_pose=torch.zeros(1, 45, requires_grad=True))


# ---------------------------------------------------------------- GPU

@pytest.mark.gpu
@pytest.mark.parametrize("use_pca,ncomps,flat", CASES)
def test_grads_match_float64_autograd(use_pca, ncomps, flat):
    m = mo.synthetic_model(7)
    arrays = list(_inputs(use_pca, ncomps))
    rs = np.random.RandomState(9)
    gv, gj = rs.randn(B, 778, 3), rs.randn(B, 16, 3)
    layer = _layer(m, use_pca, ncomps, flat)
    ref = _reference_grads(m, arrays, gv, gj, use_pca, ncomps, flat)
    _check(_kernel_grads(layer, _cuda(arrays), gv, gj), ref, NAMES)
    # global_orient and transl omitted
    arrays[1] = arrays[3] = None
    ref = _reference_grads(m, arrays, gv, gj, use_pca, ncomps, flat)
    _check(_kernel_grads(layer, _cuda(arrays), gv, gj), ref, NAMES)


@pytest.mark.gpu
def test_vertices_only_and_joints_only_upstream():
    m = mo.synthetic_model(7)
    arrays = _inputs(True, 45)
    rs = np.random.RandomState(10)
    gv, gj = rs.randn(B, 778, 3), rs.randn(B, 16, 3)
    layer = _layer(m)
    ref = _reference_grads(m, arrays, gv, np.zeros_like(gj), True, 45, True)
    _check(_kernel_grads(layer, _cuda(arrays), gv, None), ref, NAMES)
    ref = _reference_grads(m, arrays, np.zeros_like(gv), gj, True, 45, True)
    _check(_kernel_grads(layer, _cuda(arrays), None, gj), ref, NAMES)


@pytest.mark.gpu
def test_forward_bits_and_default_contract():
    m = mo.synthetic_model(7)
    ts = _cuda(_inputs(True, 45))
    kw = dict(betas=ts[0], global_orient=ts[1], hand_pose=ts[2], transl=ts[3])
    a = _layer(m, differentiable=True)(**kw)
    b = _layer(m, differentiable=False)(**kw)
    assert a.vertices.grad_fn is not None and a.joints.grad_fn is not None
    assert torch.equal(a.vertices, b.vertices) and torch.equal(a.joints, b.joints)
    assert b.vertices.grad_fn is None and b.joints.grad_fn is None and not b.vertices.requires_grad
    with torch.no_grad():
        c = _layer(m, differentiable=True)(**kw)
    assert c.vertices.grad_fn is None and torch.equal(c.vertices, a.vertices)


@pytest.mark.gpu
def test_backward_is_deterministic_and_per_hand():
    m = mo.synthetic_model(7)
    arrays = _inputs(False, 45)
    rs = np.random.RandomState(11)
    gv, gj = rs.randn(B, 778, 3), rs.randn(B, 16, 3)
    layer = _layer(m, False, 45, False)
    g1 = _kernel_grads(layer, _cuda(arrays), gv, gj)
    g2 = _kernel_grads(layer, _cuda(arrays), gv, gj)
    for x, y in zip(g1, g2):
        assert torch.equal(x, y)
    one = _kernel_grads(layer, _cuda([a[5:6] for a in arrays]), gv[5:6], gj[5:6])
    for x, y in zip(one, g1):
        assert torch.equal(x[0], y[5])


@pytest.mark.gpu
def test_bf16_inputs_get_bf16_grads():
    m = mo.synthetic_model(7)
    arrays = _inputs(True, 45)
    rs = np.random.RandomState(12)
    gv, gj = rs.randn(B, 778, 3), rs.randn(B, 16, 3)
    layer = _layer(m)
    tb = _cuda(arrays, torch.bfloat16)
    gb = _kernel_grads(layer, tb, gv, gj)
    g32 = _kernel_grads(layer, [t.detach().float().requires_grad_(True) for t in tb], gv, gj)
    for x, y in zip(gb, g32):
        assert x.dtype == torch.bfloat16 and torch.equal(x, y.to(torch.bfloat16))


@pytest.mark.gpu
def test_empty_batch():
    layer = _layer(mo.synthetic_model(7))
    ts = [torch.zeros(0, n, device="cuda", requires_grad=True) for n in (10, 3, 45, 3)]
    out = layer(betas=ts[0], global_orient=ts[1], hand_pose=ts[2], transl=ts[3])
    assert tuple(out.vertices.shape) == (0, 778, 3) and tuple(out.joints.shape) == (0, 16, 3)
    gs = torch.autograd.grad((out.vertices, out.joints), ts, (torch.zeros(0, 778, 3, device="cuda"), torch.zeros(0, 16, 3, device="cuda")))
    assert [tuple(g.shape) for g in gs] == [(0, 10), (0, 3), (0, 45), (0, 3)]


@pytest.mark.gpu
def test_cuda_graph_replay_matches_eager():
    m = mo.synthetic_model(7)
    layer = _layer(m)
    static = _cuda(_inputs(True, 45, seed=13))
    rs = np.random.RandomState(14)
    gv = torch.from_numpy(rs.randn(B, 778, 3).astype(np.float32)).cuda()
    gj = torch.from_numpy(rs.randn(B, 16, 3).astype(np.float32)).cuda()

    def step(ts):
        out = layer(betas=ts[0], global_orient=ts[1], hand_pose=ts[2], transl=ts[3])
        return (out.vertices, out.joints) + torch.autograd.grad((out.vertices, out.joints), ts, (gv, gj))

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step(static)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step(static)
    fresh = _cuda(_inputs(True, 45, seed=15))
    with torch.no_grad():
        for d, src in zip(static, fresh):
            d.copy_(src)
    graph.replay()
    torch.cuda.synchronize()
    eager = step(fresh)
    for x, y in zip(captured, eager):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_adam_fit_recovers_the_hand():
    """Test-time refinement: 50 Adam steps on (betas, global_orient, hand_pose, transl) from perturbed copies of the parameters
    that generated the target vertices."""
    m = mo.synthetic_model(11)
    rs = np.random.RandomState(12)
    n = 8
    truth = [torch.from_numpy(a.astype(np.float32)).cuda() for a in (rs.randn(n, 10), 0.5 * rs.randn(n, 3), 0.5 * rs.randn(n, 45), 0.1 * rs.randn(n, 3))]
    layer = _layer(m)
    with torch.no_grad():
        target = layer(betas=truth[0], global_orient=truth[1], hand_pose=truth[2], transl=truth[3]).vertices
    params = [(x + 0.1 * torch.from_numpy(rs.randn(*x.shape).astype(np.float32)).cuda()).requires_grad_(True) for x in truth]
    opt = torch.optim.Adam(params, lr=3e-2)

    def loss_fn():
        v = layer(betas=params[0], global_orient=params[1], hand_pose=params[2], transl=params[3]).vertices
        return ((v - target) ** 2).sum(-1).mean()

    with torch.no_grad():
        first = float(loss_fn())
    for _ in range(50):
        opt.zero_grad()
        loss = loss_fn()
        loss.backward()
        opt.step()
    with torch.no_grad():
        last = float(loss_fn())
    print("fit loss %.3e -> %.3e" % (first, last))
    assert all(p.grad is not None for p in params)
    assert last < 1e-2 * first

"""Hand-object nearest-point search: ``dvq.nearest_points``, ``dvq.HandObjectContact`` and the C entries behind them
(``dvq_nn_forward``, ``dvq_nn_backward``, ``dvq_vertex_normals``).

The contract is csrc/contact_exact.cuh's; oracle/contact_oracle.py restates it in float32 numpy, and the GPU tests compare
bits with it.  pytorch3d is not available here, so parity with pytorch3d's own bits is not pinned (DESIGN.md §2).
CPU: the oracle's FMA emulation against exact rational arithmetic, the oracle against a float64 brute force, the vertex ->
face lists, face validation, the C ABI's argument errors and the missing CPU path.
GPU: forward, backward and normals bit for bit; the interior test on a closed sphere; gradients through ``dvq.ManoLayer``
against float64 autograd; an Adam fit; CUDA-graph replay.
"""
import ctypes
from fractions import Fraction

import numpy as np
import pytest
import torch

from _mano_torch import mano_forward_torch
from oracle import contact_oracle as co
from oracle import mano_oracle as mo

TIE = 1e-6          # relative near-tie band of the float64 comparisons
FLOOR = 1e-12       # absolute floor of that band (coincident points)


def _cloud(rs, B, n, scale=1.0):
    return (scale * rs.randn(B, n, 3)).astype(np.float32)


def _bits(a):
    a = np.ascontiguousarray(np.asarray(a, np.float32))
    return a.view(np.uint32)


def _same_bits(got, ref):
    """bit equality, with every NaN equal to every NaN (the GPU's canonical NaN differs from numpy's)"""
    got, ref = np.asarray(got, np.float32), np.asarray(ref, np.float32)
    nan = np.isnan(ref)
    return np.array_equal(np.isnan(got), nan) and np.array_equal(_bits(got)[~nan], _bits(ref)[~nan])


def icosphere(r, levels=2, flip=False):
    """A closed, outward-oriented subdivided icosahedron of radius r: (verts [V,3] float64, faces [F,3] int64)."""
    p = (1 + 5 ** 0.5) / 2
    v = [(-1, p, 0), (1, p, 0), (-1, -p, 0), (1, -p, 0), (0, -1, p), (0, 1, p), (0, -1, -p), (0, 1, -p),
         (p, 0, -1), (p, 0, 1), (-p, 0, -1), (-p, 0, 1)]
    f = [(0, 11, 5), (0, 5, 1), (0, 1, 7), (0, 7, 10), (0, 10, 11), (1, 5, 9), (5, 11, 4), (11, 10, 2), (10, 7, 6), (7, 1, 8),
         (3, 9, 4), (3, 4, 2), (3, 2, 6), (3, 6, 8), (3, 8, 9), (4, 9, 5), (2, 4, 11), (6, 2, 10), (8, 6, 7), (9, 8, 1)]
    verts = [np.array(x, float) / np.linalg.norm(x) for x in v]
    for _ in range(levels):
        mid, nf = {}, []

        def m(a, b):
            k = (min(a, b), max(a, b))
            if k not in mid:
                c = verts[a] + verts[b]
                verts.append(c / np.linalg.norm(c))
                mid[k] = len(verts) - 1
            return mid[k]

        for a, b, c in f:
            ab, bc, ca = m(a, b), m(b, c), m(c, a)
            nf += [(a, ab, ca), (b, bc, ab), (c, ca, bc), (ab, bc, ca)]
        f = nf
    V, F = r * np.array(verts), np.array(f, np.int64)
    x0, x1, x2 = V[F[:, 0]], V[F[:, 1]], V[F[:, 2]]
    inward = (np.cross(x1 - x0, x2 - x0) * (x0 + x1 + x2)).sum(1) < 0
    F[inward] = F[inward][:, ::-1]
    return V, (F[:, ::-1].copy() if flip else F)


def _fibonacci(n, radius):
    k = np.arange(n) + 0.5
    phi, th = np.arccos(1 - 2 * k / n), np.pi * (1 + 5 ** 0.5) * k
    return radius * np.stack([np.cos(th) * np.sin(phi), np.sin(th) * np.sin(phi), np.cos(phi)], 1)


# ---------------------------------------------------------------- CPU

def test_fma_emulation_is_exact():
    rs = np.random.RandomState(0)
    n = 3000
    a = (rs.randn(n) * np.exp2(rs.randint(-20, 20, n))).astype(np.float32)
    b = (rs.randn(n) * np.exp2(rs.randint(-20, 20, n))).astype(np.float32)
    c = (rs.randn(n) * np.exp2(rs.randint(-40, 40, n))).astype(np.float32)
    half = n // 2                                                 # near-cancelling: c ~ -a*b
    c[:half] = (-(a[:half].astype(np.float64) * b[:half]) * (1 + rs.randn(half) * 2.0 ** -rs.randint(10, 30, half))).astype(np.float32)
    got = co.fma_f32(a, b, c)
    for x, y, z, g in zip(a, b, c, got):
        exact = Fraction(float(x)) * Fraction(float(y)) + Fraction(float(z))
        lo = np.float32(float(exact))               # float64 rounding, then float32: a neighbour of the exact result
        cands = {lo, np.nextafter(lo, np.float32(np.inf)), np.nextafter(lo, np.float32(-np.inf))}
        best = min(cands, key=lambda q: (abs(Fraction(float(q)) - exact), int(np.array(q).view(np.uint32)) & 1))
        assert g == best or (g == 0 and best == 0), (x, y, z, g, best)


def test_oracle_matches_float64_brute_force():
    rs = np.random.RandomState(1)
    src, trg = _cloud(rs, 3, 200), _cloud(rs, 3, 150)
    trg[1, 7] = trg[1, 3]                                         # a duplicated target point: lowest index wins
    src[2, :5] = trg[2, 10:15]                                    # coincident points: distance 0
    dist, idx, _ = co.nn_forward(src, trg)
    d64, i64 = co.brute_force64(src, trg)
    best64 = d64.min(-1)
    assert np.all(idx[1] != 7)
    assert np.array_equal(idx[2, :5], np.arange(10, 15)) and np.all(dist[2, :5] == 0)
    mis = idx != i64
    picked = np.take_along_axis(d64, idx[..., None], -1)[..., 0]
    assert np.all(picked[mis] - best64[mis] <= TIE * best64[mis] + FLOOR)
    assert np.abs(dist - picked).max() <= 1e-5 * max(1.0, float(best64.max()))


def test_vertex_face_lists():
    from dvq.contact import vertex_face_csr
    faces = np.array([[0, 1, 2], [2, 1, 3], [3, 3, 0], [1, 4, 0]])
    off, vf = vertex_face_csr(faces, 6)
    assert off.dtype == np.int32 and vf.dtype == np.int32
    lists = [list(vf[off[v]:off[v + 1]]) for v in range(6)]
    assert lists == [[0, 2, 3], [0, 1, 3], [0, 1], [1, 2, 2], [3], []]


def test_contact_module_validates_faces():
    import dvq
    with pytest.raises(ValueError, match=r"\[F, 3\]"):
        dvq.HandObjectContact(np.zeros((4, 4), np.int64))
    with pytest.raises(ValueError, match="ids"):
        dvq.HandObjectContact(np.array([[0, 1, -1]]))
    with pytest.raises(TypeError, match="integer"):
        dvq.HandObjectContact(np.zeros((2, 3), np.float32))
    m = dvq.HandObjectContact(mo.synthetic_model(3)["faces"])
    assert m.faces.dtype == torch.int32 and m.vf_offsets.dtype == torch.int32 and m.vf_faces.numel() == 3 * m.faces.shape[0]
    assert "faces" not in m.state_dict()
    with pytest.raises(ValueError, match="no CPU path"):
        m(torch.zeros(1, 778, 3), torch.zeros(1, 5, 3))


def test_cabi_argument_errors():
    from dvq import _cabi
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    fwd = lambda B, N1, N2, **k: _cabi.lib.dvq_nn_forward(k.get("src", p), p, B, N1, N2, k.get("nrm"), p, p, k.get("inter"), None)
    assert fwd(-1, 1, 1) == -1 and "B >= 0" in _cabi.last_error()
    assert fwd(1, -1, 1) == -1
    assert fwd(1, 1, 0) == -1 and "N2 > 0" in _cabi.last_error()
    assert fwd(4096, 3000, 200000) == -1 and "2^31" in _cabi.last_error()
    assert fwd(1, 1, 1, src=None) == -7
    assert fwd(1, 1, 1, nrm=p) == -7 and "together" in _cabi.last_error()
    bwd = lambda B, N1, N2, g=p: _cabi.lib.dvq_nn_backward(p, p, p, g, B, N1, N2, p, p, None)
    assert bwd(1, 1, 0) == -1 and bwd(-2, 1, 1) == -1
    assert bwd(1, 1, 1, g=None) == -7
    nrm = lambda B, V, F, faces=p: _cabi.lib.dvq_vertex_normals(p, B, V, faces, F, p, p, p, None)
    assert nrm(1, 0, 1) == -1 and nrm(-1, 3, 1) == -1 and nrm(1, 3, -1) == -1
    assert nrm(1, 3, 1, faces=None) == -7


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_path():
    import dvq
    from dvq import _cabi
    with pytest.raises(ValueError, match="no CPU path"):
        dvq.nearest_points(torch.zeros(1, 4, 3), torch.zeros(1, 5, 3))
    with pytest.raises(TypeError):
        dvq.nearest_points(torch.zeros(1, 4, 3, dtype=torch.float64), torch.zeros(1, 5, 3, dtype=torch.float64))
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    assert _cabi.lib.dvq_nn_forward(p, p, 1, 1, 1, None, p, p, None, None) != 0
    assert _cabi.lib.dvq_vertex_normals(p, 1, 3, p, 1, p, p, p, None) != 0


# ---------------------------------------------------------------- GPU

def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _check_forward(src, trg, normals=None):
    import dvq
    if normals is None:
        dist, idx = dvq.nearest_points(_cuda(src), _cuda(trg))
        inter = None
    else:
        from dvq.contact import _search
        dist, idx, inter = _search(_cuda(src), _cuda(trg), _cuda(normals))
    rd, ri, rint = co.nn_forward(src, trg, normals)
    assert dist.dtype == torch.float32 and idx.dtype == torch.int64 and tuple(dist.shape) == src.shape[:2]
    assert np.array_equal(idx.cpu().numpy(), ri)
    assert _same_bits(dist.cpu().numpy(), rd)
    if normals is not None:
        assert inter.dtype == torch.bool and np.array_equal(inter.cpu().numpy(), rint)
    return dist, idx


@pytest.mark.gpu
@pytest.mark.parametrize("B,N1,N2", [(5, 3000, 778), (5, 778, 3000), (2, 1, 1), (2, 33, 5000), (1, 517, 70001)])
def test_forward_bits(B, N1, N2):
    rs = np.random.RandomState(N1 + N2)
    src, trg = _cloud(rs, B, N1), _cloud(rs, B, N2)
    nrm = rs.randn(B, N2, 3).astype(np.float32)
    _check_forward(src, trg)
    _check_forward(src, trg, nrm)


@pytest.mark.gpu
def test_forward_empty():
    import dvq
    for B, N1 in ((0, 10), (3, 0)):
        dist, idx = dvq.nearest_points(torch.zeros(B, N1, 3, device="cuda"), torch.zeros(B, 7, 3, device="cuda"))
        assert tuple(dist.shape) == (B, N1) and tuple(idx.shape) == (B, N1)


@pytest.mark.gpu
def test_forward_ties_and_non_finite():
    rs = np.random.RandomState(3)
    src, trg = _cloud(rs, 2, 300), _cloud(rs, 2, 2000)
    trg[0, 1500:] = trg[0, 100]                                   # many copies of one point, and copies across stages
    trg[0, 1024], trg[0, 5] = trg[0, 40], trg[0, 40]
    src[0, :50] = trg[0, 40] + np.float32(1e-3)
    src[0, 50:60] = trg[0, 100]
    trg[1, 3] = [np.nan, 0, 0]                                    # a NaN target point never wins
    trg[1, 9] = [np.inf, 0, 0]
    src[1, 0] = [np.nan, 0, 0]                                    # NaN row: index 0, dist NaN
    src[1, 1] = [np.inf, 0, 0]                                    # inf row: +inf or NaN everywhere -> index 0
    src[1, 2] = [0, -np.inf, 0]
    src[1, 3] = [1e30, 1e30, 1e30]                                # overflowing distances: +inf everywhere -> index 0
    dist, idx = _check_forward(src, trg)
    idx = idx.cpu().numpy()
    assert np.all(idx[0, :50] == 5) and np.all(idx[0, 50:60] == 100)
    assert np.all(idx[1, :4] == 0) and np.isnan(dist[1, 0].item())


def _grads(src, trg, g, want=(True, True)):
    import dvq
    s = _cuda(src).requires_grad_(want[0])
    t = _cuda(trg).requires_grad_(want[1])
    dist, idx = dvq.nearest_points(s, t)
    live = [x for x, w in zip((s, t), want) if w]
    got = iter(torch.autograd.grad(dist, live, _cuda(g)))
    return [next(got).cpu().numpy() if w else None for w in want], idx.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("B,N1,N2", [(3, 3000, 778), (3, 778, 3000), (2, 100, 1)])
def test_backward_bits(B, N1, N2):
    rs = np.random.RandomState(7 + N2)
    src, trg = _cloud(rs, B, N1), _cloud(rs, B, N2)
    g = rs.randn(B, N1).astype(np.float32)
    (gs, gt), idx = _grads(src, trg, g)
    rs_, rt_ = co.nn_backward(src, trg, idx, g)
    assert _same_bits(gs, rs_) and _same_bits(gt, rt_)
    (gs1, _), _ = _grads(src, trg, g, (True, False))
    (_, gt1), _ = _grads(src, trg, g, (False, True))
    assert _same_bits(gs1, rs_) and _same_bits(gt1, rt_)
    (gs2, gt2), _ = _grads(src, trg, g)
    assert np.array_equal(_bits(gs2), _bits(gs)) and np.array_equal(_bits(gt2), _bits(gt))
    # float64 autograd of the brute force, gathered with the kernel's idx (a near-tie flip cannot move the gradient)
    s64 = torch.from_numpy(src.astype(np.float64)).requires_grad_(True)
    t64 = torch.from_numpy(trg.astype(np.float64)).requires_grad_(True)
    near = torch.gather(t64, 1, torch.from_numpy(idx)[..., None].expand(-1, -1, 3))
    d64 = ((s64 - near) ** 2).sum(-1)
    r64 = torch.autograd.grad(d64, (s64, t64), torch.from_numpy(g.astype(np.float64)))
    for got, ref in zip((gs, gt), r64):
        ref = ref.numpy()
        assert np.abs(got - ref).max() <= 1e-5 * np.abs(ref).max()


@pytest.mark.gpu
def test_normals_bits():
    import dvq
    rs = np.random.RandomState(5)
    sv, sf = icosphere(0.05)
    for faces, V in ((mo.synthetic_model(7)["faces"], 778), (sf, len(sv))):
        verts = (rs.randn(3, V, 3) * 0.05).astype(np.float32)
        if V == len(sv):
            verts[0] = sv
        m = dvq.HandObjectContact(faces).cuda()
        got = m.vertex_normals(_cuda(verts)).cpu().numpy()
        assert _same_bits(got, co.vertex_normals(verts, faces))


@pytest.mark.gpu
@pytest.mark.parametrize("flip", [False, True])
def test_sphere_interior(flip):
    import dvq
    r = 0.08
    sv, sf = icosphere(r, levels=3, flip=flip)
    hand = _cuda(np.stack([sv, sv + 0.3]).astype(np.float32))
    pts = np.concatenate([_fibonacci(500, 0.5 * r), _fibonacci(500, 1.5 * r)]).astype(np.float32)
    obj = _cuda(np.stack([pts, pts + 0.3]).astype(np.float32))
    m = dvq.HandObjectContact(sf).cuda()
    dist, idx, inside = m(hand, obj)
    inside = inside.cpu().numpy()
    want = np.r_[np.ones(500, bool), np.zeros(500, bool)]
    assert np.array_equal(inside, np.stack([want, want]) ^ flip)
    normals = m.vertex_normals(hand)
    rd, ri, rint = co.nn_forward(obj.cpu().numpy(), hand.cpu().numpy(), normals.cpu().numpy())
    assert np.array_equal(idx.cpu().numpy(), ri) and _same_bits(dist.cpu().numpy(), rd) and np.array_equal(inside, rint)


def _hand_setup(seed=7, B=6, P=3000):
    import dvq
    m = mo.synthetic_model(seed)
    layer = dvq.ManoLayer(m, differentiable=True).cuda()
    contact = dvq.HandObjectContact(layer.faces).cuda()
    rs = np.random.RandomState(seed + 1)
    params = [rs.randn(B, 10), 0.3 * rs.randn(B, 3), 0.5 * rs.randn(B, 45), 0.01 * rs.randn(B, 3)]
    with torch.no_grad():
        v = layer(betas=_cuda(params[0].astype(np.float32)), hand_pose=_cuda(params[2].astype(np.float32))).vertices
    centre = v.mean(1, keepdim=True).cpu().numpy()
    obj = (centre + 0.05 * rs.randn(B, P, 3)).astype(np.float32)
    return m, layer, contact, params, obj


def _kernel_loss(layer, contact, ts, obj):
    import dvq
    verts = layer(betas=ts[0], global_orient=ts[1], hand_pose=ts[2], transl=ts[3]).vertices
    d1, i1, _ = contact(verts, obj)
    d2, i2 = dvq.nearest_points(verts, obj)
    return d1.mean() + d2.mean(), i1, i2


@pytest.mark.gpu
def test_grads_through_the_hand_layer():
    m, layer, contact, params, obj = _hand_setup()
    ts = [_cuda(p.astype(np.float32)).requires_grad_(True) for p in params]
    objc = _cuda(obj)
    loss, i1, i2 = _kernel_loss(layer, contact, ts, objc)
    got = torch.autograd.grad(loss, ts)
    t64 = [torch.from_numpy(p.astype(np.float32).astype(np.float64)).requires_grad_(True) for p in params]
    v64, _ = mano_forward_torch(m, *t64)
    o64 = torch.from_numpy(obj.astype(np.float64))
    i1, i2 = torch.from_numpy(i1.cpu().numpy()), torch.from_numpy(i2.cpu().numpy())
    d1 = ((o64 - torch.gather(v64, 1, i1[..., None].expand(-1, -1, 3))) ** 2).sum(-1)
    d2 = ((v64 - torch.gather(o64, 1, i2[..., None].expand(-1, -1, 3))) ** 2).sum(-1)
    ref = torch.autograd.grad(d1.mean() + d2.mean(), t64)
    for g, r in zip(got, ref):
        r = r.numpy()
        assert np.abs(g.double().cpu().numpy() - r).max() <= 1e-4 * np.abs(r).max()
    # the kernel's idx against the float64 argmin on the same (fp32) vertices: any disagreement lies inside the near-tie band
    with torch.no_grad():
        vv = layer(betas=ts[0], global_orient=ts[1], hand_pose=ts[2], transl=ts[3]).vertices.double().cpu().numpy()
    for a, b_, idx in ((obj, vv, i1.numpy()), (vv, obj, i2.numpy())):
        d, i64 = co.brute_force64(a, b_)
        best = d.min(-1)
        picked = np.take_along_axis(d, idx[..., None], -1)[..., 0]
        mis = idx != i64
        assert np.all(picked[mis] - best[mis] <= TIE * best[mis] + FLOOR)


@pytest.mark.gpu
def test_adam_refinement_lowers_the_loss():
    _, layer, contact, params, obj = _hand_setup(seed=9, B=4, P=1000)
    ts = [_cuda(p.astype(np.float32)).requires_grad_(True) for p in params]
    objc = _cuda(obj)
    opt = torch.optim.Adam(ts, lr=1e-2)
    with torch.no_grad():
        first = float(_kernel_loss(layer, contact, ts, objc)[0])
    for _ in range(50):
        opt.zero_grad()
        _kernel_loss(layer, contact, ts, objc)[0].backward()
        opt.step()
    with torch.no_grad():
        last = float(_kernel_loss(layer, contact, ts, objc)[0])
    print("refinement loss %.4e -> %.4e" % (first, last))
    assert last < first


@pytest.mark.gpu
def test_integration_example_runs():
    """INTEGRATION.md §2's refinement loop as written, with a synthetic model in place of MANO_RIGHT.pkl."""
    import dvq
    _, hand, _, p0, obj = _hand_setup(seed=3, B=4, P=3000)
    device = "cuda"
    betas, global_orient, hand_pose, transl = [_cuda(p.astype(np.float32)) for p in p0]
    obj_xyz = _cuda(obj)
    contact = dvq.HandObjectContact(hand.faces).to(device)
    params = [p.detach().clone().requires_grad_(True) for p in (betas, global_orient, hand_pose, transl)]
    opt = torch.optim.Adam(params, lr=3e-2)
    B = obj_xyz.shape[0]
    losses = []
    for _ in range(50):
        verts = hand(betas=params[0], global_orient=params[1], hand_pose=params[2], transl=params[3]).vertices
        d, _, inside = contact(verts, obj_xyz)
        penetration = (d * inside).sum() / B
        d_hand, _ = dvq.nearest_points(verts, obj_xyz)
        loss = penetration + d_hand.min(dim=1).values.mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
        losses.append(float(loss))
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]


@pytest.mark.gpu
def test_cuda_graph_replay_matches_eager():
    _, layer, contact, params, obj = _hand_setup(seed=4, B=3, P=2000)
    static = [_cuda(p.astype(np.float32)).requires_grad_(True) for p in params]
    objc = _cuda(obj).requires_grad_(True)

    def step(ts):
        loss, i1, i2 = _kernel_loss(layer, contact, ts, objc)
        return (loss, i1, i2) + torch.autograd.grad(loss, ts + [objc])

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step(static)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step(static)
    rs = np.random.RandomState(5)
    fresh = [_cuda((p + 0.1 * rs.randn(*p.shape)).astype(np.float32)).requires_grad_(True) for p in params]
    with torch.no_grad():
        for d, src in zip(static, fresh):
            d.copy_(src)
    graph.replay()
    torch.cuda.synchronize()
    eager = step(fresh)
    for x, y in zip(captured, eager):
        assert torch.equal(x, y)

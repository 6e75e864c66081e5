"""Differentiable penetration depth: ``dvq.penetration_depth``, ``dvq.point_mesh_distance(differentiable=True)`` and the C
entries behind them (``dvq_mesh_penetration``, ``dvq_mesh_distance_backward``).

The contract is csrc/mesh_exact.cuh's; tests/_mesh_grad_oracle.py restates the gradient in float64.
CPU: the oracle's gradient against float64 central differences, the C ABI's argument errors and the missing CPU path.
GPU: the fused query against the winding + distance composition, bit for bit (spheres both ways round, boxes, soups with
degenerate, skipped and non-finite faces, both broadcasts, ragged Q, empty batches) and against GraspQuality's depth; the
backward's offset against the forward's dist2, against the oracle, across runs, under broadcasting and in a CUDA graph;
and an Adam refinement of MANO hands out of an object.
"""
import ctypes

import numpy as np
import pytest
import torch

from _mesh_grad_oracle import closest_at_face, gradients
from oracle import contact_oracle as co
from oracle import mesh_oracle as mo
from test_contact import icosphere
from test_grasp_quality import _cuda, _diag, _ellipsoid_hands, _meshes, _queries, box_mesh, rotation

EPS = 2.0 ** -23
GRAD_ULPS = 8            # offset bar, in fp32 ulps of the scene's box diagonal (DESIGN.md §2; 0.73 measured on a B200)


def _bits(x):
    return x.detach().contiguous().view(torch.int32)


# ---------------------------------------------------------------- CPU

def test_oracle_gradient_matches_central_differences():
    rs = np.random.RandomState(0)
    tris = rs.randn(40, 3, 3).astype(np.float32)
    pts = (1.5 * rs.randn(40, 3)).astype(np.float32)
    verts, faces, face = tris.reshape(-1, 3), np.arange(120).reshape(40, 3), np.arange(40)
    r = closest_at_face(pts, verts, faces, face)
    f64 = lambda p, a, b, c: float(mo.triangle_dist2(p[None, None], a[None, None], b[None, None], c[None, None],
                                                     np.zeros((1, 1), bool))[0, 0])
    h = 1e-6
    checked = 0
    for i in range(40):
        x = [pts[i].astype(np.float64)] + [tris[i, k].astype(np.float64) for k in range(3)]
        assert abs(f64(*x) - r["dist2"][i]) <= 1e-12 * max(1.0, r["dist2"][i])
        # away from region boundaries: the closest point's weights are not at 0 / 1 transitions
        lam = r["lam"][i]
        if np.any((np.abs(lam) < 1e-3) & (lam != 0)) or np.any(np.abs(lam - 1) < 1e-3) & np.all(lam != 1):
            continue
        grads = [r["g_pts"][i]] + [r["g_corners"][i, k] for k in range(3)]
        for j in range(4):
            for d in range(3):
                xp = [y.copy() for y in x]
                xm = [y.copy() for y in x]
                xp[j][d] += h
                xm[j][d] -= h
                fd = (f64(*xp) - f64(*xm)) / (2 * h)
                assert abs(fd - grads[j][d]) <= 1e-6 * max(1.0, abs(fd)), (i, j, d, fd, grads[j][d])
        checked += 1
    assert checked >= 30
    # a degenerate (repeated-vertex) face is its edges: the closest point lies on one and its weights sum to 1
    v = np.array([[0, 0, 0], [1, 0, 0], [1, 0, 0]], np.float32)
    rd = closest_at_face(np.array([[0.5, 1, 0]], np.float32), v, [[0, 1, 2]], [0])
    assert np.allclose(rd["closest"], [[0.5, 0, 0]]) and abs(rd["lam"].sum() - 1) <= 1e-12


def test_cabi_argument_errors():
    from dvq import _cabi
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    pen = lambda Bm, V, F, Bp, Q, d=p: _cabi.lib.dvq_mesh_penetration(p, Bm, V, p, F, p, Bp, Q, d, p, None)
    assert pen(1, 3, 0, 1, 1) == -1 and "F > 0" in _cabi.last_error()
    assert pen(-1, 3, 1, 1, 1) == -1 and pen(1, 0, 1, 1, 1) == -1
    assert pen(3, 3, 1, 2, 1) == -1 and "1 or the batch" in _cabi.last_error()
    assert pen(4096, 3, 1, 1, 200000) == -1 and "2^31" in _cabi.last_error()
    assert pen(1, 3, 1, 1, 1, d=None) == -7
    bw = lambda Bm, V, F, Bp, Q, gp=p, gv=p, fc=p: _cabi.lib.dvq_mesh_distance_backward(p, Bm, V, p, F, p, Bp, Q, fc, p, gp, gv, None)
    assert bw(1, 3, 1, 1, 1, gp=None, gv=None) == -7 and "both" in _cabi.last_error()
    assert bw(1, 3, 1, 1, 1, fc=None) == -7
    assert bw(2, 3, 1, 3, 1) == -1 and bw(1, 0, 1, 1, 1) == -1
    assert bw(4096, 200000, 1, 4096, 1) == -1 and "2^31" in _cabi.last_error()


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_path():
    import dvq
    from dvq import _cabi
    v, f = box_mesh([0, 0, 0], [1, 1, 1])
    ov = torch.from_numpy(v.astype(np.float32))[None]
    with pytest.raises(ValueError, match="no CPU path"):
        dvq.penetration_depth(torch.zeros(1, 4, 3), ov, f)
    with pytest.raises(ValueError, match="no CPU path"):
        dvq.point_mesh_distance(torch.zeros(1, 4, 3, requires_grad=True), ov, f, differentiable=True)
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    assert _cabi.lib.dvq_mesh_penetration(p, 1, 3, p, 1, p, 1, 1, p, p, None) != 0
    assert _cabi.lib.dvq_mesh_distance_backward(p, 1, 3, p, 1, p, 1, 1, p, p, p, p, None) != 0


# ---------------------------------------------------------------- GPU: the forward

def _composition(q, v, f):
    import dvq
    w = dvq.winding_number(q, v, f)
    d, i = dvq.point_mesh_distance(q, v, f)
    inside = w >= 0.5
    return torch.where(inside, d, torch.zeros((), device=d.device)), torch.where(inside, i, torch.full((), -1, device=d.device))


def _scene(kind, rs, B=3, Q=1300):
    """(queries [B,Q,3], verts [B,V,3], faces) with some queries inside"""
    if kind == "box":
        meshes = []
        for _ in range(B):
            v, f = box_mesh(-rs.uniform(0.01, 0.05, 3), rs.uniform(0.01, 0.05, 3))
            meshes.append(((v @ rotation(rs).T) + 0.02 * rs.randn(3)).astype(np.float32))
    else:
        meshes = [_meshes(kind, rs) for _ in range(B)]
        f = meshes[0][1]
        meshes = [m[0] for m in meshes]
    V = np.stack(meshes)
    Q_ = np.stack([_queries(m, rs, Q) for m in meshes])
    return Q_, V, np.asarray(f, np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["closed", "flipped", "box", "open", "soup", "degenerate"])
def test_penetration_equals_composition(kind):
    import dvq
    rs = np.random.RandomState({"closed": 20, "flipped": 21, "box": 22, "open": 23, "soup": 24, "degenerate": 25}[kind])
    q, v, f = _scene("closed" if kind == "degenerate" else kind, rs)
    if kind == "degenerate":                                     # a closed sphere plus exactly degenerate faces
        f = np.concatenate([f, [[0, 1, 1], [2, 2, 2], [3, 4, 4]]])
    if kind == "soup":                                           # degenerate faces and non-finite corners / queries
        v[:, f[5, 2]] = v[:, f[5, 0]] + 2 * (v[:, f[5, 1]] - v[:, f[5, 0]])
        f[6, 2] = f[6, 1]
        f[7] = f[7, 0]
        v[:, f[8, 1]] = [np.nan, 0, 0]
        v[:, f[9, 2]] = [np.inf, 0, 0]
        q[:, :3] = [[np.nan, 0, 0], [np.inf, 0, 0], [0, -np.inf, 0]]
    Q, V = _cuda(q), _cuda(v)
    d2, face = dvq.penetration_depth(Q, V, f)
    wd, wf = _composition(Q, V, f)
    assert d2.dtype == torch.float32 and face.dtype == torch.int64 and d2.shape == face.shape == (3, 1300)
    assert torch.equal(_bits(d2), _bits(wd)) and torch.equal(face, wf)
    inside = (face >= 0).sum().item()
    print("%s: %d of %d queries inside" % (kind, inside, face.numel()))
    if kind == "flipped":                                        # w = -1 inside a flipped mesh: nothing is "inside"
        assert inside == 0 and torch.all(d2 == 0)
    elif kind != "soup":                                         # an open soup has no inside
        assert inside > 50
    for qb, vb in ((Q[:1], V), (Q, V[:1])):                      # both broadcasts
        d2b, fb = dvq.penetration_depth(qb, vb, f)
        wdb, wfb = _composition(qb, vb, f)
        assert torch.equal(_bits(d2b), _bits(wdb)) and torch.equal(fb, wfb)


@pytest.mark.gpu
def test_penetration_skipped_faces_ragged_and_empty():
    from dvq.grasp_quality import _distance, _penetration, _winding
    rs = np.random.RandomState(25)
    v, f = _meshes("closed", rs)
    bad = np.insert(f, [7, 100, 100], [[0, 1, len(v)], [-1, 2, 3], [5, 2 ** 30, 1]], axis=0)
    fc = torch.from_numpy(bad.astype(np.int32)).cuda()
    for Q in (1, 511, 513, 1537):                                # Q not a multiple of the 512-query tile
        q = _cuda(_queries(v, rs, Q)[None])
        d2, face = _penetration(q, _cuda(v[None]), fc, 1)
        w = torch.empty(1, Q, device="cuda")
        _winding(q, _cuda(v[None]), fc, w=w)
        d, i = _distance(q, _cuda(v[None]), fc, 1)
        ins = w >= 0.5
        assert torch.equal(_bits(d2), _bits(torch.where(ins, d, torch.zeros((), device="cuda"))))
        assert torch.equal(face, torch.where(ins, i, torch.full((), -1, device="cuda")))
    import dvq
    for qs, vs in (((0, 5, 3), (1, len(v), 3)), ((1, 0, 3), (1, len(v), 3)), ((1, 5, 3), (0, len(v), 3))):
        d2, face = dvq.penetration_depth(torch.zeros(qs, device="cuda"), torch.zeros(vs, device="cuda"), f)
        assert d2.numel() == 0 and face.numel() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("obj", ["box", "sphere"])
def test_depth_equals_grasp_quality(obj):
    import dvq
    from test_grasp_quality import _object
    rs = np.random.RandomState(26 + (obj == "box"))
    ov, of = _object(obj)
    hands, hf = _ellipsoid_hands(rs, 512, np.zeros(3))
    gq = dvq.GraspQuality(_cuda(ov), of, hf, 0.006, 0.005).cuda()
    H = _cuda(hands)
    _, depth, _ = gq(H)
    d2, _ = dvq.penetration_depth(H, gq.obj_verts, of)
    assert (depth > 0).sum() > 50
    assert torch.equal(_bits(d2.sqrt().amax(1)), _bits(depth))


# ---------------------------------------------------------------- GPU: the backward

def _grad(q, v, f, g, fused=True, want=(True, True)):
    import dvq
    q = q.detach().clone().requires_grad_(want[0])
    v = v.detach().clone().requires_grad_(want[1])
    d2, face = dvq.penetration_depth(q, v, f) if fused else dvq.point_mesh_distance(q, v, f, differentiable=True)
    (d2 * g).sum().backward()
    return d2, face, q.grad, v.grad


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["closed", "box", "soup"])
def test_backward_offset_is_the_forward_offset(kind):
    """g = 0.5: g_pts = fl(2 g) d = d exactly, and on triangle faces fma(dz, dz, fma(dy, dy, dx dx)) of it is dist2."""
    rs = np.random.RandomState(30 + len(kind))
    q, v, f = _scene(kind, rs, B=2, Q=2000)
    if kind == "soup":
        v[:, f[5, 2]] = v[:, f[5, 0]] + 2 * (v[:, f[5, 1]] - v[:, f[5, 0]])
        f[6, 2] = f[6, 1]
        for j, fi in enumerate((5, 6)):                            # queries next to the degenerate faces
            q[:, 20 * j:20 * j + 20] = v[:, f[fi]].mean(1)[:, None] + 1e-3 * rs.randn(2, 20, 3)
    d2, face, gq, _ = _grad(_cuda(q), _cuda(v), f, 0.5, fused=False)
    d2, face, gq = d2.detach().cpu().numpy(), face.cpu().numpy(), gq.cpu().numpy()
    for b in range(2):
        tri = f[face[b]]
        a, bb, c = (v[b][tri[:, j]] for j in range(3))
        degenerate = mo.area2_f32((bb - a).astype(np.float32), (c - a).astype(np.float32)) == 0
        dx, dy, dz = gq[b, :, 0], gq[b, :, 1], gq[b, :, 2]
        norm = co.fma_f32(dz, dz, co.fma_f32(dy, dy, (dx * dx).astype(np.float32)))
        assert np.array_equal(norm[~degenerate].view(np.uint32), d2[b][~degenerate].view(np.uint32))
        if kind == "soup":
            assert degenerate.any()
            assert np.abs(norm[degenerate] - d2[b][degenerate]).max() <= 4 * EPS * d2[b][degenerate].max()


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_backward_matches_oracle(fused):
    rs = np.random.RandomState(40 + fused)
    ov, of = icosphere(0.05, 2)
    hands, hf = _ellipsoid_hands(rs, 6, np.zeros(3))
    g = rs.uniform(-2, 2, (6, hands.shape[1])).astype(np.float32)
    # hand vertices against the object (verts broadcast) and object points against the hands (points broadcast)
    for q, v, f in ((hands, ov[None].astype(np.float32), of), (_queries(ov, rs, 3000)[None] * 0.8, hands, hf)):
        B = max(len(q), len(v))
        gg = g if q.shape[1] == g.shape[1] else rs.uniform(-2, 2, (B, q.shape[1])).astype(np.float32)
        qe, ve = np.broadcast_to(q, (B,) + q.shape[1:]), np.broadcast_to(v, (B,) + v.shape[1:])
        _, face, gq, gv = _grad(_cuda(qe), _cuda(ve), f, _cuda(gg), fused=fused)
        face, gq, gv = face.cpu().numpy(), gq.cpu().numpy(), gv.cpu().numpy()
        worst_p = worst_v = 0.0
        for b in range(B):
            L = _diag(np.concatenate([ve[b], qe[b]]))
            rp, rv = gradients(qe[b], ve[b], f, face[b], gg[b])
            ep = np.abs(gq[b] - rp).max(1)
            bar_p = GRAD_ULPS * EPS * L * 2 * np.abs(gg[b])
            assert np.all(ep <= bar_p + 1e-30), (b, (ep / np.maximum(bar_p, 1e-30)).max())
            worst_p = max(worst_p, float((ep / np.maximum(2 * np.abs(gg[b]) * EPS * L, 1e-30)).max()))
            # per vertex: the sum of its terms' bars plus the rounding of the ascending sum
            keep = face[b] >= 0
            tri = f[face[b][keep]]
            gsum, tsum, n = np.zeros(len(ve[b])), np.zeros(len(ve[b])), np.zeros(len(ve[b]))
            r = closest_at_face(qe[b][keep], ve[b], f, face[b][keep]) if keep.any() else None
            for k in range(3):
                np.add.at(gsum, tri[:, k], 2 * np.abs(gg[b][keep]))
                np.add.at(n, tri[:, k], 1)
                if r is not None:
                    np.add.at(tsum, tri[:, k], np.abs(gg[b][keep, None] * r["g_corners"][:, k]).max(1))
            ev = np.abs(gv[b] - rv).max(1)
            bar_v = GRAD_ULPS * EPS * L * gsum + n * EPS * tsum
            assert np.all(ev <= bar_v + 1e-30), (b, (ev / np.maximum(bar_v, 1e-30)).max())
            worst_v = max(worst_v, float((ev / np.maximum(EPS * L * gsum + n * EPS * tsum, 1e-30)).max()))
        print("fused=%s Bp=%d: g_pts max error %.2f ulps of 2|g| diag, g_verts %.2f" % (fused, len(q), worst_p, worst_v))


@pytest.mark.gpu
def test_backward_deterministic_and_broadcast():
    rs = np.random.RandomState(50)
    ov, of = icosphere(0.05, 3)
    hands, hf = _ellipsoid_hands(rs, 64, np.zeros(3))
    H, O = _cuda(hands), _cuda(ov[None])
    G = _cuda(rs.uniform(-1, 1, (64, hands.shape[1])))
    runs = [_grad(H, O, of, G) for _ in range(2)]
    assert all(torch.equal(_bits(x), _bits(y)) for x, y in zip(runs[0][2:], runs[1][2:]))
    assert runs[0][3].shape == (1, len(ov), 3) and (runs[0][1] >= 0).sum() > 100
    # broadcast = the sum of the explicitly expanded per-item gradients (autograd's expand backward)
    for q, v in ((H, O), (_cuda(_queries(ov, rs, 2000)[None] * 0.8), H)):
        B = max(q.shape[0], v.shape[0])
        f = of if v.shape[1] == len(ov) else hf
        g = _cuda(rs.uniform(-1, 1, (B, q.shape[1])))
        _, _, gq, gv = _grad(q, v, f, g)
        qe = q.detach().clone().requires_grad_(True)
        ve = v.detach().clone().requires_grad_(True)
        import dvq
        d2, _ = dvq.penetration_depth(qe.expand(B, -1, -1), ve.expand(B, -1, -1), f)
        (d2 * g).sum().backward()
        assert torch.equal(_bits(gq), _bits(qe.grad)) and torch.equal(_bits(gv), _bits(ve.grad))


@pytest.mark.gpu
def test_cuda_graph_replay_forward_backward():
    """The launches are capturable; the faces are validated (on the host) before capture, as GraspQuality keeps them."""
    import dvq
    from dvq.grasp_quality import _MeshDistance
    rs = np.random.RandomState(51)
    ov, of = icosphere(0.05, 3)
    hands, hf = _ellipsoid_hands(rs, 32, np.zeros(3))
    O = _cuda(ov[None])
    F = torch.from_numpy(of.astype(np.int32)).cuda()
    static = _cuda(hands).requires_grad_(True)

    def step():
        static.grad = None
        d2, _ = _MeshDistance.apply(static, O, F, 32, True)
        d2.sum().backward()
        return d2.detach(), static.grad

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = step()
    fresh, _ = _ellipsoid_hands(rs, 32, np.zeros(3))
    with torch.no_grad():
        static.copy_(_cuda(fresh))
    graph.replay()
    torch.cuda.synchronize()
    x = _cuda(fresh).requires_grad_(True)
    e, _ = dvq.penetration_depth(x, O, of)
    e.sum().backward()
    assert (captured[0] > 0).any()
    assert torch.equal(_bits(captured[0]), _bits(e)) and torch.equal(_bits(captured[1]), _bits(x.grad))


@pytest.mark.gpu
def test_adam_refinement_lowers_depth_and_volume():
    """Both penetration directions through ManoLayer(differentiable=True) (synthetic tables, scaled to hand size)."""
    import dvq
    from oracle import mano_oracle as mano
    dev = "cuda"
    model = mano.synthetic_model(3)
    model["v_template"] = 0.3 * model["v_template"]
    layer = dvq.ManoLayer(model, differentiable=True).to(dev)
    ov, of = icosphere(0.05, 3)
    obj = _cuda(ov)
    quality = dvq.GraspQuality(obj, of, layer.faces, pitch=0.005, contact_tol=0.005).to(dev)
    rs = np.random.RandomState(52)
    B = 64
    t = lambda a: torch.from_numpy(np.asarray(a, np.float32)).to(dev)
    params = [t(0.3 * rs.randn(B, 10)), t(0.3 * rs.randn(B, 3)), t(0.3 * rs.randn(B, 45)), t(0.03 * rs.randn(B, 3))]
    params = [p.requires_grad_(True) for p in params]
    hand = lambda: layer(betas=params[0], global_orient=params[1], hand_pose=params[2], transl=params[3]).vertices
    with torch.no_grad():
        vol0, dep0, _ = quality(hand())
    pen = dep0 > 0
    assert pen.sum() > 20
    opt = torch.optim.Adam(params, lr=3e-3)
    for _ in range(40):
        verts = hand()
        d_hand, _ = dvq.penetration_depth(verts, obj[None], of)                 # hand vertices inside the object
        d_obj, _ = dvq.penetration_depth(quality.centres, verts, layer.faces)    # object voxels inside each hand
        loss = (d_hand.sum() + d_obj.sum()) / B
        opt.zero_grad()
        loss.backward()
        opt.step()
    with torch.no_grad():
        vol1, dep1, _ = quality(hand())
    print("mean depth %.4f -> %.4f, mean volume %.3g -> %.3g (penetrating hands: %d)"
          % (dep0[pen].mean(), dep1[pen].mean(), vol0[pen].mean(), vol1[pen].mean(), pen.sum()))
    assert dep1[pen].mean() < 0.5 * dep0[pen].mean()
    assert vol1[pen].mean() < vol0[pen].mean()

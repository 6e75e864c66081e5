"""Grasp scoring: ``dvq.winding_number``, ``dvq.point_mesh_distance``, ``dvq.GraspQuality`` and the C entries behind them
(``dvq_mesh_winding``, ``dvq_mesh_distance``).

The contract is csrc/mesh_exact.cuh's; oracle/mesh_oracle.py restates it in float64.  trimesh / igl are not available
here, so parity with their bits is not pinned (DESIGN.md §2).
CPU: the oracle on closed / flipped spheres and on analytic and densely sampled distances, the grid rule and its cap,
face validation, the C ABI's argument errors and the missing CPU path.
GPU: winding numbers and distances against the oracle, skipped faces, broadcasting, determinism, an exact volume, the
metrics against the oracle (B = 256 and a subset of B = 4096), CUDA-graph replay and the INTEGRATION.md example.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import mesh_oracle as mo
from test_contact import icosphere

EPS = 2.0 ** -23
DIST_ULPS = 4           # squared-distance bar, in fp32 ulps of the finite vertices' box diagonal^2 (0.09 measured on a B200)
TIE = 1e-6


def box_mesh(lo, hi):
    """closed, outward-oriented axis-aligned box: (verts [8,3], faces [12,3])"""
    lo, hi = np.asarray(lo, np.float64), np.asarray(hi, np.float64)
    v = np.array([[(hi if (i >> k) & 1 else lo)[k] for k in range(3)] for i in range(8)])
    quads = [(0, 2, 6, 4), (1, 5, 7, 3), (0, 4, 5, 1), (2, 3, 7, 6), (0, 1, 3, 2), (4, 6, 7, 5)]   # -x +x -y +y -z +z
    f = np.array([t for a, b, c, d in quads for t in ((a, c, b), (a, d, c))], np.int64)
    return v, f


def rotation(rs):
    q, r = np.linalg.qr(rs.randn(3, 3))
    q = q * np.sign(np.diag(r))
    return q * np.linalg.det(q)


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).cuda()


def _diag(v):
    v = np.asarray(v, np.float64)
    v = v[np.isfinite(v).all(1)]
    return float(np.linalg.norm(v.max(0) - v.min(0)))


# ---------------------------------------------------------------- CPU

@pytest.mark.parametrize("flip", [False, True])
def test_oracle_winding_on_spheres(flip):
    v, f = icosphere(0.05, 2, flip=flip)
    v = v.astype(np.float32)
    rs = np.random.RandomState(0)
    d = rs.randn(200, 3)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    inner, outer = (0.04 * d).astype(np.float32), (0.065 * d).astype(np.float32)
    w_in, w_out = mo.winding(inner, v, f), mo.winding(outer, v, f)
    assert np.abs(w_in - (-1 if flip else 1)).max() <= 1e-12
    assert np.abs(w_out).max() <= 1e-12
    far = np.array([[0.2, 0, 0], [np.nan, 0, 0]], np.float32)
    assert np.array_equal(mo.winding(far, v, f), [0.0, 0.0])          # the box rule; NaN is outside


def test_oracle_distance_analytic_and_sampled():
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [2, 0, 0], [1, 1, 0]], np.float32)
    tri = [[0, 1, 2]]
    cases = [((0.2, 0.2, 0.5), 0.25), ((-1, -1, 0.5), 2.25), ((0.5, -1, 0.5), 1.25), ((1, 1, 0), 0.5), ((2, 0, 0), 1.0),
             ((0, 2, -1), 2.0), ((0.25, 0.25, 0), 0.0)]
    for p, want in cases:
        d, face, _ = mo.distance(np.array([p], np.float32), v, tri)
        assert abs(d[0] - want) <= 1e-12 and face[0] == 0, (p, d, want)
    # degenerate: collinear (0, 1, 3), repeated vertex (1, 1, 4), one point (4, 4, 4) -> their edges / point
    degen = [[0, 1, 3], [1, 1, 4], [4, 4, 4]]
    for p, want in [((3, 1, 0), [2.0, 4.0, 4.0]), ((1, 0.5, 0), [0.25, 0.0, 0.25])]:
        _, _, d = mo.distance(np.array([p], np.float32), v, degen)
        assert np.allclose(d[0], want, atol=1e-12), (p, d)
    # dense barycentric sampling bounds the oracle from above, within the sampling resolution
    rs = np.random.RandomState(1)
    tris = rs.randn(20, 3, 3).astype(np.float32)
    tris[3, 2] = tris[3, 0] + 2 * (tris[3, 1] - tris[3, 0])                  # collinear (not exactly: fp32)
    tris[4, 2] = tris[4, 1]                                                   # repeated vertex: exactly degenerate
    verts, faces = tris.reshape(-1, 3), np.arange(60).reshape(20, 3)
    pts = (2 * rs.randn(50, 3)).astype(np.float32)
    d, face, dall = mo.distance(pts, verts, faces)
    n = 200
    s, t = np.meshgrid(np.linspace(0, 1, n), np.linspace(0, 1, n))
    keep = s + t <= 1
    s, t = s[keep], t[keep]
    for fi in range(20):
        a, b, c = tris[fi].astype(np.float64)
        samples = a + s[:, None] * (b - a) + t[:, None] * (c - a)
        ds = ((pts[:, None, :].astype(np.float64) - samples[None]) ** 2).sum(-1).min(1)
        h = np.linalg.norm(np.r_[[b - a], [c - a]], axis=1).max() / n
        assert np.all(dall[:, fi] <= ds + 1e-12)
        assert np.all(np.sqrt(ds) - np.sqrt(dall[:, fi]) <= 2 * h)
    assert np.array_equal(face, dall.argmin(1)) and np.array_equal(d, dall.min(1))


def test_grid_rule_and_cap():
    from dvq.grasp_quality import MAX_CELLS, voxel_grid
    assert voxel_grid([0, 0, 0], [1, 1, 1], 0.25) == [4, 4, 4]
    assert voxel_grid([0, 0, 0], [1, 0.3, 0], 0.25) == [4, 2, 1]            # a flat axis still has one cell
    assert voxel_grid([0, 0, 0], [1, 1, 1], 0.3) == [4, 4, 4]                # ceil
    assert voxel_grid([0, 0, 0], [1, 1, 1], 1 / 256) == [256] * 3            # 2^24 cells: at the cap
    with pytest.raises(ValueError, match="cap"):
        voxel_grid([0, 0, 0], [1, 1, 1.01], 1 / 256)
    with pytest.raises(ValueError, match="pitch"):
        voxel_grid([0, 0, 0], [1, 1, 1], 0.0)
    assert MAX_CELLS == mo.MAX_CELLS
    v, bf = box_mesh([0.1, 0.2, 0.3], [0.5, 0.25, 0.9])
    assert abs(mo.winding(np.array([[0.3, 0.22, 0.6]], np.float32), v.astype(np.float32), bf)[0] - 1) <= 1e-12   # outward
    lo, n = mo.grid(v.astype(np.float32), 0.05)
    assert n == voxel_grid(v.min(0), v.max(0), 0.05) == [8, 1, 12]
    c = mo.voxel_centres(lo, n, 0.05)
    assert c.shape == (96, 3) and np.array_equal(c[1, :2], c[0, :2]) and c[1, 2] > c[0, 2] and c[12, 1] == c[0, 1]


def test_module_validates_inputs():
    import dvq
    v, f = box_mesh([0, 0, 0], [1, 1, 1])
    ov = torch.from_numpy(v.astype(np.float32))
    with pytest.raises(ValueError, match=r"\[F, 3\]"):
        dvq.GraspQuality(ov, np.zeros((4, 4), np.int64), f, 0.1, 0.01)
    with pytest.raises(ValueError, match="ids"):
        dvq.GraspQuality(ov, np.array([[0, 1, 8]]), f, 0.1, 0.01)
    with pytest.raises(TypeError, match="integer"):
        dvq.GraspQuality(ov, f.astype(np.float32), f, 0.1, 0.01)
    with pytest.raises(ValueError, match="ids"):
        dvq.GraspQuality(ov, f, np.array([[0, -1, 2]]), 0.1, 0.01)
    with pytest.raises(TypeError, match="fp32"):
        dvq.GraspQuality(ov.double(), f, f, 0.1, 0.01)
    with pytest.raises(ValueError, match="cap"):
        dvq.GraspQuality(ov, f, f, 1e-3, 0.01)
    with pytest.raises(ValueError, match="contact_tol"):
        dvq.GraspQuality(ov, f, f, 0.1, -1.0)


def test_cabi_argument_errors():
    from dvq import _cabi
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    wn = lambda Bm, V, F, Bp, Q, w=p, cnt=p, pts=p: _cabi.lib.dvq_mesh_winding(p, Bm, V, p, F, pts, Bp, Q, w, cnt, None)
    assert wn(-1, 3, 1, 1, 1) == -1 and "Bm >= 0" in _cabi.last_error()
    assert wn(1, 0, 1, 1, 1) == -1 and "V > 0" in _cabi.last_error()
    assert wn(1, 3, -1, 1, 1) == -1 and wn(1, 3, 1, 1, -1) == -1
    assert wn(2, 3, 1, 3, 1) == -1 and "1 or the batch" in _cabi.last_error()
    assert wn(4096, 3, 1, 1, 200000) == -1 and "2^31" in _cabi.last_error()
    assert wn(1, 3, 1, 1, 1, w=None, cnt=None) == -7 and "both" in _cabi.last_error()
    assert wn(1, 3, 1, 1, 1, pts=None) == -7
    dist = lambda Bm, V, F, Bp, Q, d=p: _cabi.lib.dvq_mesh_distance(p, Bm, V, p, F, p, Bp, Q, d, p, None)
    assert dist(1, 3, 0, 1, 1) == -1 and "F > 0" in _cabi.last_error()
    assert dist(3, 3, 1, 2, 1) == -1 and dist(1, 3, 1, 1, 1, d=None) == -7


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU failure mode")
def test_no_cpu_path():
    import dvq
    from dvq import _cabi
    v, f = box_mesh([0, 0, 0], [1, 1, 1])
    ov = torch.from_numpy(v.astype(np.float32))
    with pytest.raises(ValueError, match="no CPU path"):
        dvq.winding_number(torch.zeros(1, 4, 3), ov[None], f)
    with pytest.raises(ValueError, match="no CPU path"):
        dvq.point_mesh_distance(torch.zeros(1, 4, 3), ov[None], f)
    with pytest.raises(ValueError, match="no CPU path"):
        dvq.GraspQuality(ov, f, f, 0.1, 0.01)
    with pytest.raises(TypeError):
        dvq.winding_number(torch.zeros(1, 4, 3, dtype=torch.float64), ov[None].double(), f)
    buf = (ctypes.c_float * 64)()
    p = ctypes.addressof(buf)
    assert _cabi.lib.dvq_mesh_winding(p, 1, 3, p, 1, p, 1, 1, p, None, None) != 0
    assert _cabi.lib.dvq_mesh_distance(p, 1, 3, p, 1, p, 1, 1, p, p, None) != 0


# ---------------------------------------------------------------- GPU

def _meshes(kind, rs):
    """(verts [V,3] float32, faces) of a test mesh, under a random rigid transform"""
    if kind == "soup":
        c = rs.randn(200, 1, 3) * 0.03
        v = (c + 0.01 * rs.randn(200, 3, 3)).reshape(-1, 3)
        f = np.arange(600).reshape(200, 3)
    else:
        v, f = icosphere(0.05, 2, flip=kind == "flipped")
        if kind == "open":
            f = f[v[f].mean(1)[:, 2] < 0.03]                   # a cap cut off: open
    v = v @ rotation(rs).T + 0.1 * rs.randn(3)
    return v.astype(np.float32), np.asarray(f, np.int64)


def _queries(v, rs, n):
    lo, hi = v.min(0), v.max(0)
    mid, half = (lo + hi) / 2, (hi - lo) / 2
    return (mid + 1.3 * half * rs.uniform(-1, 1, (n, 3))).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["closed", "flipped", "open", "soup"])
def test_winding_matches_oracle(kind):
    import dvq
    from dvq.grasp_quality import _winding
    rs = np.random.RandomState({"closed": 0, "flipped": 1, "open": 2, "soup": 3}[kind])
    meshes = [_meshes(kind, rs) for _ in range(3)]
    f = meshes[0][1]
    V = np.stack([m[0] for m in meshes])
    Q = np.stack([_queries(m[0], rs, 3000) for m in meshes])
    w = dvq.winding_number(_cuda(Q), _cuda(V), f).cpu().numpy()
    count = torch.zeros(3, dtype=torch.int32, device="cuda")
    w2 = torch.empty(3, Q.shape[1], device="cuda")
    _winding(_cuda(Q), _cuda(V), torch.from_numpy(f.astype(np.int32)).cuda(), w=w2, count=count)
    assert np.array_equal(w2.cpu().numpy(), w) and np.array_equal(count.cpu().numpy(), (w >= 0.5).sum(1))
    for b in range(3):
        w64 = mo.winding(Q[b], V[b], f)
        lo, hi = mo.box(V[b])
        out = ~mo.in_box(Q[b], lo, hi)
        assert out.any() and np.all(w[b][out] == 0)
        d64, _, _ = mo.distance(Q[b], V[b], f)
        far = np.sqrt(d64) >= 1e-3 * _diag(V[b])
        err = np.abs(w[b] - w64)[far]
        print("%s item %d: max |dw| %.3g over %d queries" % (kind, b, err.max(), far.sum()))
        assert err.max() <= 1e-4
        clear = np.abs(w64 - 0.5) >= 1e-3
        assert np.array_equal((w[b] >= 0.5)[clear], (w64 >= 0.5)[clear])
        if kind != "soup":
            sign = -1 if kind == "flipped" else 1                 # both sides of the surface are well represented
            assert (sign * w64 >= 0.5).sum() > 100 and (np.abs(w64) < 1e-3).sum() > 100


def _check_distance(Q, V, f, dist2, face):
    bar = DIST_ULPS * EPS * _diag(V) ** 2
    d64, f64, dall = mo.distance(Q, V, f)
    fin = np.isfinite(d64)
    assert np.array_equal(np.isfinite(dist2), fin) and np.all(face[~fin] == 0)
    err = np.abs(dist2[fin] - d64[fin])
    print("distance: max error %.2f ulps of diag^2" % (err.max() / (EPS * _diag(V) ** 2)))
    assert err.max() <= bar
    mis = (face != f64) & fin
    picked = dall[np.arange(len(Q)), face]
    assert np.all(picked[mis] - d64[mis] <= TIE * d64[mis] + bar)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["closed", "soup"])
def test_distance_matches_oracle(kind):
    import dvq
    rs = np.random.RandomState(10 + (kind == "soup"))
    v, f = _meshes(kind, rs)
    if kind == "soup":                                           # exactly degenerate faces: collinear, repeated vertex, a point
        v[f[5, 2]] = v[f[5, 0]] + 2 * (v[f[5, 1]] - v[f[5, 0]])
        f[6, 2] = f[6, 1]
        f[7] = f[7, 0]
        v[f[8, 1]] = [np.nan, 0, 0]                              # non-finite corners: the face never wins
        v[f[9, 2]] = [np.inf, 0, 0]
    q = _queries(v[np.isfinite(v).all(1)], rs, 4000)
    q[:3] = [[np.nan, 0, 0], [np.inf, 0, 0], [0, -np.inf, 0]]
    dist2, face = dvq.point_mesh_distance(_cuda(q[None]), _cuda(v[None]), f)
    assert dist2.dtype == torch.float32 and face.dtype == torch.int64
    dist2, face = dist2[0].cpu().numpy(), face[0].cpu().numpy()
    assert np.all(face[:3] == 0) and np.all(dist2[:3] == np.inf)
    _check_distance(q[3:], v, f, dist2[3:], face[3:])
    if kind == "soup":
        d64, _, dall = mo.distance(q[3:], v, f)
        assert np.all(np.isinf(dall[:, 8])) and np.all(np.isinf(dall[:, 9]))


@pytest.mark.gpu
def test_skipped_faces_contribute_nothing():
    """Through the C entries (the Python layer validates faces): a face with an id outside [0, V) changes no bit."""
    from dvq.grasp_quality import _distance, _winding
    rs = np.random.RandomState(4)
    v, f = _meshes("closed", rs)
    q = _cuda(_queries(v, rs, 1500)[None])
    bad = np.insert(f, [7, 100, 100], [[0, 1, len(v)], [-1, 2, 3], [5, 2 ** 30, 1]], axis=0)
    keep = np.r_[np.arange(7), np.arange(8, 101), np.arange(103, len(bad))]
    assert np.array_equal(bad[keep], f)
    fc = lambda x: torch.from_numpy(x.astype(np.int32)).cuda()
    w1, w2 = torch.empty(1, 1500, device="cuda"), torch.empty(1, 1500, device="cuda")
    _winding(q, _cuda(v[None]), fc(f), w=w1)
    _winding(q, _cuda(v[None]), fc(bad), w=w2)
    assert torch.equal(w1, w2)
    d1, i1 = _distance(q, _cuda(v[None]), fc(f), 1)
    d2, i2 = _distance(q, _cuda(v[None]), fc(bad), 1)
    assert torch.equal(d1, d2) and np.array_equal(keep[i1.cpu().numpy()], i2.cpu().numpy())


@pytest.mark.gpu
def test_broadcast_and_determinism():
    import dvq
    rs = np.random.RandomState(5)
    B = 4
    meshes = [_meshes("closed", rs) for _ in range(B)]
    f = meshes[0][1]
    V = _cuda(np.stack([m[0] for m in meshes]))
    Q = _cuda(np.stack([_queries(meshes[0][0], rs, 1000) for _ in range(B)]))
    for q, v in ((Q[:1], V), (Q, V[:1]), (Q[:1], V[:1])):
        qe, ve = q.expand(B, -1, -1).contiguous(), v.expand(B, -1, -1).contiguous()
        assert torch.equal(dvq.winding_number(q, v, f), dvq.winding_number(qe, ve, f)[: max(q.shape[0], v.shape[0])])
        d, i = dvq.point_mesh_distance(q, v, f)
        de, ie = dvq.point_mesh_distance(qe, ve, f)
        n = max(q.shape[0], v.shape[0])
        assert torch.equal(d, de[:n]) and torch.equal(i, ie[:n])
    runs = [(dvq.winding_number(Q, V, f), *dvq.point_mesh_distance(Q, V, f)) for _ in range(3)]
    for r in runs[1:]:
        assert all(torch.equal(x, y) for x, y in zip(r, runs[0]))


@pytest.mark.gpu
def test_exact_volume_of_boxes():
    """Box "hands" in a box object whose faces lie on cell boundaries: every centre is half a cell from every face, so
    the count is the analytic product of the overlaps.  The pitch is a power of two: the grid is exact in fp32."""
    import dvq
    p = 2.0 ** -7
    ov, of = box_mesh([0, 0, 0], [10 * p, 8 * p, 6 * p])
    gq = dvq.GraspQuality(_cuda(ov), of, of, p, 0.25 * p).cuda()
    assert gq.grid == [10, 8, 6] and gq.num_voxels == 480
    hands, want = [], []
    rs = np.random.RandomState(6)
    for _ in range(32):
        lo = rs.randint(-3, 9, 3)
        hi = lo + rs.randint(1, 6, 3)
        hv, _ = box_mesh(lo * p, hi * p)
        hands.append(hv)
        ov_ = [max(0, min(h, n) - max(l, 0)) for l, h, n in zip(lo, hi, (10, 8, 6))]
        want.append(ov_[0] * ov_[1] * ov_[2])
    volume, depth, contact = gq(_cuda(np.stack(hands)))
    assert np.array_equal(volume.cpu().numpy(), (np.array(want) * p ** 3).astype(np.float32))
    assert volume.dtype == torch.float32 and depth.dtype == torch.float32 and contact.dtype == torch.bool


def _ellipsoid_hands(rs, B, around):
    """B closed hand-sized ellipsoids (levels-2 icosphere, half-axes 4.5 x 2 x 1.2 cm) at random poses around `around`"""
    v, f = icosphere(1.0, 2)
    v = v * np.array([0.045, 0.02, 0.012])
    d = rs.randn(B, 3)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    r = rs.uniform(0.0, 0.11, (B, 1))
    hands = np.stack([v @ rotation(rs).T for _ in range(B)]) + (around + r * d)[:, None, :]
    return hands.astype(np.float32), f


def _object(kind):
    if kind == "box":
        v, f = box_mesh([-0.04, -0.03, -0.05], [0.04, 0.03, 0.05])
    else:
        v, f = icosphere(0.05, 2)
    return v.astype(np.float32), f


def _check_metrics(gq, ov, of, hands, hf, got, items, pitch, tol):
    volume, depth, contact = (x.cpu().numpy() for x in got)
    centres = gq.centres[0].cpu().numpy()
    ref = mo.grasp_metrics(centres, ov, of, hands[items], hf, pitch, tol)
    bar = DIST_ULPS * EPS * _diag(ov) ** 2
    tol2 = float(np.float32(np.float32(tol) * np.float32(tol)))
    for j, b in enumerate(items):
        amb_c = (np.abs(ref["w_centres"][j] - 0.5) < 1e-3).sum()
        count = round(float(volume[b]) / float(np.float32(pitch)) ** 3)
        assert volume[b] == np.float32(count * float(np.float32(pitch)) ** 3)
        assert abs(count - ref["count"][j]) <= amb_c, (b, count, ref["count"][j], amb_c)
        amb_v = np.abs(ref["w_verts"][j] - 0.5) < 1e-3
        slack = bar + (ref["dist2"][j][amb_v].max() if amb_v.any() else 0.0)
        assert abs(float(depth[b]) ** 2 - ref["depth"][j] ** 2) <= slack + 2 * bar, (b, depth[b], ref["depth"][j])
        near_tol = np.abs(ref["dist2"][j] - tol2) <= bar
        if not (amb_v.any() or near_tol.any()):
            assert contact[b] == ref["contact"][j], b
    return ref


@pytest.mark.gpu
@pytest.mark.parametrize("obj", ["box", "sphere"])
def test_metrics_match_oracle(obj):
    import dvq
    rs = np.random.RandomState(7 + (obj == "box"))
    ov, of = _object(obj)
    hands, hf = _ellipsoid_hands(rs, 256, np.zeros(3))
    pitch, tol = 0.006, 0.005
    gq = dvq.GraspQuality(_cuda(ov), of, hf, pitch, tol).cuda()
    # the kept centres against the oracle's float64 decisions
    lo, n = mo.grid(ov, pitch)
    assert gq.grid == n
    allc = mo.voxel_centres(lo, n, pitch)
    w64 = mo.winding(allc, ov, of)
    clear = np.abs(w64 - 0.5) >= 1e-3
    got = {tuple(c) for c in gq.centres[0].cpu().numpy().view(np.uint32)}
    want = {tuple(c) for c in allc[(w64 >= 0.5) & clear].view(np.uint32)}
    unsure = {tuple(c) for c in allc[~clear].view(np.uint32)}
    assert want <= got and got - want <= unsure
    res = gq(_cuda(hands))
    ref = _check_metrics(gq, ov, of, hands, hf, res, np.arange(256), pitch, tol)
    # the poses cover separated hands, hands touching within tol without penetrating, and deep penetration
    inside_any = np.array([(w >= 0.5).any() for w in ref["w_verts"]])
    touching = np.array(ref["contact"]) & ~inside_any & (ref["count"] == 0)
    print("%s: separated %d, touching %d, penetrating %d, max depth %.4f" % (obj, (~ref["contact"]).sum(), touching.sum(),
                                                                             inside_any.sum(), ref["depth"].max()))
    assert (~ref["contact"]).sum() > 10 and touching.sum() > 0 and (ref["depth"] > 0.01).sum() > 10


@pytest.mark.gpu
def test_large_batch():
    import dvq
    rs = np.random.RandomState(9)
    ov, of = _object("sphere")
    hands, hf = _ellipsoid_hands(rs, 4096, np.zeros(3))
    gq = dvq.GraspQuality(_cuda(ov), of, hf, 0.006, 0.005).cuda()
    res = gq(_cuda(hands))
    assert all(x.shape == (4096,) for x in res)
    _check_metrics(gq, ov, of, hands, hf, res, np.sort(rs.choice(4096, 24, replace=False)), 0.006, 0.005)


@pytest.mark.gpu
def test_cuda_graph_replay_matches_eager():
    import dvq
    rs = np.random.RandomState(11)
    ov, of = _object("sphere")
    hands, hf = _ellipsoid_hands(rs, 64, np.zeros(3))
    gq = dvq.GraspQuality(_cuda(ov), of, hf, 0.006, 0.005).cuda()
    static = _cuda(hands)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            gq(static)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        captured = gq(static)
    fresh, _ = _ellipsoid_hands(rs, 64, np.zeros(3))
    static.copy_(_cuda(fresh))
    graph.replay()
    torch.cuda.synchronize()
    eager = gq(_cuda(fresh))
    for x, y in zip(captured, eager):
        assert torch.equal(x, y)


@pytest.mark.gpu
def test_integration_example_runs():
    """INTEGRATION.md's scoring example as written, with a synthetic MANO model and a uniform prior."""
    import dvq
    from oracle import mano_oracle as mano
    device = "cuda"
    rh_mano = dvq.ManoLayer(mano.synthetic_model(3)).to(device)
    gen = dvq.GraspGenerator(hand_layer=rh_mano).to(device).eval()
    rs = np.random.RandomState(12)
    obj_pc = _cuda(0.05 * rs.randn(64, 4, 3000))
    sv, sf = icosphere(0.05, 3)
    obj_verts, obj_faces = _cuda(sv), sf
    v_max = 2e-6                                                  # 2 cm^3

    quality = dvq.GraspQuality(obj_verts, obj_faces, rh_mano.faces, pitch=0.005, contact_tol=0.005).to(device)
    recon, recon_pos = gen.gen(obj_pc)                            # obj_pc [B, 4, 3000]
    verts = rh_mano(betas=recon[:, :10], global_orient=recon_pos[:, :3], hand_pose=recon[:, 10:],
                    transl=recon_pos[:, 3:]).vertices
    volume, depth, contact = quality(verts)                       # [B] each; no host synchronisation
    keep = contact & (volume < v_max)
    good = verts[keep]

    assert volume.shape == depth.shape == contact.shape == keep.shape == (64,)
    assert good.shape[1:] == verts.shape[1:] and torch.isfinite(volume).all() and (depth >= 0).all()

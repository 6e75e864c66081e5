"""float64 restatement of the mesh contract (d-vqvae_b200/csrc/mesh_exact.cuh): winding numbers with the box rule, point-to-mesh
distances with the degenerate-face and tie rules, the voxel grid and the grasp metrics, for tests of dvq_mesh_winding /
dvq_mesh_distance / dvq.GraspQuality.

The fp32 steps the contract names are taken in fp32 here too: the corner offsets fl(v - q), the degenerate-face decision
(fp32 area^2 without FMA), the box, the voxel centres fl(lo + fl((i + 0.5) pitch)) and contact_tol^2.  Everything else is
float64, and the distance is computed independently of the kernel's region cascade: the minimum over the three edge
segments and, when the projection falls inside the triangle, the distance to its plane.
"""
import math

import numpy as np

f32, f64 = np.float32, np.float64
MAX_CELLS = 1 << 24


def valid_faces(faces, V):
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    return f[np.all((f >= 0) & (f < V), axis=1)], np.all((f >= 0) & (f < V), axis=1)


def box(verts):
    """per-axis (lo, hi) of verts [V,3] with NaN coordinates ignored (an all-NaN axis gives lo = +inf, hi = -inf)"""
    v = np.asarray(verts, f32)
    return np.where(np.isnan(v), np.inf, v).min(0), np.where(np.isnan(v), -np.inf, v).max(0)


def in_box(points, lo, hi):
    p = np.asarray(points, f32)
    with np.errstate(invalid="ignore"):
        return np.all((lo <= p) & (p <= hi), axis=-1)


def winding(points, verts, faces, chunk=64):
    """points [Q,3], verts [V,3] (float32) -> w [Q] float64; 0 outside the vertex box (the box rule)."""
    p, v = np.asarray(points, f32), np.asarray(verts, f32)
    f, _ = valid_faces(faces, len(v))
    lo, hi = box(v)
    w = np.zeros(len(p))
    todo = np.nonzero(in_box(p, lo, hi))[0]
    for i in range(0, len(todo), chunk):
        q = p[todo[i:i + chunk], None, :]
        with np.errstate(invalid="ignore", over="ignore"):
            a, b, c = ((v[f[:, j]][None] - q).astype(f32).astype(f64) for j in range(3))
            det = (a * np.cross(b, c)).sum(-1)
            la, lb, lc = (np.sqrt((x * x).sum(-1)) for x in (a, b, c))
            den = la * lb * lc + (a * b).sum(-1) * lc + (b * c).sum(-1) * la + (c * a).sum(-1) * lb
            w[todo[i:i + chunk]] = (2 * np.arctan2(det, den)).sum(1) / (4 * np.pi)
    return w


def area2_f32(e1, e2):
    """|e1 x e2|^2 in fp32, every operation rounded (the kernel's degenerate-face test)"""
    e1, e2 = np.asarray(e1, f32), np.asarray(e2, f32)
    with np.errstate(invalid="ignore", over="ignore"):
        nx = (e1[..., 1] * e2[..., 2]).astype(f32) - (e1[..., 2] * e2[..., 1]).astype(f32)
        ny = (e1[..., 2] * e2[..., 0]).astype(f32) - (e1[..., 0] * e2[..., 2]).astype(f32)
        nz = (e1[..., 0] * e2[..., 1]).astype(f32) - (e1[..., 1] * e2[..., 0]).astype(f32)
        nx, ny, nz = nx.astype(f32), ny.astype(f32), nz.astype(f32)
        return (((nx * nx).astype(f32) + (ny * ny).astype(f32)).astype(f32) + (nz * nz).astype(f32)).astype(f32)


def _segment(p, s, e):
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        d = e - s
        dd = (d * d).sum(-1)
        t = np.where(dd > 0, np.clip(((p - s) * d).sum(-1) / np.where(dd > 0, dd, 1), 0, 1), 0)
        r = p - s - t[..., None] * d
        return (r * r).sum(-1)


def triangle_dist2(p, a, b, c, degenerate):
    """float64 squared distances [Q,F] from p [Q,1,3] to the triangles (a, b, c) [1,F,3]; degenerate [F] -> edges only.
    A non-degenerate face with a non-finite corner gives NaN (the kernel's arithmetic does), which counts as +inf."""
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        d = np.fmin(np.fmin(_segment(p, a, b), _segment(p, a, c)), _segment(p, b, c))
        n = np.cross(b - a, c - a)
        nn = (n * n).sum(-1)
        h = ((p - a) * n).sum(-1)
        proj = p - (h / np.where(nn > 0, nn, 1))[..., None] * n
        inside = np.ones(d.shape, bool)
        for s, e in ((a, b), (b, c), (c, a)):
            inside &= (np.cross(e - s, proj - s) * n).sum(-1) >= 0
        plane = np.where(inside & (nn > 0) & ~degenerate, h * h / np.where(nn > 0, nn, 1), np.inf)
        finite = np.isfinite(a).all(-1) & np.isfinite(b).all(-1) & np.isfinite(c).all(-1)
        return np.where(degenerate, d, np.where(finite, np.fmin(d, plane), np.nan))


def distance(points, verts, faces, chunk=64):
    """points [Q,3], verts [V,3] (float32) -> (dist2 [Q] float64, face [Q] int64, d [Q,F] float64 of every face, +inf for
    skipped faces): the lowest f among the float64 minima (NaN as +inf); face 0 and +inf when nothing is finite."""
    p, v = np.asarray(points, f32), np.asarray(verts, f32)
    faces = np.asarray(faces, np.int64).reshape(-1, 3)
    _, ok = valid_faces(faces, len(v))
    fs = np.where(ok[:, None], faces, 0)
    a32, b32, c32 = (v[fs[:, j]] for j in range(3))
    with np.errstate(invalid="ignore", over="ignore"):
        degenerate = area2_f32((b32 - a32).astype(f32), (c32 - a32).astype(f32)) == 0
    a, b, c = (x.astype(f64)[None] for x in (a32, b32, c32))
    d = np.empty((len(p), len(faces)))
    for i in range(0, len(p), chunk):
        d[i:i + chunk] = triangle_dist2(p[i:i + chunk, None, :].astype(f64), a, b, c, degenerate[None])
    d = np.where(ok[None] & ~np.isnan(d), d, np.inf)
    face = d.argmin(1) if len(faces) else np.zeros(len(p), np.int64)
    best = d[np.arange(len(p)), face]
    face[~np.isfinite(best)] = 0
    return np.where(np.isfinite(best), best, np.inf), face, d


def grid(verts, pitch):
    """(lo fp32 [3], n [3]) of the object's voxel grid: n = max(1, ceil((hi - lo) / pitch)) per axis, quotient in float64"""
    v = np.asarray(verts, f32)
    lo, hi, p = v.min(0), v.max(0), f32(pitch)
    n = [max(1, int(math.ceil((float(h) - float(l)) / float(p)))) for l, h in zip(lo, hi)]
    if n[0] * n[1] * n[2] > MAX_CELLS:
        raise ValueError("cell cap")
    return lo, n


def voxel_centres(lo, n, pitch):
    """every cell centre fl(lo + fl((i + 0.5) pitch)) in (i, j, k) order, k fastest: [n0 n1 n2, 3] fp32"""
    ijk = np.stack(np.meshgrid(*[np.arange(k) for k in n], indexing="ij"), -1).reshape(-1, 3).astype(f32)
    return (np.asarray(lo, f32) + ((ijk + f32(0.5)).astype(f32) * f32(pitch)).astype(f32)).astype(f32)


def grasp_metrics(centres, obj_verts, obj_faces, hand_verts, hand_faces, pitch, contact_tol):
    """centres [M,3] (the object's kept voxel centres), hand_verts [B,Vh,3] -> dict of float64 per-hand results:
    count (centres with w64 >= 0.5), volume, depth, contact, and the per-hand winding numbers / distances they came from."""
    hv = np.asarray(hand_verts, f32)
    tol2 = float(f32(f32(contact_tol) * f32(contact_tol)))
    out = {k: [] for k in ("count", "w_centres", "w_verts", "dist2", "depth", "contact")}
    for b in range(len(hv)):
        wc = winding(centres, hv[b], hand_faces)
        wv = winding(hv[b], obj_verts, obj_faces)
        d2, _, _ = distance(hv[b], obj_verts, obj_faces)
        inside = wv >= 0.5
        out["count"].append(int((wc >= 0.5).sum()))
        out["w_centres"].append(wc)
        out["w_verts"].append(wv)
        out["dist2"].append(d2)
        out["depth"].append(float(np.sqrt(d2[inside]).max()) if inside.any() else 0.0)
        out["contact"].append(bool(inside.any() or (d2 <= tol2).any()))
    out = {k: np.array(v) for k, v in out.items()}
    out["volume"] = out["count"] * float(f32(pitch)) ** 3
    return out

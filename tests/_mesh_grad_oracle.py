"""float64 restatement of the gradient of the point-to-mesh squared distance (csrc/mesh_exact.cuh) at a given face, for
tests of dvq_mesh_distance_backward / dvq.penetration_depth.  It sits beside oracle/mesh_oracle.py and uses its fp32
degenerate-face decision.

The closest point is found independently of the kernel's region cascade: the projection onto the plane when it falls
inside the triangle, else the best of the three edge segments (a face with fp32 area^2 = 0 is its edges).  With the
closest point's barycentrics lam held fixed (the envelope theorem), d dist2 / d point = 2 (p - closest) and
d dist2 / d corner k = -2 lam_k (p - closest).
"""
import numpy as np

from oracle.mesh_oracle import area2_f32

f32, f64 = np.float32, np.float64


def closest_at_face(points, verts, faces, face):
    """points [Q,3], verts [V,3] float32, faces [F,3], face [Q] (valid ids) -> dict of float64 closest [Q,3], lam [Q,3]
    (the corners' weights), dist2 [Q], g_pts [Q,3] and g_corners [Q,3,3] (corner k's gradient)."""
    p = np.asarray(points, f32).astype(f64)
    v = np.asarray(verts, f32)
    tri = np.asarray(faces, np.int64).reshape(-1, 3)[np.asarray(face, np.int64)]
    a32, b32, c32 = (v[tri[:, j]] for j in range(3))
    degenerate = area2_f32((b32 - a32).astype(f32), (c32 - a32).astype(f32)) == 0
    a, b, c = (x.astype(f64) for x in (a32, b32, c32))
    best = np.full(len(p), np.inf)
    lam = np.zeros((len(p), 3))
    for (i, j), (s, e) in zip(((0, 1), (0, 2), (1, 2)), ((a, b), (a, c), (b, c))):
        d = e - s
        dd = (d * d).sum(-1)
        t = np.where(dd > 0, np.clip(((p - s) * d).sum(-1) / np.where(dd > 0, dd, 1), 0, 1), 0)
        r = p - s - t[:, None] * d
        d2 = (r * r).sum(-1)
        better = d2 < best
        best = np.where(better, d2, best)
        lam[better] = 0
        lam[better, i], lam[better, j] = 1 - t[better], t[better]
    n = np.cross(b - a, c - a)
    nn = (n * n).sum(-1)
    ok = (nn > 0) & ~degenerate
    den = np.where(ok, nn, 1)[:, None]
    proj = p - (((p - a) * n).sum(-1)[:, None] / den) * n
    # barycentrics of the projection from signed sub-triangle areas; the projection is inside when all are >= 0
    bary = np.stack([(np.cross(c - b, proj - b) * n).sum(-1), (np.cross(a - c, proj - c) * n).sum(-1),
                     (np.cross(b - a, proj - a) * n).sum(-1)], 1) / den
    plane = ok & np.all(bary >= 0, axis=1)
    lam[plane] = bary[plane]
    closest = (lam[:, :, None] * np.stack([a, b, c], 1)).sum(1)
    off = p - closest
    g_pts = 2 * off
    return {"closest": closest, "lam": lam, "dist2": (off * off).sum(-1), "g_pts": g_pts,
            "g_corners": -lam[:, :, None] * g_pts[:, None, :]}


def gradients(points, verts, faces, face, g):
    """float64 (g_pts [Q,3], g_verts [V,3]) of sum_i g[i] dist2_i at the faces face[i]; entries with face[i] < 0 add
    nothing"""
    face = np.asarray(face, np.int64)
    keep = face >= 0
    g = np.asarray(g, f64)
    g_pts = np.zeros((len(face), 3))
    g_verts = np.zeros((len(verts), 3))
    if keep.any():
        r = closest_at_face(np.asarray(points)[keep], verts, faces, face[keep])
        g_pts[keep] = g[keep, None] * r["g_pts"]
        tri = np.asarray(faces, np.int64).reshape(-1, 3)[face[keep]]
        for k in range(3):
            np.add.at(g_verts, tri[:, k], g[keep, None] * r["g_corners"][:, k])
    return g_pts, g_verts

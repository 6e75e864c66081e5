"""float32 restatement of the hand-object nearest-point contract (d-vqvae_b200/csrc/contact_exact.cuh) in numpy, for
bit-for-bit tests of dvq_nn_forward / dvq_nn_backward / dvq_vertex_normals.

numpy has no fp32 fused multiply-add, so ``fma_f32`` emulates one by rounding to odd: the float64 product of two float32
values is exact; the float64 sum with the addend is made sticky (when its TwoSum error is non-zero and its last bit is
even, it steps one ulp toward the error), and the final cast to float32 then rounds the exact result correctly, because
float64 carries more than 2 * 24 + 2 bits.  ``np.add.at`` on a float32 array adds in index order, which is the ascending
order of the contract's sums.
"""
import numpy as np

f32 = np.float32


def fma_f32(a, b, c):
    """fl32(a * b + c) with one rounding, elementwise over float32 arrays."""
    a, b, c = (np.asarray(x, dtype=np.float32).astype(np.float64) for x in (a, b, c))
    p = a * b                                   # exact: 24 + 24 bits
    with np.errstate(invalid="ignore", over="ignore"):
        s = p + c
        bb = s - p
        err = (p - (s - bb)) + (c - bb)         # TwoSum: s + err == p + c exactly (finite s)
        sticky = np.isfinite(s) & (err != 0) & ((s.view(np.int64) & 1) == 0)
    s = np.where(sticky, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    with np.errstate(over="ignore", invalid="ignore"):
        return s.astype(np.float32)


def sq_dist(s, t):
    """d = fma(dz, dz, fma(dy, dy, fl(dx * dx))), dv = fl(s - t); s [..., 3] and t [..., 3] broadcast."""
    with np.errstate(invalid="ignore", over="ignore"):
        dv = (np.asarray(s, f32) - np.asarray(t, f32)).astype(f32)
        dx, dy, dz = dv[..., 0], dv[..., 1], dv[..., 2]
        return fma_f32(dz, dz, fma_f32(dy, dy, (dx * dx).astype(f32))), dv


def nn_forward(src, trg, trg_normals=None, chunk=64):
    """src [B,N1,3], trg [B,N2,3] float32 -> (dist [B,N1] float32, idx [B,N1] int64, interior [B,N1] bool or None)."""
    src, trg = np.asarray(src, f32), np.asarray(trg, f32)
    B, N1, N2 = src.shape[0], src.shape[1], trg.shape[1]
    dist, idx = np.zeros((B, N1), f32), np.zeros((B, N1), np.int64)
    for b in range(B):
        for i0 in range(0, N1, chunk):
            d, _ = sq_dist(src[b, i0:i0 + chunk, None, :], trg[b, None, :, :])
            key = np.where(np.isnan(d), np.inf, d)
            j = np.argmin(key, axis=1)                          # the first index of the minimum
            j[key[np.arange(len(j)), j] == np.inf] = 0          # nothing below +inf: index 0
            idx[b, i0:i0 + chunk] = j
    if B * N1:
        dist, dv = sq_dist(src, np.take_along_axis(trg, idx[..., None], axis=1))
    interior = None
    if trg_normals is not None:
        interior = np.zeros((B, N1), bool)
        if B * N1:
            interior = interior_test(dv, np.take_along_axis(np.asarray(trg_normals, f32), idx[..., None], axis=1))
    return dist, idx, interior


def interior_test(dv, n):
    """dot(fl(t - s), n) > 0 with dot = fl(fl(fl(ax nx) + fl(ay ny)) + fl(az nz)) and fl(t - s) = -dv."""
    a = -np.asarray(dv, f32)
    with np.errstate(invalid="ignore", over="ignore"):
        dot = ((a[..., 0] * n[..., 0]).astype(f32) + (a[..., 1] * n[..., 1]).astype(f32)).astype(f32) + (a[..., 2] * n[..., 2]).astype(f32)
    return dot.astype(f32) > 0


def nn_backward(src, trg, idx, g_dist):
    """-> (g_src [B,N1,3], g_trg [B,N2,3]) float32: term_i = fl(fl(2 g) dv), g_src = term, g_trg[j] = -(ascending-i sum)."""
    src, trg, g = np.asarray(src, f32), np.asarray(trg, f32), np.asarray(g_dist, f32)
    B, N2 = src.shape[0], trg.shape[1]
    dv = (src - np.take_along_axis(trg, idx[..., None], axis=1)).astype(f32)
    term = ((f32(2) * g).astype(f32)[..., None] * dv).astype(f32)
    acc = np.zeros((B, N2, 3), f32)
    for b in range(B):
        np.add.at(acc[b], idx[b], term[b])
    return term, -acc


def vertex_normals(verts, faces):
    """verts [B,V,3] float32, faces [F,3] -> unit normals [B,V,3] float32 (area-weighted, F.normalize eps 1e-6)."""
    v = np.asarray(verts, f32)
    faces = np.asarray(faces, np.int64)
    B, V = v.shape[0], v.shape[1]
    out = np.zeros((B, V, 3), f32)
    for b in range(B):
        v0, v1, v2 = v[b, faces[:, 0]], v[b, faces[:, 1]], v[b, faces[:, 2]]
        a, c = (v2 - v1).astype(f32), (v0 - v1).astype(f32)
        cr = lambda i, j: ((a[:, i] * c[:, j]).astype(f32) - (a[:, j] * c[:, i]).astype(f32)).astype(f32)
        nf = np.stack([cr(1, 2), cr(2, 0), cr(0, 1)], axis=1)
        acc = np.zeros((V, 3), f32)
        np.add.at(acc, faces.reshape(-1), np.repeat(nf, 3, axis=0))    # face-major: ascending f per vertex
        n2 = (((acc[:, 0] * acc[:, 0]).astype(f32) + (acc[:, 1] * acc[:, 1]).astype(f32)).astype(f32)
              + (acc[:, 2] * acc[:, 2]).astype(f32)).astype(f32)
        den = np.maximum(np.sqrt(n2), f32(1e-6)).astype(f32)
        out[b] = (acc / den[:, None]).astype(f32)
    return out


def brute_force64(src, trg):
    """float64 reference: squared distances [B,N1,N2] and their argmin (small shapes only)."""
    d = ((np.asarray(src, np.float64)[:, :, None, :] - np.asarray(trg, np.float64)[:, None, :, :]) ** 2).sum(-1)
    return d, d.argmin(-1)

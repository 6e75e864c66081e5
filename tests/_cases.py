"""Shared case table: regenerates the seeded inputs of oracle/gen_golden.py
without the reference (numpy legacy RandomState is bit-stable)."""
import hashlib
import os

import numpy as np

from oracle import vq_oracle as vo

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

VQ_CASES = {
    "vq_k512_d64": (1024, 512, 64, 1.0, 0.25, "default", None),
    "vq_k128_d256": (512, 128, 256, 1.0, 0.25, "default", None),
    "vq_k128_d1024": (256, 128, 1024, 0.0, 2.0, "default", None),
    "vq_variant_b": (1024, 512, 64, 1.0, 0.25, "variant_b", None),
    "vq_dupes": (777, 64, 16, 1.0, 0.25, "dupes", None),
    "vq_3d_view": (4 * 9 * 5, 96, 24, 0.5, 0.75, "default", (4, 9, 5, 24)),
    "vq_ragged": (333, 200, 40, 1.0, 0.25, "default", None),
    "vq_one_row": (1, 128, 256, 1.0, 0.25, "default", None),
}
PN_CASES = ["pointnet_c4_p3000", "pointnet_c3_p778", "pointnet_c4_p100", "pointnet_c4_p129"]


def vq_inputs(name):
    n, k, d, al, beta, kind, shape = VQ_CASES[name]
    seed = int(hashlib.sha256(name.encode()).hexdigest()[:6], 16)
    if kind == "variant_b":
        z, E = vo.variant_b(n, k, d, seed)
    else:
        E = vo.default_codebook(k, d, seed)
        z = vo.normal_latents(n, d, seed + 1)
        if kind == "dupes":
            E[k // 2:] = E[:k // 2]
    if shape is not None:
        z = z.reshape(shape)
    return z, E, al, beta


def load_gold(name):
    """Where a VQ case's z_q arrays would make its file larger than 1 MB, the file keeps their SHA-256 instead: they
    are rebuilt from the seeded inputs and the reference's indices (z_q is bit-exact given the index) and must match."""
    g = np.load(os.path.join(GOLD, name + ".npz"))
    if name not in VQ_CASES or "zq_train" in g.files:
        return g
    g = dict(g)
    z, E, _, _ = vq_inputs(name)
    for key, zq in (("zq_train", vo.zq_train_from_idx(z, E, g["idx_train"].astype(np.int64))),
                    ("zq_infer", vo.zq_infer_from_idx(E, g["idx_infer"].astype(np.int64)))):
        zq = np.ascontiguousarray(zq.reshape(z.shape))
        assert hashlib.sha256(zq.tobytes()).hexdigest() == str(g.pop(key + "_sha256")), (name, key)
        g[key] = zq
    return g


def rel_err(a, b):
    a, b = float(a), float(b)
    return abs(a - b) / max(abs(b), 1e-30)

"""GPU: pins the tcgen05 shared-memory descriptor convention the VQ kernel relies on
(K-major, no swizzle: 8x16-byte core matrices, LBO = byte stride between core matrices along K,
SBO = along M/N) by running real tcgen05.mma on caller-built operand images and comparing the
TMEM accumulator with a CPU matmul."""
import ctypes
import json

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def build_image(vals: np.ndarray, lbo: int, sbo: int, total: int) -> np.ndarray:
    """vals [rows, Kp] fp16 -> byte image with offset(r,k) = (k//8)*lbo + (r//8)*sbo + (r%8)*16 + (k%8)*2."""
    rows, kp = vals.shape
    img = np.zeros(total, dtype=np.uint8)
    r = np.arange(rows)[:, None]
    k = np.arange(kp)[None, :]
    off = (k // 8) * lbo + (r // 8) * sbo + (r % 8) * 16 + (k % 8) * 2
    raw = vals.view(np.uint16)
    img_u16 = img.view(np.uint16)
    img_u16[(off // 2).reshape(-1)] = raw.reshape(-1)
    return img


def run_probe(A, B, a_lbo, a_sbo, b_lbo, b_sbo, desc=None):
    from dvq import _cabi
    m, kp = A.shape
    n = B.shape[0]
    a_total = (kp // 8) * a_lbo if a_lbo > a_sbo else (m // 8) * a_sbo
    b_total = (kp // 8) * b_lbo if b_lbo > b_sbo else (n // 8) * b_sbo
    a_total = (a_total + 15) // 16 * 16
    b_total = (b_total + 15) // 16 * 16
    a_img = torch.from_numpy(build_image(A, a_lbo, a_sbo, a_total)).cuda()
    b_img = torch.from_numpy(build_image(B, b_lbo, b_sbo, b_total)).cuda()
    d = desc or (a_lbo, a_sbo, 2 * a_lbo, b_lbo, b_sbo, 2 * b_lbo)
    strides = (ctypes.c_uint32 * 6)(*d)
    idesc = (1 << 4) | ((n >> 3) << 17) | ((128 >> 4) << 24)
    out = torch.full((128, n), float("nan"), device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    _cabi.check(_cabi.lib.dvq_debug_umma(a_img.data_ptr(), a_total, b_img.data_ptr(), b_total, kp // 16, strides, idesc, n,
                                         out.data_ptr(), err.data_ptr(), None), "dvq_debug_umma")
    torch.cuda.synchronize()
    return out.cpu().numpy(), int(err.item())


def test_umma_descriptor_convention():
    rs = np.random.RandomState(0)
    report = {}
    for n in (256, 128):
        kp = 80
        A = rs.standard_normal((128, kp)).astype(np.float16)
        B = rs.standard_normal((n, kp)).astype(np.float16)
        ref = A.astype(np.float32) @ B.astype(np.float32).T
        variants = {
            # image [kchunk][rowgroup][8][16B]; A k-chunk blocks padded by 32 B (bank spreading)
            "kchunk_major_padded": dict(a_lbo=128 * 16 + 32, a_sbo=128, b_lbo=n * 16, b_sbo=128),
            # image [rowgroup][kchunk][8][16B]
            "rowgroup_major": dict(a_lbo=128, a_sbo=(kp // 8) * 128, b_lbo=128, b_sbo=(kp // 8) * 128),
        }
        for name, v in variants.items():
            got, err = run_probe(A, B, **v)
            bad = float(np.nanmax(np.abs(got - ref))) if not np.isnan(got).all() else float("inf")
            report["%s_n%d" % (name, n)] = dict(err=err, max_abs_diff=bad, nan=int(np.isnan(got).sum()))
    print(json.dumps(report))
    for key in ("kchunk_major_padded_n256", "kchunk_major_padded_n128", "rowgroup_major_n256", "rowgroup_major_n128"):
        assert report[key]["err"] == 0 and report[key]["max_abs_diff"] < 2e-2, report

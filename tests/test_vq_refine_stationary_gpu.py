"""GPU: the code-stationary exact refine (csrc/vq_refine_stationary.cu) against the per-row refine and the all-FP32 kernel.

The stationary kernel covers the mask-mode codebooks whose K/32 warps hold e_dim code floats per lane in registers: every
K <= 992 at e_dim 16, K <= 512 at e_dim 32 / 64, K <= 256 at e_dim 128.  On those shapes it must give the per-row kernel's
idx, z_q and usage histogram bit for bit (same FP32 expression per (row, code), same lexicographic (distance, code)
minimum), and loss / perplexity up to the order of the fp64 SSE sum.  Against the all-FP32 kernel: every index within
the near-tie rule, bit-identical on the degenerate rows (zero / huge: the refine scans every code for them)."""
import numpy as np
import pytest
import torch

from oracle import vq_oracle as vo
from _cases import rel_err

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
SIMT, TC = 0x10, 0x20
AUTO_MODE, PER_ROW, STATIONARY = 0, 1, 3
# each e_dim at the smallest K, one inside and the largest K the kernel covers
COVERED = [(32, 16), (544, 16), (992, 16), (32, 32), (224, 32), (512, 32), (32, 64), (160, 64), (512, 64),
           (32, 128), (96, 128), (256, 128)]


def _set_refine(mode):
    from dvq import _cabi
    _cabi.check(_cabi.lib.dvq_vq_set_refine(mode, 0), "dvq_vq_set_refine")


def _module(E, path):
    import dvq
    m = dvq.VectorQuantizer(E.shape[0], E.shape[1], 0.25, 1.0).cuda()
    with torch.no_grad():
        m.embedding.weight.copy_(torch.from_numpy(E))
    m.path = path
    m.onehot_limit_bytes = 0
    return m


def _run(E, zt, path, mode):
    """One train call with the refine mode forced; (idx, z_q bits, histogram, loss, ppl, rows refined)."""
    K = E.shape[0]
    N = zt.shape[0]
    try:
        _set_refine(mode)
        m = _module(E, path)
        with torch.no_grad():
            loss, zq, ppl, _, idx = m(zt, True)
        n_ref, err = m.last_counters(N)
    finally:
        _set_refine(AUTO_MODE)
    assert err == 0
    bits = zq.view(torch.int16 if zq.dtype == BF else torch.int32)
    return (idx.reshape(-1).cpu().numpy(), bits.cpu().numpy(), m.last_stats[:K].cpu().numpy(), loss.item(), ppl.item(), n_ref)


def _latents(N, D, seed):
    z = vo.normal_latents(N, D, seed)
    z[::211] = 0.0          # degenerate rows: every sub-chunk is a candidate
    z[3::307] *= 1e18
    return z


def _compare(E, z, zt):
    st = _run(E, zt, TC, STATIONARY)
    pr = _run(E, zt, TC, PER_ROW)
    simt = _run(E, zt, SIMT, AUTO_MODE)
    assert st[5] > 0 and st[5] == pr[5]                      # the refine stage ran, on the same list
    for a, what in ((0, "idx"), (1, "z_q"), (2, "histogram")):
        assert np.array_equal(st[a], pr[a]), what
    assert rel_err(st[3], pr[3]) < 1e-7 and rel_err(st[4], pr[4]) < 1e-7
    zu = zt.float().cpu().numpy()
    n_mis, n_bad, worst = vo.allowed_index_mismatch(zu, E, st[0], simt[0])
    assert n_bad == 0, (n_mis, worst)
    same = st[0] == simt[0]
    assert np.array_equal(st[1][same], simt[1][same])
    degenerate = np.zeros(len(z), bool)
    degenerate[::211] = True
    degenerate[3::307] = True
    assert np.array_equal(st[0][degenerate], simt[0][degenerate])
    assert rel_err(st[3], simt[3]) < 1e-5
    return st


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("K,D", COVERED)
def test_stationary_equals_per_row_and_fp32(K, D, dtype):
    """Default-init codebook (a few % undecided rows) plus zero / huge rows; N is not a multiple of the 128-row batch."""
    N = 50000 + 13
    E = vo.default_codebook(K, D, 61)
    z = _latents(N, D, 62)
    zt = torch.from_numpy(z).cuda()
    if dtype == "bf16":
        zt = zt.to(BF)
    _compare(E, z, zt)


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_stationary_config2_size(dtype):
    """Config 2's shape (K = 512, e_dim 64) at 3M rows: ~80 k listed rows, several staged batches per CTA."""
    N = 3000000 + 17
    E = vo.default_codebook(512, 64, 71)
    z = _latents(N, 64, 72)
    zt = torch.from_numpy(z).cuda()
    if dtype == "bf16":
        zt = zt.to(BF)
    st = _compare(E, z, zt)
    assert st[5] > 148 * 3 * 128


def test_stationary_empty_list():
    """A tie-free input the filter decides completely: the refine kernel runs on an empty list and changes nothing."""
    z, E = vo.variant_b(40000 + 3, 512, 64, 81)
    zt = torch.from_numpy(z).cuda()
    st = _run(E, zt, TC, STATIONARY)
    simt = _run(E, zt, SIMT, AUTO_MODE)
    assert st[5] == 0
    assert np.array_equal(st[0], simt[0]) and np.array_equal(st[1], simt[1]) and np.array_equal(st[2], simt[2])


@pytest.mark.parametrize("K,D", [(544, 32), (544, 64), (288, 128), (128, 256), (1024, 16)])
def test_stationary_rejects_shapes_it_does_not_cover(K, D):
    """Forcing the stationary kernel on a shape outside its register budget (or in list mode) is an error, not a silent
    fall-back; the automatic choice still runs those shapes."""
    E = vo.default_codebook(K, D, 91)
    zt = torch.from_numpy(vo.normal_latents(3000, D, 92)).cuda()
    try:
        _set_refine(STATIONARY)
        m = _module(E, TC)
        with pytest.raises(RuntimeError, match="code-stationary"):
            with torch.no_grad():
                m(zt, True)
    finally:
        _set_refine(AUTO_MODE)
    m = _module(E, TC)
    with torch.no_grad():
        m(zt, True)
    assert m.last_counters(3000)[1] == 0

"""GPU: bf16 latents (DVQ_Z_BF16).  The bf16 call is defined as the fp32 call on z.float(): idx and the usage histogram
bit-identical, z_q the fp32 z_q rounded to nearest-even bf16, loss / perplexity within 1e-6; the backward's dz is bf16
(the fp32 formulas on the upcast values, rounded once) and dE fp32.  The fp32 call is itself pinned to the reference by
tests/test_vq_gpu.py, so most checks here compare the two calls of this library."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import vq_oracle as vo
from _cases import VQ_CASES, rel_err, vq_inputs

pytestmark = pytest.mark.gpu

BF = torch.bfloat16
SIMT, AUTO, TC = 0x10, 0x00, 0x20
CONFIG4_SHAPES = [(K, D) for K in (512, 1024, 2048, 4096, 8192, 16384) for D in (64, 128, 256, 512)]
EXTRA_SHAPES = [(800, 64), (1536, 32), (128, 256), (992, 128), (960, 256), (32, 16), (256, 32)]


def _module(E, path, al=1.0, beta=0.25):
    import dvq
    E = torch.as_tensor(E)
    m = dvq.VectorQuantizer(E.shape[0], E.shape[1], beta, al).cuda()
    with torch.no_grad():
        m.embedding.weight.copy_(E)
    m.path = path
    m.onehot_limit_bytes = 0
    return m


def _bits_equal(a, b):
    """Bit equality of two tensors of one dtype; positions where both are NaN count as equal."""
    a, b = a.detach(), b.detach()
    assert a.dtype == b.dtype and a.shape == b.shape
    nan = torch.isnan(a) & torch.isnan(b)
    iv = {torch.float32: torch.int32, BF: torch.int16}[a.dtype]
    return bool(torch.equal(a[~nan].view(iv), b[~nan].view(iv))) and bool(torch.equal(torch.isnan(a), torch.isnan(b)))


def _scalar_close(a, b, tol=1e-6):
    a, b = (float(x.detach()) if torch.is_tensor(x) else float(x) for x in (a, b))
    if np.isnan(a) or np.isnan(b):
        return np.isnan(a) and np.isnan(b)
    return a == b or rel_err(a, b) <= tol


def _calls(E, zb, path, train):
    """(bf16 call, fp32 call on the upcast z) on two fresh modules; returns their outputs and last_stats."""
    out = []
    for z in (zb, zb.float()):
        m = _module(E, path)
        with torch.no_grad():
            o = m(z, train)
        out.append((o, m.last_stats.clone() if train else None, m))
    return out


def _assert_contract(E, zb, path, train, counters=False):
    K = E.shape[0]
    (ob, sb, mb), (of, sf, mf) = _calls(E, zb, path, train)
    if train:
        lb, qb, pb, _, ib = ob
        lf, qf, pf, _, if_ = of
        assert lb.dtype == torch.float32 and pb.dtype == torch.float32
        assert _scalar_close(lb, lf) and _scalar_close(pb, pf), (lb.item(), lf.item(), pb.item(), pf.item())
        assert torch.equal(sb[:K], sf[:K])
    else:
        ib, qb = ob
        if_, qf = of
    assert qb.dtype == BF and qb.shape == zb.shape
    assert torch.equal(ib, if_)
    assert _bits_equal(qb, qf.to(BF))
    if counters:
        n = zb.numel() // E.shape[1]
        assert mb.last_counters(n)[1] == 0 and mf.last_counters(n)[1] == 0
    return ib, qb


# 1 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("pname,path", [("simt", SIMT), ("auto", AUTO)])
@pytest.mark.parametrize("name", list(VQ_CASES))
def test_golden_cases_bf16_equal_fp32_call(name, pname, path):
    z, E, al, beta = vq_inputs(name)
    zb = torch.from_numpy(z).cuda().to(BF)
    zu = zb.float().cpu().numpy().reshape(-1, E.shape[1])
    ridx, _ = vo.forward_infer(zu, E)
    for train in (True, False):
        idx, zq = _assert_contract(E, zb, path, train)
        n_mis, n_bad, worst = vo.allowed_index_mismatch(zu, E, idx.cpu().numpy(), ridx)
        assert n_bad == 0, (train, n_mis, worst)
        # z_q is the oracle's z_q of the upcast rows given our index, rounded to bf16
        want = vo.zq_train_from_idx(zu, E, idx.cpu().numpy()) if train else vo.zq_infer_from_idx(E, idx.cpu().numpy())
        assert _bits_equal(zq.reshape(-1, E.shape[1]).cpu(), torch.from_numpy(np.ascontiguousarray(want)).reshape(-1, E.shape[1]).to(BF))


# 2 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,D", CONFIG4_SHAPES + EXTRA_SHAPES)
@pytest.mark.parametrize("variant", ["default", "variant_b"])
def test_streamed_shapes_bf16_equal_fp32_call(K, D, variant):
    N = (20000 if K * D <= 2048 * 512 else 6000) + 37
    if variant == "default":
        E = vo.default_codebook(K, D, 31)
        z = vo.normal_latents(N, D, 32)
    else:
        z, E = vo.variant_b(N, K, D, 33)
    zb = torch.from_numpy(z).cuda().to(BF)
    for path in (TC, SIMT):
        _assert_contract(E, zb, path, True, counters=True)


# 3 ---------------------------------------------------------------------------------------------------------------------
_VARIANT_SNIPPET = r"""
import os, sys
import torch
root = sys.argv[1]
sys.path.insert(0, root); sys.path.insert(0, os.path.join(root, "d-vqvae_b200"))
import dvq
from oracle import vq_oracle as vo
for K, D in ((4096, 64), (2048, 32), (1024, 128), (2048, 256), (544, 128), (1024, 512)):
    N = 30000 + 19
    E = vo.default_codebook(K, D, 51); z = torch.from_numpy(vo.normal_latents(N, D, 52)).cuda().to(torch.bfloat16)
    z[::199] = 0.0
    out = []
    for zz in (z, z.float()):
        m = dvq.VectorQuantizer(K, D, 0.25, 1.0).cuda(); m.path = 0x20; m.onehot_limit_bytes = 0
        with torch.no_grad():
            m.embedding.weight.copy_(torch.from_numpy(E))
            loss, zq, ppl, _, idx = m(zz, True)
        assert m.last_counters(N)[1] == 0
        out.append((idx, zq, m.last_stats.clone(), loss.item()))
    (ib, qb, sb, lb), (i32, q32, s32, l32) = out
    assert qb.dtype == torch.bfloat16
    assert torch.equal(ib, i32) and torch.equal(sb[:K], s32[:K]), (K, D)   # (sb[K]: the SSE, an fp64 sum by atomics)
    assert torch.equal(qb.view(torch.int16), q32.to(torch.bfloat16).view(torch.int16)), (K, D)
    assert abs(lb - l32) <= 1e-6 * abs(l32), (K, D, lb, l32)
print("VARIANT_OK")
"""


@pytest.mark.parametrize("pair", ["0", "1"], ids=["single_cta_only", "cta_pair_everywhere"])
def test_kernel_variants_bf16_equal_fp32_call(pair):
    """DVQ_TC_PAIR=0 / 1 (read once per process: a fresh interpreter each): odd tile count, ragged last chunk (K = 544),
    e_dim 512."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _VARIANT_SNIPPET, root], env=dict(os.environ, DVQ_TC_PAIR=pair),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "VARIANT_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])


# 4 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,D", [(512, 64), (2048, 64), (1024, 256), (128, 256)])
def test_refine_modes_bf16_identical(K, D):
    """Per-row refine, binned refine and the binned -> per-row hand-back (pair_cap = 64) on bf16 rows incl. zero and huge
    rows: identical to each other and to the fp32 call with the same mode."""
    from dvq import _cabi
    N = 50000 + 13
    E = vo.default_codebook(K, D, 41)
    z = vo.normal_latents(N, D, 42)
    z[::211] = 0.0
    z[3::307] *= 1e18
    zb = torch.from_numpy(z).cuda().to(BF)
    res = {}
    try:
        for name, mode, cap in (("per_row", 1, 0), ("binned", 2, 0), ("handback", 2, 64)):
            _cabi.check(_cabi.lib.dvq_vq_set_refine(mode, cap), "dvq_vq_set_refine")
            idx, zq = _assert_contract(E, zb, TC, True, counters=True)
            m = _module(E, TC)
            with torch.no_grad():
                m(zb, True)
            assert m.last_counters(N)[0] > 0                     # the refine stage did run
            res[name] = (idx, zq)
    finally:
        _cabi.check(_cabi.lib.dvq_vq_set_refine(0, 0), "dvq_vq_set_refine")
    for name in ("binned", "handback"):
        assert torch.equal(res[name][0], res["per_row"][0]) and _bits_equal(res[name][1], res["per_row"][1]), name


# 5 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,D", [(512, 64), (2048, 64), (2048, 128)])
def test_degenerate_rows_and_duplicate_codes_bf16(K, D):
    N = 3000 + 11
    rng = np.random.default_rng(5)
    half = (rng.standard_normal((K // 2, D)) * 0.05).astype(np.float32)
    half = torch.from_numpy(half).to(BF).float().numpy()          # codes exactly representable in bf16
    E = np.concatenate([half, half], axis=0)
    z = rng.standard_normal((N, D)).astype(np.float32)
    z[::97] = 0.0                      # zero rows
    z[5::101] *= 1e18                  # outside the FP16 fold range
    z[7::103] = half[rng.integers(0, K // 2, size=len(z[7::103]))]   # exactly on a (duplicated) code
    z[11::211] = np.inf
    z[13::223, 3] = np.nan
    z[17::227, :2] = -np.inf
    other = set(range(0, N, 97)) | set(range(5, N, 101)) | set(range(11, N, 211)) | set(range(13, N, 223)) | set(range(17, N, 227))
    on_code = sorted(set(range(7, N, 103)) - other)
    zb = torch.from_numpy(z).cuda().to(BF)
    for path in (TC, SIMT):
        for train in (False, True):
            idx, _ = _assert_contract(E, zb, path, train, counters=path == TC)
            assert int(idx[on_code].max()) < K // 2               # exact ties -> lowest index


# 6 ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("variant", ["default", "variant_b"])
def test_config2_full_size_bf16_equal_fp32_call(variant):
    N, K, D = 4194304, 512, 64
    gen = torch.Generator(device="cuda").manual_seed(2000)
    if variant == "default":
        E = (torch.rand(K, D, device="cuda", generator=gen) * 2 - 1) / K
        z = torch.randn(N, D, device="cuda", generator=gen)
    else:
        E = torch.randn(K, D, device="cuda", generator=gen)
        z = E[torch.randint(0, K, (N,), device="cuda", generator=gen)] + 0.1 * torch.randn(N, D, device="cuda", generator=gen)
    zb = z.to(BF)
    del z
    _assert_contract(E.cpu(), zb, AUTO, True, counters=True)


# 7 ---------------------------------------------------------------------------------------------------------------------
def _ulp_bf16(x):
    _, e = torch.frexp(x.float())
    return torch.ldexp(torch.ones_like(x, dtype=torch.float32), e - 8)


def _torch_reference_grads(zb, E, idx, al, beta, g_loss, g_zq, rows=None):
    z = zb.detach().float().requires_grad_()
    w = torch.as_tensor(E).cuda().float().requires_grad_()
    zq = w[idx.view(-1)].view_as(z)
    n = z.numel() if rows is None else rows * z.shape[-1]
    loss = al * ((zq.detach() - z) ** 2).sum() / n + beta * ((zq - z.detach()) ** 2).sum() / n
    out = z + (zq - z).detach()
    torch.autograd.backward([loss, out], [g_loss, g_zq.float()])
    return z.grad, w.grad


@pytest.mark.parametrize("case", ["fused_k512_d64", "fused_k128_d256", "simt_d24", "fallback_d30", "fallback_odd_offset"])
def test_autograd_bf16(case):
    """dz (bf16) within one bf16 ulp of torch autograd in fp32 on the upcast values, rounded; dE (fp32) within 1e-5.  The
    fused backward kernel (tcgen05 and FP32 forward shapes) and the torch fallback (e_dim 30; a 2-byte aligned view)."""
    K, D, path, odd = {"fused_k512_d64": (512, 64, AUTO, False), "fused_k128_d256": (128, 256, AUTO, False),
                       "simt_d24": (96, 24, AUTO, False), "fallback_d30": (96, 30, AUTO, False),
                       "fallback_odd_offset": (512, 64, AUTO, True)}[case]
    N = 4096 + 5
    E = vo.default_codebook(K, D, 71)
    z = torch.from_numpy(vo.normal_latents(N, D, 72)).cuda().to(BF)
    if odd:   # a view 2 bytes into its storage: neither the tcgen05 path nor the vector backward kernel takes it
        buf = torch.empty(N * D + 1, dtype=BF, device="cuda")
        buf[1:].copy_(z.view(-1))
        z = buf[1:].view(N, D)
    al, beta = 0.5, 0.75
    m = _module(E, path, al, beta)
    zin = z.detach().clone() if not odd else z.detach()
    zin.requires_grad_()
    loss, zq, ppl, _, idx = m(zin, True)
    assert zq.dtype == BF and loss.dtype == torch.float32
    g_zq = torch.randn(N, D, device="cuda").to(BF)
    g_loss = torch.tensor(1.7, device="cuda")
    torch.autograd.backward([loss, zq], [g_loss, g_zq])
    dz_ref, dE_ref = _torch_reference_grads(z, E, idx, al, beta, g_loss, g_zq)
    assert zin.grad.dtype == BF and m.embedding.weight.grad.dtype == torch.float32
    ref16 = dz_ref.to(BF)
    diff = (zin.grad.float() - ref16.float()).abs()
    assert bool((diff <= torch.maximum(_ulp_bf16(ref16), _ulp_bf16(zin.grad))).all()), float(diff.max())
    gw = m.embedding.weight.grad
    assert float((gw - dE_ref).abs().max()) <= 1e-5 * float(dE_ref.abs().max()) + 1e-12


def test_backward_ex_sharded_row_count_bf16():
    """dvq_vq_backward_ex with DVQ_Z_BF16 and a row count that is not the local N (row-sharded loss): equals the fp32
    formulas on the upcast values, dz rounded once."""
    from dvq import _cabi
    K, D, N = 512, 64, 10000 + 3
    E = torch.from_numpy(vo.default_codebook(K, D, 81)).cuda()
    zb = torch.from_numpy(vo.normal_latents(N, D, 82)).cuda().to(BF)
    idx = torch.randint(0, K, (N,), device="cuda")
    gq = torch.randn(N, D, device="cuda").to(BF)
    gl = torch.tensor([0.9], device="cuda")
    rows = torch.tensor([3.0 * N], device="cuda")
    al, beta = 1.0, 0.25
    dz = torch.empty_like(zb)
    dE = torch.zeros_like(E)
    _cabi.check(_cabi.lib.dvq_vq_backward_ex(zb.data_ptr(), E.data_ptr(), idx.data_ptr(), gq.data_ptr(), gl.data_ptr(),
                                             rows.data_ptr(), N, K, D, al, beta, _cabi.DVQ_Z_BF16, dz.data_ptr(), dE.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream), "dvq_vq_backward_ex")
    torch.cuda.synchronize()
    scale = 2.0 * 0.9 / (3.0 * N * D)
    d = zb.float() - E[idx]
    ref = (scale * al * d + gq.float()).to(BF)
    diff = (dz.float() - ref.float()).abs()
    assert bool((diff <= _ulp_bf16(ref)).all())
    ref_e = torch.zeros_like(E).index_add_(0, idx, -scale * beta * d)
    assert float((dE - ref_e).abs().max()) <= 1e-5 * float(ref_e.abs().max())


# 8 ---------------------------------------------------------------------------------------------------------------------
def test_autocast_end_to_end():
    """nn.Linear -> VectorQuantizer under torch.autocast("cuda", bfloat16), loss.backward(): the quantizer sees the bf16
    activations; its outputs and gradients equal the explicit bf16 call on the same activations."""
    K, D, N = 512, 64, 8192 + 7
    torch.manual_seed(3)
    lin = torch.nn.Linear(32, D).cuda()
    x = torch.randn(N, 32, device="cuda")
    m = _module(vo.default_codebook(K, D, 91), AUTO)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        h = lin(x)
        h.retain_grad()
        loss, zq, ppl, enc, idx = m(h, True)
        total = loss + (zq.float() ** 2).mean()
    assert h.dtype == BF and zq.dtype == BF and loss.dtype == torch.float32
    total.backward()
    assert lin.weight.grad is not None and bool(torch.isfinite(lin.weight.grad).all())
    g_auto, gw_auto = h.grad.clone(), m.embedding.weight.grad.clone()
    m.embedding.weight.grad = None
    h2 = h.detach().clone().requires_grad_()
    loss2, zq2, ppl2, _, idx2 = m(h2, True)
    (loss2 + (zq2.float() ** 2).mean()).backward()
    assert torch.equal(idx, idx2) and _bits_equal(zq.detach(), zq2.detach())
    assert _scalar_close(loss, loss2) and ppl.item() == ppl2.item()
    assert _bits_equal(g_auto, h2.grad)
    assert torch.allclose(gw_auto, m.embedding.weight.grad, rtol=1e-6, atol=1e-9)


# 9 ---------------------------------------------------------------------------------------------------------------------
def test_ema_hooks_bf16_equal_fp32():
    K, D, N = 512, 64, 20000 + 1
    E = vo.default_codebook(K, D, 95)
    zb = torch.from_numpy(vo.normal_latents(N, D, 96)).cuda().to(BF)
    mods = []
    for z in (zb, zb.float()):
        m = _module(E, AUTO)
        with torch.no_grad():
            _, _, _, _, idx = m(z, True)
        sums = m.code_sums(z, idx)
        assert sums.dtype == torch.float32
        hist = m.ema_update(z, idx, decay=0.9)
        mods.append((m, idx, sums, hist))
    (mb, ib, sb, hb), (mf, if_, sf, hf) = mods
    assert torch.equal(ib, if_) and torch.equal(hb, hf)
    # (per-code fp32 sums by atomic adds: the order of the additions may differ between the calls)
    assert torch.allclose(sb, sf, rtol=1e-5, atol=1e-5)
    assert torch.allclose(mb.embedding.weight, mf.embedding.weight, rtol=1e-5, atol=1e-7)
    ref = torch.zeros(K, D, device="cuda").index_add_(0, ib.view(-1), zb.float())
    assert torch.allclose(sb, ref, rtol=1e-5, atol=1e-5)
    # index_add_ fallback (e_dim not a multiple of 4) upcasts
    m = _module(vo.default_codebook(96, 30, 97), AUTO)
    z24 = torch.from_numpy(vo.normal_latents(999, 30, 98)).cuda().to(BF)
    with torch.no_grad():
        _, _, _, _, i24 = m(z24, True)
    assert torch.allclose(m.code_sums(z24, i24), m.code_sums(z24.float(), i24), rtol=1e-5, atol=1e-5)
    # usage reset draws the same rows
    g1, g2 = torch.Generator(device="cuda").manual_seed(5), torch.Generator(device="cuda").manual_seed(5)
    ma, mf2 = _module(E, AUTO), _module(E, AUTO)
    with torch.no_grad():
        ma(zb[:300], True)
        mf2(zb[:300].float(), True)
    assert ma.reset_unused_codes(zb[:300], 1, g1) == mf2.reset_unused_codes(zb[:300].float(), 1, g2) > 0
    assert torch.equal(ma.embedding.weight, mf2.embedding.weight)


# 10 --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,D", [(512, 64), (4096, 128)])
def test_codebook_cache_with_interleaved_dtypes(K, D):
    N = 20000 + 37
    E = vo.default_codebook(K, D, 101)
    z32 = torch.from_numpy(vo.normal_latents(N, D, 102)).cuda()
    zb = z32.to(BF)
    cached, fresh = _module(E, AUTO), _module(E, AUTO)
    fresh.cache_codebook = False
    for z in (z32, zb, z32, zb):
        with torch.no_grad():
            a = cached(z, True)
            b = fresh(z, True)
        assert torch.equal(a[4], b[4]) and _bits_equal(a[1], b[1]) and _scalar_close(a[0], b[0])
        assert torch.equal(cached.last_stats[:K], fresh.last_stats[:K])   # (the histogram; [K] holds the SSE)


# 11 --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,D", [(512, 64), (2048, 128), (1024, 512)], ids=["resident", "cta_pair_d128", "cta_pair_d512"])
def test_cuda_graph_replay_bf16(K, D):
    N = 20000 + 37
    m = _module(vo.default_codebook(K, D, 61), TC)
    z_static = torch.from_numpy(vo.normal_latents(N, D, 62)).cuda().to(BF)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.no_grad():
        for _ in range(2):
            m(z_static, False)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph), torch.no_grad():
        idx_g, zq_g = m(z_static, False)
    for seed in (63, 64):
        z_new = torch.from_numpy(vo.normal_latents(N, D, seed)).cuda().to(BF)
        z_static.copy_(z_new)
        graph.replay()
        torch.cuda.synchronize()
        with torch.no_grad():
            idx_e, zq_e = m(z_new, False)
        assert torch.equal(idx_g, idx_e) and _bits_equal(zq_g, zq_e), (K, D, seed)
    assert m.last_counters(N)[1] == 0


# 12 --------------------------------------------------------------------------------------------------------------------
def test_alignment_and_validation_bf16():
    import dvq
    from dvq import _cabi
    K, D, N = 512, 64, 5000 + 3
    E = vo.default_codebook(K, D, 111)
    z = torch.from_numpy(vo.normal_latents(N, D, 112)).cuda().to(BF)
    buf = torch.empty(N * D + 1, dtype=BF, device="cuda")
    buf[1:].copy_(z.view(-1))
    zv = buf[1:].view(N, D)                              # 2-byte aligned view
    assert zv.data_ptr() % 16 == 2
    for train in (True, False):
        a = _module(E, AUTO)(zv, train)
        b = _module(E, AUTO)(zv.clone(), train)
        ia, qa = (a[4], a[1]) if train else a
        ib, qb = (b[4], b[1]) if train else b
        assert torch.equal(ia, ib) and _bits_equal(qa, qb)
        if train:
            assert _scalar_close(a[0], b[0])
    with pytest.raises(RuntimeError, match="BAD_ALIGN"):
        with torch.no_grad():
            _module(E, TC)(zv, False)
    # dtypes other than fp32 / bf16 and a bf16 codebook keep failing
    with pytest.raises(TypeError):
        _module(E, AUTO)(z.half(), False)
    with pytest.raises(TypeError):
        _module(E, AUTO)(z.double(), False)
    mb = dvq.VectorQuantizer(K, D, 0.25, 1.0).cuda().to(BF)
    with pytest.raises(ValueError):
        mb(z, False)
    # the host-buffer entry is fp32-only
    ctx = ctypes.c_void_p()
    _cabi.check(_cabi.lib.dvq_host_ctx_create(1024, K, D, ctypes.byref(ctx)), "dvq_host_ctx_create")
    try:
        zh = np.zeros((16, D), np.float32)
        eh = np.ascontiguousarray(E)
        zq = np.zeros((16, D), np.float32)
        ih = np.zeros(16, np.int64)
        rc = _cabi.lib.dvq_vq_forward_host(ctx, zh.ctypes.data, eh.ctypes.data, 16, K, D, _cabi.DVQ_Z_BF16, 1.0, 0.25,
                                           zq.ctypes.data, ih.ctypes.data, None, None)
        assert rc == -7, rc
    finally:
        _cabi.lib.dvq_host_ctx_destroy(ctx)


# 13 --------------------------------------------------------------------------------------------------------------------
def test_no_hidden_copy_of_z():
    """A bf16 call makes as many library launches as the fp32 call, and at N = 4M, e_dim 64 its peak-memory growth is
    the outputs plus the workspace (an fp32 copy of z would add 1 GiB)."""
    from dvq import _cabi
    N, K, D = 4194304, 512, 64
    E = vo.default_codebook(K, D, 121)
    gen = torch.Generator(device="cuda").manual_seed(122)
    zb = torch.randn(N, D, device="cuda", generator=gen).to(BF)
    counts = {}
    for name, z in (("fp32", zb[:65536].float()), ("bf16", zb[:65536])):
        m = _module(E, AUTO)
        with torch.no_grad():
            m(z, True)                        # workspace + codebook preparation
            c0 = _cabi.launch_count()
            m(z, True)
            counts[name] = _cabi.launch_count() - c0
    assert counts["bf16"] == counts["fp32"], counts
    m = _module(E, AUTO)
    m.cache_codebook = False
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    with torch.no_grad():
        out = m(zb, True)
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    allowed = N * D * 2 + N * 8 + (K + 1) * 8 + _cabi.vq_workspace_bytes(N, K, D, _cabi.DVQ_TRAIN | _cabi.DVQ_Z_BF16) + (64 << 20)
    assert growth <= allowed, (growth, allowed)
    del out

"""GPU parity tests of the VQ path (run on the B200 box: pytest -m gpu).  Every call goes through
the C ABI (dvq.* modules are ctypes front-ends).  Checker = oracle/ + golden vectors of the real
reference.  Bars: indices identical outside the FP64 near-tie band (rel gap < 1e-6), z_q bit-exact
given the index, loss / perplexity within 1e-5 relative."""
import ctypes
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import vq_oracle as vo
from _cases import VQ_CASES, load_gold, rel_err, vq_inputs

pytestmark = pytest.mark.gpu
REL = 1e-5


def _paths():
    from dvq import _cabi
    return [("simt", _cabi.DVQ_PATH_SIMT), ("auto", _cabi.DVQ_PATH_AUTO)]


def _module(E, al, beta, path):
    import dvq
    m = dvq.VectorQuantizer(E.shape[0], E.shape[1], beta, al).cuda()
    with torch.no_grad():
        m.embedding.weight.copy_(torch.from_numpy(E))
    m.path = path
    return m


@pytest.mark.parametrize("pname,path", _paths() if torch.cuda.is_available() else [("simt", 0x10)])
@pytest.mark.parametrize("name", list(VQ_CASES))
def test_forward_matches_reference_golden(name, pname, path):
    z, E, al, beta = vq_inputs(name)
    g = load_gold(name)
    m = _module(E, al, beta, path)
    zt = torch.from_numpy(z).cuda()
    with torch.no_grad():
        loss, zq, ppl, enc, idx = m(zt, True)
        idx_i, zq_i = m(zt, False)
    assert idx.shape == g["idx_train"].shape and idx.dtype == torch.int64
    assert zq.shape == zt.shape and zq_i.shape == zt.shape and loss.dim() == 0 and ppl.dim() == 0
    idx_n, idxi_n = idx.cpu().numpy(), idx_i.cpu().numpy()
    n_mis, n_bad, worst = vo.allowed_index_mismatch(z, E, idx_n, g["idx_train"])
    assert n_bad == 0, (n_mis, worst)
    assert vo.allowed_index_mismatch(z, E, idxi_n, g["idx_infer"])[1] == 0
    assert np.array_equal(idx_n, idxi_n)
    # z_q bit-exact given OUR index (oracle arithmetic), and bit-equal to the reference where indices agree
    assert np.array_equal(zq_i.cpu().numpy().view(np.uint32), vo.zq_infer_from_idx(E, idx_n).reshape(z.shape).view(np.uint32))
    assert np.array_equal(zq.cpu().numpy().view(np.uint32), vo.zq_train_from_idx(z, E, idx_n).reshape(z.shape).view(np.uint32))
    same = idx_n.reshape(-1) == g["idx_train"].reshape(-1)
    assert np.array_equal(zq.cpu().numpy().reshape(-1, E.shape[1])[same].view(np.uint32),
                          g["zq_train"].reshape(-1, E.shape[1])[same].view(np.uint32))
    assert rel_err(loss.item(), g["loss"]) < REL
    if n_mis == 0:
        assert rel_err(ppl.item(), g["perplexity"]) < REL
    hist = np.bincount(idx_n.reshape(-1), minlength=E.shape[0])
    assert rel_err(ppl.item(), vo.perplexity_from_hist(hist, idx_n.shape[0])) < REL
    # min_encodings: fp32 one-hot [N,K] (quantizer.py:40-42)
    assert enc.dtype == torch.float32 and tuple(enc.shape) == (idx_n.shape[0], E.shape[0])
    assert np.array_equal(enc.cpu().numpy(), vo.one_hot(idx_n, E.shape[0]))
    stats = m.last_stats.cpu().numpy()
    assert np.array_equal(stats[:E.shape[0]], hist)


def test_exact_ties_pick_lowest_index():
    z, E, al, beta = vq_inputs("vq_dupes")
    for _, path in _paths():
        m = _module(E, al, beta, path)
        idx, _ = m(torch.from_numpy(z).cuda(), False)
        assert int(idx.max()) < E.shape[0] // 2


@pytest.mark.parametrize("pname,path", _paths() if torch.cuda.is_available() else [("simt", 0x10)])
def test_config1_full_size(pname, path):
    """BASELINE config 1 (N=65536, D=64, K=512), BASELINE.md recipe, all rows against the real
    reference's indices; known answers loss 1.248528003692627 / perplexity 455.29669189453125."""
    g = load_gold("vq_config1_full")
    torch.manual_seed(0)
    emb = torch.nn.Embedding(512, 64)
    emb.weight.data.uniform_(-1.0 / 512, 1.0 / 512)
    z = torch.randn(65536, 64)
    if hashlib.sha256(z.numpy().tobytes()).hexdigest() != str(g["z_sha256"]):
        pytest.skip("torch CPU RNG stream differs from the build container")
    E = emb.weight.detach().numpy()
    m = _module(E, 1, 0.25, path)
    m.onehot_limit_bytes = 0
    with torch.no_grad():
        loss, zq, ppl, enc, idx = m(z.cuda(), True)
    n_mis, n_bad, worst = vo.allowed_index_mismatch(z.numpy(), E, idx.cpu().numpy(), g["idx"].astype(np.int64))
    assert n_bad == 0 and n_mis < 200, (n_mis, worst)
    assert rel_err(loss.item(), 1.248528003692627) < REL
    assert rel_err(ppl.item(), 455.29669189453125) < REL
    assert type(enc).__name__ == "LazyOneHot" and tuple(enc.shape) == (65536, 512)
    assert torch.equal(enc.materialize().argmax(1, keepdim=True), idx)
    same = (idx.cpu().numpy().reshape(-1) == g["idx"].astype(np.int64))
    ref_zq = vo.zq_train_from_idx(z.numpy(), E, g["idx"].astype(np.int64))
    assert np.array_equal(zq.cpu().numpy()[same].view(np.uint32), ref_zq[same].view(np.uint32))


@pytest.mark.parametrize("pname,path", _paths() if torch.cuda.is_available() else [("simt", 0x10)])
@pytest.mark.parametrize("variant", ["default", "variant_b"])
def test_config2_full_size_properties(variant, pname, path):
    """BASELINE config 2 (N=4M, D=64, K=512): size-independent properties on all rows + an
    oracle check (band rule) on a 65 536-row seeded subsample."""
    N, K, D = 4194304, 512, 64
    gen = torch.Generator(device="cuda").manual_seed(2000)
    if variant == "default":
        E = (torch.rand(K, D, device="cuda", generator=gen) * 2 - 1) / K
        z = torch.randn(N, D, device="cuda", generator=gen)
    else:
        E = torch.randn(K, D, device="cuda", generator=gen)
        z = E[torch.randint(0, K, (N,), device="cuda", generator=gen)] + 0.1 * torch.randn(N, D, device="cuda", generator=gen)
    m = _module(E.cpu().numpy(), 1.0, 0.25, path)
    with torch.no_grad():
        loss, zq, ppl, enc, idx = m(z, True)
        idx_i, zq_i = m(z, False)
    assert type(enc).__name__ == "LazyOneHot"
    flat = idx.view(-1)
    assert int(flat.min()) >= 0 and int(flat.max()) < K and torch.equal(idx, idx_i)
    e = E[flat]
    assert torch.equal(zq_i, e)                                        # gather bit-exact
    assert torch.equal(zq, z + (e - z))                                # two roundings, no FMA
    hist = torch.bincount(flat, minlength=K)
    assert int(hist.sum()) == N
    assert torch.equal(m.last_stats[:K], hist)                         # checksum of checksums
    mse = ((e - z).double() ** 2).mean().item()
    assert rel_err(loss.item(), np.float32(np.float32(1.0) * np.float32(mse) + np.float32(0.25) * np.float32(mse))) < REL
    p = hist.double() / N
    assert rel_err(ppl.item(), torch.exp(-(p * torch.log(p + 1e-10)).sum()).item()) < REL
    # every row against the all-FP32 kernel of the same library (band rule on the rows that differ)
    from dvq import _cabi
    if path != _cabi.DVQ_PATH_SIMT:
        ms = _module(E.cpu().numpy(), 1.0, 0.25, _cabi.DVQ_PATH_SIMT)
        with torch.no_grad():
            idx_s, zq_s = ms(z, False)
        _assert_rows_within_band(z, E, flat, idx_s.view(-1))
        same = flat == idx_s.view(-1)
        assert torch.equal(zq_i[same], zq_s[same])
        del idx_s, zq_s
    # idempotence: quantising z_q returns the same codes with zero error
    idx2, zq2 = m(zq_i, False)
    d_self = vo.allowed_index_mismatch(zq_i[:65536].cpu().numpy(), E.cpu().numpy(), idx2[:65536].cpu().numpy(), idx[:65536].cpu().numpy())
    assert d_self[1] == 0
    # oracle on a seeded subsample spread over the whole tensor
    rows = torch.from_numpy(np.random.RandomState(7).choice(N, 65536, replace=False)).cuda()
    zs = z[rows].cpu().numpy()
    ridx, _ = vo.forward_infer(zs, E.cpu().numpy())
    n_mis, n_bad, worst = vo.allowed_index_mismatch(zs, E.cpu().numpy(), flat[rows].cpu().numpy(), ridx)
    assert n_bad == 0, (n_mis, worst)


def _assert_rows_within_band(z, E, idx_a, idx_b, max_rows=200000):
    """All rows compared on the GPU; the (few) rows whose indices differ are copied to the host and must satisfy
    the FP64 near-tie rule (oracle.allowed_index_mismatch)."""
    rows = (idx_a != idx_b).nonzero().view(-1)
    assert rows.numel() <= max_rows, rows.numel()
    if rows.numel() == 0:
        return 0
    zs = z[rows].cpu().numpy()
    n_mis, n_bad, worst = vo.allowed_index_mismatch(zs, E.cpu().numpy(), idx_a[rows].cpu().numpy(), idx_b[rows].cpu().numpy())
    assert n_bad == 0, (n_mis, worst)
    return n_mis


@pytest.mark.parametrize("N,K,D", [(16777216, 16384, 64), (4194304, 4096, 256), (2097152 + 128, 2048, 512)])
def test_config4_corners_full_size_all_rows(N, K, D):
    """Corners of BASELINE config 4 at full per-GPU size (16.8M rows on one GPU on the single-CTA streamed kernel; the
    4-GPU shard of an e_dim 256 shape and the 8-GPU shard (+ one tile: an odd tile count) of an e_dim 512 shape, both on
    the CTA-pair kernel): every row of the tcgen05 path against the all-FP32 kernel (band rule on differing rows),
    z_q / histogram / loss consistency on all rows."""
    from dvq import _cabi
    gen = torch.Generator(device="cuda").manual_seed(4000 + K + D)
    E = (torch.rand(K, D, device="cuda", generator=gen) * 2 - 1) / K
    z = torch.randn(N, D, device="cuda", generator=gen)
    mt = _module(E.cpu().numpy(), 1.0, 0.25, _cabi.DVQ_PATH_TC)
    mt.onehot_limit_bytes = 0
    with torch.no_grad():
        loss, zq, ppl, _, idx = mt(z, True)
    assert mt.last_counters(N)[1] == 0
    flat = idx.view(-1)
    hist = torch.bincount(flat, minlength=K)
    assert int(hist.sum()) == N and torch.equal(mt.last_stats[:K], hist)
    CH = 1 << 21
    sse = 0.0
    for s0 in range(0, N, CH):                                   # chunked: no second N x D temporary
        e = E[flat[s0:s0 + CH]]
        zc = z[s0:s0 + CH]
        assert torch.equal(zq[s0:s0 + CH], zc + (e - zc))
        sse += float(((e - zc).double() ** 2).sum())
    mse = sse / (N * D)
    assert rel_err(loss.item(), np.float32(np.float32(mse) + np.float32(0.25) * np.float32(mse))) < REL
    del zq
    ms = _module(E.cpu().numpy(), 1.0, 0.25, _cabi.DVQ_PATH_SIMT)
    with torch.no_grad():
        idx_s, zq_s = ms(z, False)
    del zq_s
    _assert_rows_within_band(z, E, flat, idx_s.view(-1), max_rows=N // 50)


@pytest.mark.parametrize("name", ["vq_ragged", "vq_3d_view", "vq_k512_d64"])
@pytest.mark.parametrize("pname,path", _paths() if torch.cuda.is_available() else [("simt", 0x10)])
def test_backward_matches_reference_autograd(name, pname, path):
    """Gradients through dvq.VectorQuantizer == gradients of the REAL reference's autograd graph
    (tests/golden/vq_grads_*.npz, made by oracle/gen_golden_grads.py from network/vqvae/quantizer.py:36-60)."""
    import hashlib
    z, E, al, beta = vq_inputs(name)
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vq_grads_%s.npz" % name))
    seed = int(hashlib.sha256(("grad" + name).encode()).hexdigest()[:6], 16)
    w = torch.from_numpy(np.random.RandomState(seed).standard_normal(z.shape).astype(np.float32)).cuda()
    m = _module(E, al, beta, path)
    zt = torch.from_numpy(z).cuda().requires_grad_(True)
    loss, zq, ppl, enc, idx = m(zt, True)
    obj = 3.0 * loss + (zq * zq).sum() + 0.5 * (zq * w).sum()
    obj.backward()
    assert rel_err(obj.item(), g["obj"]) < 1e-5
    same = (idx.cpu().numpy().reshape(-1) == g["idx"].reshape(-1))
    dz = zt.grad.cpu().numpy().reshape(-1, E.shape[1])
    assert np.allclose(dz[same], g["dz"].reshape(-1, E.shape[1])[same], rtol=1e-5, atol=1e-7)
    if same.all():
        assert np.allclose(m.embedding.weight.grad.cpu().numpy(), g["dE"], rtol=1e-5, atol=1e-8)


def test_get_emb_and_wrapper_api():
    import dvq
    z, E, al, beta = vq_inputs("vq_k128_d256")
    g = load_gold("vq_get_emb")
    w = dvq.VQVAE(128, 32, 2, 128, 256, 0.25, a=1).cuda()
    with torch.no_grad():
        w.vector_quantization.embedding.weight.copy_(torch.from_numpy(E))
    for p, ref in zip(g["picks"], g["embs"]):
        out = w.get_embbeding(torch.tensor([int(p)], device="cuda"), 256)      # gen_net.py:101-106 call shape
        assert tuple(out.shape) == (1, 256)
        assert np.array_equal(out.cpu().numpy()[0].view(np.uint32), ref.view(np.uint32))
    batch = w.get_embbeding(torch.from_numpy(g["picks"]).cuda(), 256)          # batched meaning
    assert np.array_equal(batch.cpu().numpy().view(np.uint32), g["embs"].view(np.uint32))
    with torch.no_grad():
        l3 = w(torch.from_numpy(z).cuda())
        i2 = w.inference(torch.from_numpy(z).cuda())
    assert len(l3) == 3 and len(i2) == 2
    assert rel_err(l3[0].item(), g["wrapper_loss"]) < REL and rel_err(l3[2].item(), g["wrapper_ppl"]) < REL
    assert vo.allowed_index_mismatch(z, E, i2[0].cpu().numpy(), g["wrapper_idx"])[1] == 0


def test_backward_matches_reference_formulas():
    """Autograd through the fused forward == autograd through the reference's torch ops."""
    z, E, al, beta = vq_inputs("vq_ragged")
    m = _module(E, al, beta, 0x10)
    zt = torch.from_numpy(z).cuda().requires_grad_(True)
    loss, zq, ppl, enc, idx = m(zt, True)
    (loss * 3.0 + (zq * zq).sum()).backward()
    zr = torch.from_numpy(z).cuda().requires_grad_(True)
    W = torch.from_numpy(E).cuda().requires_grad_(True)
    e = W[idx.view(-1)]
    l_ref = al * torch.mean((e.detach() - zr) ** 2) + beta * torch.mean((e - zr.detach()) ** 2)
    zq_ref = zr + (e - zr).detach()
    (l_ref * 3.0 + (zq_ref * zq_ref).sum()).backward()
    assert torch.allclose(zt.grad, zr.grad, rtol=1e-5, atol=1e-7)
    assert torch.allclose(m.embedding.weight.grad, W.grad, rtol=1e-5, atol=1e-7)


def test_input_validation_and_abi_errors():
    import dvq
    from dvq import _cabi
    m = dvq.VectorQuantizer(16, 8, 0.25, 1).cuda()
    with pytest.raises(TypeError):
        m(torch.randn(4, 8, device="cuda").half(), True)
    with pytest.raises(RuntimeError, match="invalid for input of size"):
        m(torch.randn(3, 7, device="cuda"), True)
    # non-contiguous z (e.g. a slice h[:, :8] of a wider activation, which the reference's .view accepts): copied once
    wide = torch.randn(6, 24, device="cuda")
    i_s, q_s = m(wide[:, :8], False)
    i_c, q_c = m(wide[:, :8].contiguous(), False)
    assert torch.equal(i_s, i_c) and torch.equal(q_s, q_c)
    # an odd storage offset (4-byte aligned only): AUTO takes the FP32 kernel instead of failing the tcgen05 alignment check
    m64 = dvq.VectorQuantizer(64, 64, 0.25, 1).cuda()
    buf = torch.randn(300 * 64 + 1, device="cuda")
    i_o, q_o = m64(buf[1:].view(300, 64), False)
    i_a, q_a = m64(buf[1:].view(300, 64).clone(), False)
    assert torch.equal(i_o, i_a) and torch.equal(q_o, q_a)
    l, q, p, e, i = m(torch.empty(0, 8, device="cuda"), True)
    assert tuple(q.shape) == (0, 8) and tuple(i.shape) == (0, 1)
    i0, q0 = m(torch.empty(0, 8, device="cuda"), False)
    assert tuple(i0.shape) == (0, 1)
    z = torch.randn(32, 8, device="cuda")
    zq = torch.empty_like(z)
    idx = torch.empty(32, dtype=torch.int64, device="cuda")
    ws = torch.empty(256, dtype=torch.uint8, device="cuda")
    rc = _cabi.lib.dvq_vq_forward(z.data_ptr(), m.embedding.weight.data_ptr(), 32, 16, 8, 0, zq.data_ptr(), idx.data_ptr(),
                                  None, None, None, ws.data_ptr(), 16, None)
    assert rc == -4 and "workspace too small" in _cabi.last_error()
    rc = _cabi.lib.dvq_vq_forward(z.data_ptr(), m.embedding.weight.data_ptr(), 32, 16, 8, _cabi.DVQ_TRAIN, zq.data_ptr(),
                                  idx.data_ptr(), None, None, None, ws.data_ptr(), 256, None)
    assert rc == -7
    sm, major, minor = _cabi.device_info()
    assert major == 10 and sm > 100


@pytest.mark.parametrize("train", [False, True])
def test_host_buffer_entry_equals_device_entry(train):
    """dvq_vq_forward_host (chunked, 3-stream pipeline, ragged last chunk) == dvq_vq_forward."""
    import dvq
    N, K, D = 100000 + 37, 512, 64
    rs = np.random.RandomState(5)
    E = vo.default_codebook(K, D, 5)
    z = rs.standard_normal((N, D)).astype(np.float32)
    hq = dvq.HostQuantizer(chunk_rows=16384, n_e_max=K, e_dim_max=D)
    zt = torch.from_numpy(z).pin_memory()
    Et = torch.from_numpy(E).pin_memory()
    m = _module(E, 1.0, 0.25, 0)
    with torch.no_grad():
        if train:
            loss_h, zq_h, ppl_h, idx_h = hq.forward(zt, Et, True, 1.0, 0.25)
            loss, zq, ppl, _, idx = m(zt.cuda(), True)
            assert rel_err(loss_h, loss.item()) < 1e-6 and rel_err(ppl_h, ppl.item()) < 1e-6
        else:
            idx_h, zq_h = hq.forward(zt, Et, False)
            idx, zq = m(zt.cuda(), False)
    assert torch.equal(idx_h, idx.cpu()) and torch.equal(zq_h, zq.cpu())
    hq.close()


# every (K, e_dim) pair of BASELINE config 4 — the streamed kernel picks a shared-memory plan per shape
# (smem_layout in vq_tc_sm100.cu), so each pair is its own code path — plus ragged / real-model shapes
CONFIG4_SHAPES = [(K, D) for K in (512, 1024, 2048, 4096, 8192, 16384) for D in (64, 128, 256, 512)]
EXTRA_SHAPES = [(800, 64), (1536, 32), (128, 256), (992, 128), (960, 256), (32, 16), (256, 32)]


@pytest.mark.parametrize("K,D", CONFIG4_SHAPES + EXTRA_SHAPES)
@pytest.mark.parametrize("variant", ["default", "variant_b"])
def test_streamed_codebook_tc_path(K, D, variant):
    """Codebooks larger than the shared-memory-resident limit are streamed block by block through the
    tcgen05 kernel, e_dim > 64 is contracted in 64-column slices (BASELINE config 4 shapes and the real
    model's K = 128, D = 256 codebooks), K > 992 records candidates as sub-chunk lists: parity against the
    all-FP32 kernel and the oracle (band rule), ragged N."""
    from dvq import _cabi
    N = (20000 if K * D <= 2048 * 512 else 6000) + 37        # (bounds the CPU oracle's N x K x e_dim product)
    if variant == "default":
        E = vo.default_codebook(K, D, 31)
        z = vo.normal_latents(N, D, 32)
    else:
        z, E = vo.variant_b(N, K, D, 33)
    out = {}
    for name, path in (("simt", _cabi.DVQ_PATH_SIMT), ("tc", _cabi.DVQ_PATH_TC)):
        m = _module(E, 1.0, 0.25, path)
        m.onehot_limit_bytes = 0
        with torch.no_grad():
            out[name] = m(torch.from_numpy(z).cuda(), True) + (m.last_stats.clone(),)
        assert m.last_counters(N)[1] == 0                       # no pipeline protocol error
    (ls, qs, ps, _, is_, ss), (lt, qt, pt, _, it, st) = out["simt"], out["tc"]
    idx_t, idx_s = it.cpu().numpy(), is_.cpu().numpy()
    n_mis, n_bad, worst = vo.allowed_index_mismatch(z, E, idx_t, idx_s)
    assert n_bad == 0, (n_mis, worst)
    ridx, _ = vo.forward_infer(z, E)
    assert vo.allowed_index_mismatch(z, E, idx_t, ridx)[1] == 0
    assert np.array_equal(qt.cpu().numpy().view(np.uint32), vo.zq_train_from_idx(z, E, idx_t).view(np.uint32))
    hist = np.bincount(idx_t.reshape(-1), minlength=K)
    assert np.array_equal(st[:K].cpu().numpy(), hist)
    assert rel_err(lt.item(), ls.item()) < REL
    if n_mis == 0:
        assert rel_err(pt.item(), ps.item()) < REL


@pytest.mark.parametrize("K,D", [(512, 64), (2048, 64), (2048, 128)])
def test_degenerate_rows_and_duplicate_codes_take_the_exact_path(K, D):
    """Zero rows, huge rows and a codebook whose second half duplicates the first (every row has an exact
    tie, K/2 .. many candidates) must come out exactly as the all-FP32 kernel gives them: the filter routes
    them to the refine lists (mask mode at K = 512, sub-chunk lists + the overflow list above K = 992)."""
    from dvq import _cabi
    N = 3000 + 11
    rng = np.random.default_rng(5)
    half = (rng.standard_normal((K // 2, D)) * 0.05).astype(np.float32)
    E = np.concatenate([half, half], axis=0)
    z = rng.standard_normal((N, D)).astype(np.float32)
    z[::97] = 0.0                      # zero rows
    z[5::101] *= 1e18                  # outside the FP16 fold range
    z[7::103] = half[rng.integers(0, K // 2, size=len(z[7::103]))]   # exactly on a (duplicated) code
    out = {}
    for name, path in (("simt", _cabi.DVQ_PATH_SIMT), ("tc", _cabi.DVQ_PATH_TC)):
        m = _module(E, 1.0, 0.25, path)
        m.onehot_limit_bytes = 0
        with torch.no_grad():
            idx, zq = m(torch.from_numpy(z).cuda(), False)
        out[name] = (idx.cpu().numpy().reshape(-1), zq.cpu().numpy())
        assert m.last_counters(N)[1] == 0
    assert int(out["tc"][0].max()) < K // 2          # ties -> lowest index, as torch.argmin
    assert np.array_equal(out["tc"][0], out["simt"][0])
    assert np.array_equal(out["tc"][1].view(np.uint32), out["simt"][1].view(np.uint32))


def _bits_equal_nan(a, b):
    """Bit equality of two uint32 views of fp32 arrays; positions where both are NaN count as equal."""
    nan_a, nan_b = np.isnan(a.view(np.float32)), np.isnan(b.view(np.float32))
    return np.array_equal(nan_a, nan_b) and np.array_equal(a[~nan_a], b[~nan_b])


@pytest.mark.parametrize("K,D", [(512, 64), (2048, 64), (1024, 256), (128, 256)])
def test_refine_variants_give_identical_results(K, D):
    """The exact refine stage of the tcgen05 path has three implementations (one warp per undecided row;
    (row, sub-chunk) pairs bucketed by sub-chunk; code-stationary, for the mask-mode shapes it covers) plus a
    device-side hand-back from the binned kernels to the per-row kernel when the pair list overflows.  All must
    produce the same idx / z_q / histogram bit for bit — they evaluate the same FP32 expression and take the same
    lexicographic (distance, code) minimum — and equal the all-FP32 kernel.  Inputs: default-init codebook (a few %
    undecided rows) plus zero / huge rows (paired with every sub-chunk); and the same rows with some made non-finite
    (+inf, -inf, a single NaN element), whose distances are NaN or inf on every code."""
    from dvq import _cabi
    N = 50000 + 13
    E = vo.default_codebook(K, D, 41)
    z = vo.normal_latents(N, D, 42)
    z[::211] = 0.0
    z[3::307] *= 1e18
    z_nf = z.copy()
    z_nf[11::401] = np.inf
    z_nf[13::409, 3] = np.nan
    z_nf[17::419, :2] = -np.inf
    inputs = {"finite": torch.from_numpy(z).cuda(), "nonfinite": torch.from_numpy(z_nf).cuda()}
    arms = [("simt", _cabi.DVQ_PATH_SIMT, 0, 0), ("per_row", _cabi.DVQ_PATH_TC, 1, 0), ("binned", _cabi.DVQ_PATH_TC, 2, 0),
            ("handback", _cabi.DVQ_PATH_TC, 2, 64)]
    if (K, D) == (512, 64):                                        # the one shape here the code-stationary kernel covers
        arms.append(("stationary", _cabi.DVQ_PATH_TC, 3, 0))
    res = {}
    try:
        for name, path, mode, cap in arms:
            _cabi.check(_cabi.lib.dvq_vq_set_refine(mode, cap), "dvq_vq_set_refine")
            m = _module(E, 1.0, 0.25, path)
            m.onehot_limit_bytes = 0
            for which, zt in inputs.items():
                with torch.no_grad():
                    loss, zq, ppl, _, idx = m(zt, True)
                n_ref, err = m.last_counters(N)
                assert err == 0
                if name != "simt":
                    assert n_ref > 0                               # the refine stage did run
                res[name, which] = (idx.cpu().numpy().reshape(-1), zq.cpu().numpy().view(np.uint32), m.last_stats[:K].cpu().numpy(),
                                    loss.item(), ppl.item())
    finally:
        _cabi.check(_cabi.lib.dvq_vq_set_refine(0, 0), "dvq_vq_set_refine")
    for name in [a[0] for a in arms if a[0] not in ("simt", "per_row")]:
        for which in inputs:
            got, want = res[name, which], res["per_row", which]
            assert np.array_equal(got[0], want[0]), (name, which)
            assert _bits_equal_nan(got[1], want[1]), (name, which)
            assert np.array_equal(got[2], want[2]), (name, which)
            assert rel_err(got[4], want[4]) < 1e-7
        got, want = res[name, "finite"], res["per_row", "finite"]
        assert rel_err(got[3], want[3]) < 1e-7                      # (the SSE of a non-finite row is NaN)
    n_mis, n_bad, worst = vo.allowed_index_mismatch(z, E, res["binned", "finite"][0], res["simt", "finite"][0])
    assert n_bad == 0, (n_mis, worst)


_VARIANT_SNIPPET = r"""
import os, sys
import numpy as np, torch
root = sys.argv[1]
sys.path.insert(0, root); sys.path.insert(0, os.path.join(root, "d-vqvae_b200"))
import dvq
from dvq import _cabi
from oracle import vq_oracle as vo
for K, D in ((4096, 64), (2048, 32), (1024, 128), (2048, 256), (544, 128), (1024, 512)):
    N = 30000 + 19
    E = vo.default_codebook(K, D, 51); z = vo.normal_latents(N, D, 52)
    z[::199] = 0.0
    out = {}
    for name, path in (("simt", _cabi.DVQ_PATH_SIMT), ("tc", _cabi.DVQ_PATH_TC)):
        m = dvq.VectorQuantizer(K, D, 0.25, 1.0).cuda(); m.path = path; m.onehot_limit_bytes = 0
        with torch.no_grad():
            m.embedding.weight.copy_(torch.from_numpy(E))
            loss, zq, ppl, _, idx = m(torch.from_numpy(z).cuda(), True)
        assert m.last_counters(N)[1] == 0
        out[name] = (idx.cpu().numpy().reshape(-1), zq.cpu().numpy().view(np.uint32), loss.item())
    n_mis, n_bad, worst = vo.allowed_index_mismatch(z, E, out["tc"][0], out["simt"][0])
    assert n_bad == 0, (K, D, n_mis, worst)
    same = out["tc"][0] == out["simt"][0]
    assert np.array_equal(out["tc"][1][same], out["simt"][1][same])
    assert abs(out["tc"][2] - out["simt"][2]) <= 1e-5 * abs(out["simt"][2])
print("VARIANT_OK")
"""


@pytest.mark.parametrize("env", [{"DVQ_TC_CE": "1"}, {"DVQ_TC_ST": "1"}, {"DVQ_TC_PAIR": "0"}, {"DVQ_TC_PAIR": "1"},
                                 {"DVQ_TC_PAIR": "1", "DVQ_TC_CE": "1"}, {"DVQ_TC_PAIR": "1", "DVQ_TC_ST": "1"}],
                         ids=["converters_join_filter", "two_subchunk_filter", "single_cta_only", "cta_pair_everywhere",
                              "cta_pair_converters_join", "cta_pair_two_subchunk"])
def test_streamed_kernel_variants_behind_env_switches(env):
    """The streamed-codebook kernel has optional variants selected by environment switches that are read once
    per process (DVQ_TC_CE: the converter warps filter as a fourth warp per TMEM lane quarter; DVQ_TC_ST: epilogue
    warps with 104 registers filter two sub-chunks per step; DVQ_TC_PAIR: 0 = never use the CTA-pair (cta_group::2)
    kernel, 1 = use it for every streamed shape, default = for e_dim >= 128).  Each must agree with the all-FP32
    kernel under the same parity rule as the default variant; a fresh interpreter per variant.  N gives an odd
    number of row tiles, so the pair kernel's last tile pair has an empty second half; K = 544 a ragged last chunk."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _VARIANT_SNIPPET, root], env=dict(os.environ, **env), capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "VARIANT_OK" in r.stdout, (r.stdout[-2000:], r.stderr[-2000:])


@pytest.mark.parametrize("K,D", [(2048, 128), (1024, 512), (4096, 64)], ids=["cta_pair_d128", "cta_pair_d512", "single_cta_streamed"])
def test_streamed_kernels_replay_from_a_cuda_graph(K, D):
    """The streamed kernels — incl. the CTA-pair kernel's cluster launch (cudaLaunchKernelEx) and its per-call tensor maps —
    are ordinary stream work: a captured inference call replays with new inputs and gives the eager results."""
    N = 20000 + 37
    E = vo.default_codebook(K, D, 61)
    m = _module(E, 1.0, 0.25, 0x20)   # tcgen05 path
    m.onehot_limit_bytes = 0
    z_static = torch.from_numpy(vo.normal_latents(N, D, 62)).cuda()
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
        z_new = torch.from_numpy(vo.normal_latents(N, D, seed)).cuda()
        z_static.copy_(z_new)
        graph.replay()
        torch.cuda.synchronize()
        with torch.no_grad():
            idx_e, zq_e = m(z_new, False)
        assert torch.equal(idx_g, idx_e) and torch.equal(zq_g, zq_e), (K, D, seed)
    assert m.last_counters(N)[1] == 0


def test_backward_kernel_sharded_scale_and_ema_hooks():
    """dvq_vq_backward with a row count that is NOT the local N (the row-sharded case: the loss is a mean over the
    global rows), dvq_vq_code_sums, and the EMA / usage-reset hooks against their torch restatements."""
    import dvq
    from dvq import _cabi
    z, E, al, beta = vq_inputs("vq_k512_d64")
    m = _module(E, al, beta, 0)
    zt = torch.from_numpy(z).cuda()
    with torch.no_grad():
        loss, zq, ppl, enc, idx = m(zt, True)
    flat_idx = idx.view(-1)
    e = m.embedding.weight.detach()[flat_idx]
    # --- backward kernel, rows = 3 * N (as if two more equal shards existed)
    gz = torch.empty_like(zt)
    gw = torch.zeros_like(m.embedding.weight)
    g_zq = torch.randn_like(zt)
    gl = torch.tensor([1.7], device="cuda")
    rows = torch.tensor([3.0 * zt.shape[0]], device="cuda")
    _cabi.check(_cabi.lib.dvq_vq_backward(zt.data_ptr(), m.embedding.weight.data_ptr(), idx.data_ptr(), g_zq.data_ptr(), gl.data_ptr(),
                                          rows.data_ptr(), zt.shape[0], 512, 64, al, beta, gz.data_ptr(), gw.data_ptr(), None), "bwd")
    scale = 2.0 * 1.7 / (3.0 * zt.shape[0] * 64)
    assert torch.allclose(gz, g_zq + scale * al * (zt - e), rtol=1e-5, atol=1e-8)
    ref_gw = torch.zeros_like(gw).index_add_(0, flat_idx, scale * beta * (e - zt))
    assert torch.allclose(gw, ref_gw, rtol=1e-4, atol=1e-9)
    # --- code sums + EMA step
    sums = m.code_sums(zt, idx)
    ref_sums = torch.zeros(512, 64, device="cuda").index_add_(0, flat_idx, zt)
    assert torch.allclose(sums, ref_sums, rtol=1e-5, atol=1e-6)
    w0 = m.embedding.weight.detach().clone()
    hist = m.ema_update(zt, idx, decay=0.9, eps=1e-5)
    cs = 0.1 * hist
    ew = 0.9 * w0 + 0.1 * ref_sums
    tot = cs.sum()
    ref_w = ew / (((cs + 1e-5) / (tot + 512 * 1e-5) * tot).unsqueeze(1))
    assert torch.allclose(m.embedding.weight.detach(), ref_w, rtol=1e-5, atol=1e-7)
    # --- usage reset: a codebook with far-away rows that no latent selects
    E2 = E.copy()
    E2[100:110] += 50.0
    m2 = _module(E2, al, beta, 0)
    with torch.no_grad():
        m2(zt, True)
    g = torch.Generator(device="cuda").manual_seed(3)
    n_reset = m2.reset_unused_codes(zt, min_usage=1, generator=g)
    assert n_reset >= 10
    assert float(m2.embedding.weight.detach()[100:110].abs().max()) < 10.0
    with torch.no_grad():
        m2(zt, True)
    assert int((m2.last_stats[100:110] > 0).sum()) == 10            # the re-seeded codes are latents now: each is used


@pytest.mark.gpu
@pytest.mark.parametrize("path", [0x00, 0x10])
def test_codebook_preparation_is_cached_and_invalidated(path):
    """DVQ_CODEBOOK_CACHED: the second call with an unchanged codebook reuses the workspace's code norms / operand image
    (bit-identical outputs); a version bump, a different N or invalidate_codebook_cache() rebuild them."""
    import dvq
    from dvq import _cabi
    rs = np.random.RandomState(11)
    K, D, N = 512, 64, 20000
    E = ((rs.rand(K, D) * 2 - 1) / K).astype(np.float32)
    z = torch.from_numpy(rs.randn(N, D).astype(np.float32)).cuda()
    m = _module(E, 1.0, 0.25, path)
    m.onehot_limit_bytes = 0
    seen = []
    real = _cabi.lib.dvq_vq_forward

    def spy(*a):
        seen.append(int(a[5]) & _cabi.DVQ_CODEBOOK_CACHED)
        return real(*a)

    _cabi.lib.dvq_vq_forward = spy
    try:
        with torch.no_grad():
            a = m(z, True)
            b = m(z, True)                                  # cached
            assert seen == [0, _cabi.DVQ_CODEBOOK_CACHED]
            for x, y in zip(a, b):
                if isinstance(x, torch.Tensor):
                    assert torch.equal(x, y)
            i_inf, _ = m(z, False)                          # inference flags, same codebook and N: still cached
            assert seen[-1] == _cabi.DVQ_CODEBOOK_CACHED and torch.equal(i_inf, a[4])
            m(z[:1000].contiguous(), True)                  # another N -> another workspace layout: rebuilt
            assert seen[-1] == 0
            m.embedding.weight.mul_(-1.0)                   # version bump: rebuilt, and the result follows the new codebook
            c = m(z, True)
            assert seen[-1] == 0
            fresh = _module(-E, 1.0, 0.25, path)
            fresh.onehot_limit_bytes = 0
            d = fresh(z, True)
            assert torch.equal(c[4], d[4]) and torch.equal(c[1], d[1])
            m.embedding.weight.data.mul_(-1.0)              # no version bump: the caller invalidates
            m.invalidate_codebook_cache()
            e = m(z, True)
            assert seen[-1] == 0 and torch.equal(e[4], a[4]) and torch.equal(e[1], a[1])
            m.cache_codebook = False
            m(z, True)
            assert seen[-1] == 0
    finally:
        _cabi.lib.dvq_vq_forward = real
    assert m.last_counters(N)[1] == 0


@pytest.mark.parametrize("K,D", [(512, 128), (1024, 256), (2048, 512)])
def test_sliced_path_row_scale_estimate_is_rigorous(K, D):
    """e_dim > 64: the converter picks the row's FP16 scale from the FIRST slice's norm (estimate = norm x slices) and accumulates
    the true norm while converting.  Rows whose energy is spread unevenly over the slices — the estimate off by 0.1x .. 30x —
    must still get the exact kernel's index: in range they are filtered with an off-nominal scale (every bound uses the true
    norm), out of range they go to the exact kernel."""
    from dvq import _cabi
    N = 4000 + 13
    E = vo.default_codebook(K, D, 41)
    z = vo.normal_latents(N, D, 42)
    w = D // (D // 64 if D <= 256 else D // 32)          # columns of the first slice
    for i, f in enumerate((1e-4, 0.03, 0.1, 0.3, 3.0, 10.0, 30.0)):
        z[i::16, :w] *= f                                 # first slice scaled against the rest
    z[7::16, w:] = 0.0                                    # energy in the first slice only
    z[8::16, :w] = 0.0                                    # none in the first slice
    out = {}
    for name, path in (("simt", _cabi.DVQ_PATH_SIMT), ("tc", _cabi.DVQ_PATH_TC)):
        m = _module(E, 1.0, 0.25, path)
        m.onehot_limit_bytes = 0
        with torch.no_grad():
            out[name] = m(torch.from_numpy(z).cuda(), True)
        assert m.last_counters(N)[1] == 0
    idx_t, idx_s = out["tc"][4].cpu().numpy(), out["simt"][4].cpu().numpy()
    n_mis, n_bad, worst = vo.allowed_index_mismatch(z, E, idx_t, idx_s)
    assert n_bad == 0, (n_mis, worst)
    assert vo.allowed_index_mismatch(z, E, idx_t, vo.forward_infer(z, E)[0])[1] == 0
    assert np.array_equal(out["tc"][1].cpu().numpy().view(np.uint32), vo.zq_train_from_idx(z, E, idx_t).view(np.uint32))
    assert rel_err(out["tc"][0].item(), out["simt"][0].item()) < REL

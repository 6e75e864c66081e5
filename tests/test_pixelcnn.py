"""PixelCNN prior: the row-cached sampler against golden vectors of the real reference
(tests/golden/pixelcnn_small.npz, made by oracle/gen_golden_pixelcnn.py) and against its own full forward.
CPU tests (the sampler is torch code over library GEMMs); the GPU variant checks the same on cuda:0."""
import os

import numpy as np
import pytest
import torch

import dvq
from dvq.pixelcnn import GatedPixelCNN

GOLD = os.path.join(os.path.dirname(__file__), "golden", "pixelcnn_small.npz")


def _load():
    g = np.load(GOLD)
    input_dim, dim, n_layers, n_classes = (int(v) for v in g["cfg"])
    m = GatedPixelCNN(input_dim, dim, n_layers, n_classes).eval()
    sd = {k[3:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("sd.")}
    assert set(sd) == set(m.state_dict())                       # same parameter names and shapes as the reference
    m.load_state_dict(sd)
    return g, m


def test_state_dict_layout_matches_reference_and_full_forward():
    g, m = _load()
    x, label = torch.from_numpy(g["x_full"]), torch.from_numpy(g["label"])
    with torch.no_grad():
        out = m(x, label)
    assert np.allclose(out.numpy(), g["full_logits"], rtol=1e-5, atol=1e-5)


def test_cached_sampler_logits_equal_reference_full_forward_at_every_step():
    g, m = _load()
    x_full, label = torch.from_numpy(g["x_full"]), torch.from_numpy(g["label"])
    x, logits = m.generate(x_full, label, shape=(3, 3), batch_size=x_full.shape[0], forced=x_full, return_logits=True)
    assert torch.equal(x, x_full)
    for n, (i, j) in enumerate((i, j) for i in range(3) for j in range(3)):
        ref = g["logits_%d%d" % (i, j)]
        assert np.allclose(logits[n].numpy(), ref, rtol=1e-5, atol=1e-5), (i, j, np.abs(logits[n].numpy() - ref).max())


def test_sampling_reproduces_reference_generate_under_the_same_seed():
    g, m = _load()
    x_full, label = torch.from_numpy(g["x_full"]), torch.from_numpy(g["label"])
    torch.manual_seed(123)
    x = m.generate(x_full, label, shape=(3, 3), batch_size=x_full.shape[0])
    assert np.array_equal(x.numpy(), g["sample_seed123"])


@pytest.mark.parametrize("cfg", [(32, 16, 6, 10), (64, 24, 15, 128)])
def test_cached_sampler_equals_own_full_forward(cfg):
    torch.manual_seed(11)
    m = GatedPixelCNN(*cfg).eval()
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.copy_(0.05 * torch.randn_like(p))
    B = 7
    x_full = torch.randint(0, cfg[0], (B, 3, 3))
    label = torch.randint(0, cfg[3], (B,))
    _, logits = m.generate(None, label, shape=(3, 3), batch_size=B, forced=x_full, return_logits=True)
    x = torch.zeros_like(x_full)
    n = 0
    with torch.no_grad():
        for i in range(3):
            for j in range(3):
                ref = m(x, label)[:, :, i, j]
                assert torch.allclose(logits[n], ref, rtol=2e-5, atol=2e-5), (i, j)
                x[:, i, j] = x_full[:, i, j]
                n += 1


def test_n_valid_restricts_the_sampled_classes():
    torch.manual_seed(3)
    m = GatedPixelCNN(64, 16, 3, 8).eval()
    x = m.generate(None, torch.zeros(9, dtype=torch.int64), batch_size=9, n_valid=5)
    assert int(x.max()) < 5 and x.shape == (9, 3, 3)


@pytest.mark.gpu
def test_cached_sampler_on_gpu_and_as_grasp_prior():
    g, m = _load()
    m = m.cuda()
    x_full, label = torch.from_numpy(g["x_full"]).cuda(), torch.from_numpy(g["label"]).cuda()
    _, logits = m.generate(x_full, label, shape=(3, 3), batch_size=x_full.shape[0], forced=x_full, return_logits=True)
    for n, (i, j) in enumerate((i, j) for i in range(3) for j in range(3)):
        assert np.allclose(logits[n].cpu().numpy(), g["logits_%d%d" % (i, j)], rtol=1e-4, atol=1e-4)
    # as the prior of the grasp pipeline (gen_net.py:92-100): random-init PixelCNN restricted to the 128 codebook rows
    from dvq.grasp import GraspGenerator, pixelcnn_prior
    torch.manual_seed(0)
    prior_net = GatedPixelCNN(512, 64, 3, 128).cuda().eval()
    gen = GraspGenerator(prior=pixelcnn_prior(prior_net, n_valid=128)).cuda().eval()
    obj = torch.randn(8, 4, 256, device="cuda") * 0.1
    recon, pos = gen.gen(obj)
    assert recon.shape == (8, 55) and pos.shape == (8, 6) and torch.isfinite(recon).all()


def _build_tc_model():
    """The dim-256 model of tests/golden/pixelcnn_tc.npz, rebuilt from the seed (oracle/gen_golden_pixelcnn_tc.py)."""
    import hashlib
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "pixelcnn_tc.npz"))
    input_dim, dim, n_layers, n_classes = (int(v) for v in g["cfg"])
    torch.manual_seed(7)
    m = GatedPixelCNN(input_dim, dim, n_layers, n_classes).eval()
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.copy_(0.1 * torch.randn_like(p))
        m.layers[0].make_causal()                           # the reference's state after its first forward
    h = hashlib.sha256()
    for k, v in sorted(m.state_dict().items()):
        h.update(k.encode())
        h.update(v.detach().cpu().numpy().tobytes())
    return g, m, h.hexdigest() == str(g["sd_sha256"])


def test_tc_golden_model_rebuilds_from_seed_and_fp32_sampler_matches_reference():
    g, m, same = _build_tc_model()
    if not same:
        pytest.skip("torch CPU RNG stream differs from the build container")
    x_full, label = torch.from_numpy(g["x_full"]), torch.from_numpy(g["label"])
    _, logits = m.generate(x_full, label, shape=(3, 3), batch_size=x_full.shape[0], forced=x_full, return_logits=True)
    for n, (i, j) in enumerate((i, j) for i in range(3) for j in range(3)):
        assert np.allclose(logits[n].numpy(), g["logits_%d%d" % (i, j)], rtol=1e-4, atol=1e-4), (i, j)


@pytest.mark.gpu
def test_tc_kernel_sampler_matches_reference_logits():
    """precision = "fp16_tc": every contraction on the repo's tcgen05 GEMM kernel (FP16 operands, FP32 accumulation,
    tanh.approx gates).  Bar: 5e-3 of the logit scale (measured 6.4e-4) against the REAL reference's fp32 logits at every step
    (three gated layers + head; measured error printed), plus batch independence with a batch that is not a multiple of 128."""
    g, m, same = _build_tc_model()
    if not same:
        pytest.skip("torch CPU RNG stream differs from the build container")
    m = m.cuda()
    m.precision = "fp16_tc"
    x_full, label = torch.from_numpy(g["x_full"]).cuda(), torch.from_numpy(g["label"]).cuda()
    _, logits = m.generate(x_full, label, shape=(3, 3), batch_size=x_full.shape[0], forced=x_full, return_logits=True)
    m._tc_sampler.check()
    worst = 0.0
    for n, (i, j) in enumerate((i, j) for i in range(3) for j in range(3)):
        ref = g["logits_%d%d" % (i, j)]
        err = np.abs(logits[n].cpu().numpy() - ref).max() / np.abs(ref).max()
        worst = max(worst, err)
        assert err < 5e-3, (i, j, err)
    print("fp16_tc sampler: worst relative logit error %.2e" % worst)
    # a larger batch (two row tiles, ragged): rows must not depend on their neighbours
    B2 = 200
    gen = torch.Generator(device="cuda").manual_seed(5)
    xb = torch.randint(0, 256, (B2, 3, 3), device="cuda", generator=gen)
    lb = torch.randint(0, 8, (B2,), device="cuda", generator=gen)
    xb[:5], lb[:5] = x_full, label
    _, lg2 = m.generate(xb, lb, shape=(3, 3), batch_size=B2, forced=xb, return_logits=True)
    m._tc_sampler.check()
    for n in range(9):
        assert torch.allclose(lg2[n][:5], logits[n], rtol=0, atol=1e-5), n
    m.precision = "tf32"
    _, lg3 = m.generate(xb, lb, shape=(3, 3), batch_size=B2, forced=xb, return_logits=True)
    for n in range(9):
        assert float((lg2[n] - lg3[n]).abs().max()) < 2e-2 * float(lg3[n].abs().max()), n


@pytest.fixture(scope="module")
def bench_prior():
    """The grasp benchmark's prior, GatedPixelCNN(512, 512, 15, 128) sampled with precision = "fp16_tc" at B = 4096
    (seeded random biases, forced random grid and labels), its float64 copy, and a 256-row subset spread over the batch."""
    import copy
    torch.manual_seed(13)
    m = GatedPixelCNN(512, 512, 15, 128).eval()
    with torch.no_grad():
        for n, p in m.named_parameters():
            if n.endswith("bias"):
                p.copy_(0.05 * torch.randn_like(p))
    m = m.cuda()
    m64 = copy.deepcopy(m).double()
    m.precision = "fp16_tc"
    B = 4096
    gen = torch.Generator(device="cuda").manual_seed(14)
    x = torch.randint(0, 512, (B, 3, 3), device="cuda", generator=gen)
    label = torch.randint(0, 128, (B,), device="cuda", generator=gen)
    _, logits = m.generate(None, label, shape=(3, 3), batch_size=B, forced=x, return_logits=True)
    m._tc_sampler.check()
    rows = torch.randperm(B, device="cuda", generator=gen)[:256].sort().values
    return dict(m=m, m64=m64, x=x, label=label, logits=logits, rows=rows, gen=gen)


def _same_bits(a, b):
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.gpu
def test_tc_sampler_at_bench_shape_is_equivariant_under_batch_permutation(bench_prior):
    """A row's logits do not depend on which tile or CTA computed them: permuting the batch permutes all 9 steps' logits
    bit for bit (every row of the multi-tile launches: 384-tile vertical stacks, 256-tile head)."""
    p = bench_prior
    perm = torch.randperm(p["x"].shape[0], device="cuda", generator=p["gen"])
    _, lp = p["m"].generate(None, p["label"][perm], shape=(3, 3), batch_size=len(perm), forced=p["x"][perm], return_logits=True)
    p["m"]._tc_sampler.check()
    for n in range(9):
        assert _same_bits(lp[n], p["logits"][n][perm]), n


@pytest.mark.gpu
def test_tc_sampler_at_bench_shape_does_not_depend_on_batch_size(bench_prior):
    """256 rows spread over the batch, sampled alone (B = 256: 2 row tiles per grid column), equal their rows of the
    B = 4096 run bit for bit."""
    p = bench_prior
    r = p["rows"]
    _, ls = p["m"].generate(None, p["label"][r], shape=(3, 3), batch_size=len(r), forced=p["x"][r], return_logits=True)
    p["m"]._tc_sampler.check()
    for n in range(9):
        assert _same_bits(ls[n], p["logits"][n][r]), n


@pytest.mark.gpu
def test_tc_sampler_at_bench_shape_matches_float64_forward(bench_prior):
    """The fp16_tc logits of 256 rows of the B = 4096 run against the float64 reference forward of the grid as the
    sampler sees it at step (i, j) (later positions 0), over 15 gated layers and the head.
    Bar: 3e-3 of the logit scale, about 4x the error measured on a B200 (7.2e-4; worst step printed)."""
    p = bench_prior
    r = p["rows"]
    x, label = p["x"][r], p["label"][r]
    grids = []
    for i in range(3):
        for j in range(3):
            g = torch.zeros_like(x)
            g.view(len(r), 9)[:, :3 * i + j] = x.view(len(r), 9)[:, :3 * i + j]
            grids.append(g)
    with torch.no_grad():
        full = p["m64"](torch.cat(grids), label.repeat(9))
    worst = 0.0
    for n in range(9):
        i, j = divmod(n, 3)
        ref = full[n * len(r):(n + 1) * len(r), :, i, j]
        err = float((p["logits"][n][r].double() - ref).abs().max() / ref.abs().max())
        worst = max(worst, err)
    print("fp16_tc sampler, GatedPixelCNN(512, 512, 15): worst relative logit error %.2e vs float64" % worst)
    assert worst < 3e-3, worst

"""GPU: which exact refine kernels the automatic refine plan launches for a shape (launch_vq_refine_stage, csrc/vq_refine.cu).

Every refine kernel gives the same bits, so no output-based test can tell them apart; this one reads the kernel names of one
train forward on the tcgen05 path from torch.profiler.  The rules: the code-stationary kernel at K >= 128 up to e_dim 64 and
K >= 256 at e_dim 128 where it covers the shape; else the per-row kernel while the FP32 codebook fits its shared memory; else
the binned kernels followed by the per-row kernel for their hand-back list."""
import pytest
import torch

from oracle import vq_oracle as vo

pytestmark = pytest.mark.gpu

TC = 0x20
# substring of the kernel name -> label; "vq_refine_kernel" is not a substring of "vq_refine_stationary_kernel"
KERNELS = {"vq_refine_stationary_kernel": "stationary", "vq_refine_kernel": "per_row", "refine_prep_kernel": "prep",
           "refine_scatter_kernel": "scatter", "refine_pairs_kernel": "pairs", "refine_emit_kernel": "emit"}
STATIONARY = {"stationary"}
PER_ROW = {"per_row"}
BINNED = {"prep", "scatter", "pairs", "emit", "per_row"}
PLAN = [(512, 64, "fp32", STATIONARY), (512, 64, "bf16", STATIONARY), (256, 128, "fp32", STATIONARY),
        (64, 64, "fp32", PER_ROW), (128, 128, "fp32", PER_ROW), (544, 64, "fp32", PER_ROW), (128, 256, "fp32", PER_ROW),
        (1024, 16, "fp32", PER_ROW),
        (2048, 64, "fp32", BINNED), (1024, 256, "fp32", BINNED), (4096, 128, "fp32", BINNED)]


@pytest.mark.parametrize("K,D,dtype,expected", PLAN, ids=["K%d-D%d-%s" % p[:3] for p in PLAN])
def test_automatic_refine_plan(K, D, dtype, expected):
    import dvq
    from dvq import _cabi
    _cabi.check(_cabi.lib.dvq_vq_set_refine(0, 0), "dvq_vq_set_refine")
    m = dvq.VectorQuantizer(K, D, 0.25, 1.0).cuda()
    with torch.no_grad():
        m.embedding.weight.copy_(torch.from_numpy(vo.default_codebook(K, D, 31)))
    m.path = TC
    m.onehot_limit_bytes = 0
    z = torch.from_numpy(vo.normal_latents(50000, D, 32)).cuda()
    if dtype == "bf16":
        z = z.to(torch.bfloat16)
    with torch.no_grad():
        m(z, True)   # module loading and workspace allocation outside the profiled call
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            m(z, True)
            torch.cuda.synchronize()
    assert m.last_counters(50000)[1] == 0
    launched = set()
    for ev in prof.events():
        for sub, label in KERNELS.items():
            if sub in ev.name:
                launched.add(label)
    assert launched == expected, (K, D, dtype, sorted(launched))

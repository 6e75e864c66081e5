"""GPU: the launch sequence of one dvq_vq_forward call (csrc/dvq_api.cu) for each way through it.

The SIMT and tcgen05 paths, a cached and an uncached codebook preparation give the same indices, so no output-based test
can tell them apart; this one reads the ordered kernel names of a call from torch.profiler and the number of library
launches from dvq_launch_count.  The sequences:
- code norms unless DVQ_CODEBOOK_CACHED, then
- the tcgen05 path (a tcgen05 shape, 16-byte aligned z / E / z_q, not DVQ_PATH_SIMT): the codebook preparation (or, when
  cached, only the reset of the per-call counters), the filter, then the refine plan's kernels (code-stationary for
  K = 512 / e_dim 64; binned plus the per-row kernel on their hand-back list for K = 2048);
- otherwise the FP32 kernel;
- the one-hot kernel last under DVQ_WRITE_ONEHOT.
N = 0 launches the code norms only, and a forced DVQ_PATH_TC call on a 4-byte-aligned view fails with DVQ_ERR_BAD_ALIGN.
The profiled calls run in one fresh interpreter: after this module's profiler sessions in the same process, the later
profiler-based tests of the suite (test_vq_refine_plan_gpu, test_vq_tc_plan_gpu) found kernels missing from their traces."""
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from oracle import vq_oracle as vo

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif("DVQ_REFINE_PER_ROW" in os.environ, reason="DVQ_REFINE_PER_ROW overrides the refine plan")]

TRAIN, ONEHOT, CACHED, SIMT, TC, BF16 = 0x1, 0x2, 0x200, 0x10, 0x20, 0x400
N = 50000
NORMS = ["code_norms_kernel"]
PREP = ["tc_cb_stats_kernel", "tc_cb_image_kernel"]
STATIONARY = ["vq_refine_stationary_kernel"]
BINNED = ["refine_prep_kernel", "refine_scatter_kernel", "refine_pairs_kernel", "refine_emit_kernel", "vq_refine_kernel"]
FILTER = ["vq_tc_kernel"]
SIMT_KERNEL = ["vq_simt_kernel"]


class Call:
    """Operands and workspace of dvq_vq_forward calls over n rows; z (and z_q) start `offset` elements into their buffers."""

    def __init__(self, K, D, flags, n=N, offset=0):
        from dvq import _cabi
        self.K, self.D, self.flags, self.n = K, D, flags, n
        dtype = torch.bfloat16 if flags & BF16 else torch.float32
        self.E = torch.from_numpy(vo.default_codebook(K, D, 51)).cuda()
        z = torch.from_numpy(vo.normal_latents(n, D, 52)).cuda().to(dtype).reshape(-1)
        self.z = torch.cat([torch.zeros(offset, dtype=dtype, device="cuda"), z])[offset:]
        self.z_q = torch.empty(n * D + offset, dtype=dtype, device="cuda")[offset:]
        self.idx = torch.empty(n, dtype=torch.int64, device="cuda")
        self.onehot = torch.empty((n, K), dtype=torch.float32, device="cuda") if flags & ONEHOT else None
        self.stats = torch.zeros(K + 1, dtype=torch.int64, device="cuda") if flags & TRAIN else None
        self.ws = torch.empty(max(_cabi.vq_workspace_bytes(n, K, D, flags), 256), dtype=torch.uint8, device="cuda")

    def __call__(self, extra=0):
        from dvq import _cabi
        st = self.stats
        return _cabi.lib.dvq_vq_forward(
            self.z.data_ptr(), self.E.data_ptr(), self.n, self.K, self.D, self.flags | extra, self.z_q.data_ptr(),
            self.idx.data_ptr(), self.onehot.data_ptr() if self.onehot is not None else None,
            st.data_ptr() if st is not None else None, st.data_ptr() + 8 * self.K if st is not None else None,
            self.ws.data_ptr(), self.ws.numel(), torch.cuda.current_stream().cuda_stream)


def profiled(call, extra=0):
    """(ordered library kernel names, library launches) of one call."""
    from dvq import _cabi
    torch.cuda.synchronize()
    before = _cabi.launch_count()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _cabi.check(call(extra), "dvq_vq_forward")
        torch.cuda.synchronize()
    launches = _cabi.launch_count() - before
    kernels = sorted((ev for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda ev: ev.time_range.start)
    names = [m.group(1) for ev in kernels for m in [re.search(r"(\w+_kernel\w*)", ev.name)] if m]
    return names, launches


# (K, D, flags, rows, z offset) -> kernels of an uncached call, kernels of the same call with DVQ_CODEBOOK_CACHED
PLAN = [
    ((512, 64, TRAIN, N, 0), NORMS + PREP + FILTER + STATIONARY, ["tc_reset_kernel"] + FILTER + STATIONARY),   # config 2
    ((512, 64, TRAIN | BF16, N, 0), NORMS + PREP + FILTER + STATIONARY, ["tc_reset_kernel"] + FILTER + STATIONARY),
    ((512, 64, 0, N, 0), NORMS + PREP + FILTER + STATIONARY, ["tc_reset_kernel"] + FILTER + STATIONARY),
    ((2048, 64, TRAIN, N, 0), NORMS + PREP + FILTER + BINNED, ["tc_reset_kernel"] + FILTER + BINNED),
    ((512, 64, TRAIN, N, 1), NORMS + SIMT_KERNEL, SIMT_KERNEL),                 # odd storage offset under DVQ_PATH_AUTO
    ((512, 64, TRAIN | SIMT, N, 0), NORMS + SIMT_KERNEL, SIMT_KERNEL),
    ((512, 24, TRAIN, N, 0), NORMS + SIMT_KERNEL, SIMT_KERNEL),                 # e_dim 24: not a tcgen05 shape
    ((512, 64, TRAIN | ONEHOT, N, 0), NORMS + PREP + FILTER + STATIONARY + ["onehot_kernel_v4"],
     ["tc_reset_kernel"] + FILTER + STATIONARY + ["onehot_kernel_v4"]),
    ((512, 64, TRAIN, 0, 0), NORMS, []),
]


def _id(case):
    K, D, flags, n, offset = case
    kind = "+".join(name for bit, name in ((TRAIN, "train"), (BF16, "bf16"), (SIMT, "simt"), (ONEHOT, "onehot")) if flags & bit)
    return "K%d-D%d-%s-N%d-off%d" % (K, D, kind or "infer", n, offset)


_SNIPPET = """
import json, sys
root = sys.argv[1]
sys.path[:0] = [root, root + "/d-vqvae_b200", root + "/tests"]
from test_vq_forward_plan_gpu import PLAN, sequences
print("SEQUENCES " + json.dumps([sequences(case) for case, _, _ in PLAN]))
"""


def sequences(case):
    """(kernels, launches) of an uncached and of a cached call, after one unprofiled call that loads the modules."""
    from dvq import _cabi
    _cabi.check(_cabi.lib.dvq_vq_set_refine(0, 0), "dvq_vq_set_refine")
    call = Call(*case)
    _cabi.check(call(), "dvq_vq_forward")
    return profiled(call), profiled(call, CACHED)


@pytest.fixture(scope="module")
def recorded():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _SNIPPET, root], capture_output=True, text=True, timeout=600)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("SEQUENCES ")]
    assert r.returncode == 0 and lines, (r.stdout[-2000:], r.stderr[-2000:])
    got = json.loads(lines[-1][len("SEQUENCES "):])
    return {tuple(case): tuple(tuple(seq) for seq in g) for (case, _, _), g in zip(PLAN, got)}


@pytest.mark.parametrize("case,first,cached", PLAN, ids=[_id(c) for c, _, _ in PLAN])
def test_forward_launch_sequence(recorded, case, first, cached):
    assert recorded[case] == ((first, len(first)), (cached, len(cached))), case


def test_forced_tc_path_on_unaligned_view():
    from dvq import _cabi
    call = Call(512, 64, TRAIN | TC, N, 1)
    assert call() == -2     # DVQ_ERR_BAD_ALIGN
    assert _cabi.last_error() == "tcgen05 path needs 16-byte aligned z / E / z_q"

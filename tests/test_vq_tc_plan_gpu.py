"""GPU: which vq_tc_kernel instance the tcgen05 filter's plan launches for a shape (plan_vq_tc, csrc/vq_tc_sm100.cu).

Every filter variant gives the same bits, so no output-based test can tell them apart; this one reads the template
arguments <DT, TRAIN, LIST, CE, ST, PAIR, ZT> of the one vq_tc_kernel launch of a forward from torch.profiler.  The rules:
DT = 64 for the resident mask-mode e_dim 64 shapes; LIST from K > 992; the CTA-pair kernel for streamed codebooks at
e_dim 512 and at e_dim 128 / 256 from K = 2048 on, with at least two row tiles; CE / ST only behind their switches, for
fp32 latents.  The switches are read once per process, so those cases run in fresh interpreters."""
import json
import os
import re
import subprocess
import sys

import pytest
import torch

from oracle import vq_oracle as vo

pytestmark = pytest.mark.gpu

TC = 0x20
N = 50000
SWITCHES = ("DVQ_TC_PAIR", "DVQ_TC_LAYOUT", "DVQ_TC_CE", "DVQ_TC_ST")
_BOOL = {"true": True, "false": False, "(bool)1": True, "(bool)0": False}


def _parse(args):
    dt, *flags, zt = [a.strip() for a in args.split(",")]
    return [int(dt.replace("(int)", ""))] + [_BOOL[f] for f in flags] + ["bf16" if "bfloat16" in zt else zt]


def launched(K, D, dtype, train, n=N):
    """[DT, TRAIN, LIST, CE, ST, PAIR, ZT] of every vq_tc_kernel launch of one forward on the tcgen05 path."""
    import dvq
    m = dvq.VectorQuantizer(K, D, 0.25, 1.0).cuda()
    with torch.no_grad():
        m.embedding.weight.copy_(torch.from_numpy(vo.default_codebook(K, D, 41)))
    m.path = TC
    m.onehot_limit_bytes = 0
    z = torch.from_numpy(vo.normal_latents(n, D, 42)).cuda()
    if dtype == "bf16":
        z = z.to(torch.bfloat16)
    with torch.no_grad():
        m(z, train)   # module loading and workspace allocation outside the profiled call
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            m(z, train)
            torch.cuda.synchronize()
    assert m.last_counters(n)[1] == 0
    return [_parse(mt.group(1)) for ev in prof.events() for mt in [re.search(r"vq_tc_kernel<([^<>]*)>", ev.name)] if mt]


def _k(dt=0, train=True, list_=False, ce=False, st=False, pair=False, zt="float"):
    return [dt, train, list_, ce, st, pair, zt]


# (K, D, dtype, train, rows) -> the one kernel launched
PLAN = [
    ((512, 64, "fp32", True, N), _k(dt=64)),                                    # config 2: resident image
    ((512, 64, "fp32", False, N), _k(dt=64, train=False)),
    ((512, 64, "bf16", True, N), _k(dt=64, zt="bf16")),
    ((512, 64, "bf16", False, N), _k(dt=64, train=False, zt="bf16")),
    ((768, 64, "fp32", True, N), _k()),                                         # streamed, mask mode
    ((2048, 64, "fp32", True, N), _k(list_=True)),                              # streamed, list mode, single CTA
    ((512, 128, "fp32", True, N), _k()),                                        # streamed, single CTA
    ((2048, 128, "fp32", True, N), _k(list_=True, pair=True)),                  # CTA pair
    ((2048, 128, "bf16", False, N), _k(train=False, list_=True, pair=True, zt="bf16")),
    ((1024, 512, "fp32", True, N), _k(list_=True, pair=True)),
    ((16384, 512, "fp32", True, 128), _k(list_=True)),                          # one row tile: nothing to pair
    ((128, 256, "fp32", True, N), _k()),                                        # the grasp codebooks
]


@pytest.mark.skipif(any(k in os.environ for k in SWITCHES), reason="a DVQ_TC_* switch overrides the automatic plan")
@pytest.mark.parametrize("case,expected", PLAN, ids=["K%d-D%d-%s-%s-N%d" % (c[0], c[1], c[2], "train" if c[3] else "infer", c[4]) for c, _ in PLAN])
def test_automatic_filter_plan(case, expected):
    assert launched(*case) == [expected], case


# switch -> [(case, expected)], run in one fresh interpreter per switch
SWITCHED = {
    "DVQ_TC_PAIR=0": [((2048, 128, "fp32", True), _k(list_=True)), ((1024, 512, "fp32", True), _k(list_=True))],
    "DVQ_TC_PAIR=1": [((768, 64, "fp32", True), _k(pair=True)), ((512, 64, "fp32", True), _k(dt=64))],
    "DVQ_TC_CE=1": [((2048, 64, "fp32", True), _k(list_=True, ce=True)), ((2048, 64, "bf16", True), _k(list_=True, zt="bf16")),
                    ((512, 64, "fp32", True), _k(dt=64))],
    "DVQ_TC_ST=1": [((2048, 64, "fp32", True), _k(list_=True, st=True)), ((2048, 64, "bf16", True), _k(list_=True, zt="bf16")),
                    ((512, 64, "fp32", True), _k(dt=64))],
}
_SNIPPET = """
import json, sys
root = sys.argv[1]
sys.path[:0] = [root, root + "/d-vqvae_b200", root + "/tests"]
from test_vq_tc_plan_gpu import launched
print("PLANS " + json.dumps([launched(*case) for case in json.loads(sys.argv[2])]))
"""


@pytest.mark.parametrize("switch", sorted(SWITCHED))
def test_filter_plan_behind_env_switches(switch):
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cases = [c for c, _ in SWITCHED[switch]]
    name, value = switch.split("=")
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES}
    env[name] = value
    r = subprocess.run([sys.executable, "-c", _SNIPPET, root, json.dumps(cases)], env=env, capture_output=True, text=True, timeout=600)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("PLANS ")]
    assert r.returncode == 0 and lines, (r.stdout[-2000:], r.stderr[-2000:])
    got = json.loads(lines[-1][len("PLANS "):])
    assert len(got) == len(cases)
    for (case, expected), kernels in zip(SWITCHED[switch], got):
        assert kernels == [expected], (switch, case, kernels)

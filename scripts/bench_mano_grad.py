"""Forward and forward+backward of the MANO hand layer: dvq.ManoLayer(differentiable=True) against the torch op sequence that
the `mano` / `smplx` layer launches (tests/_mano_torch.py `mano_forward_torch`, float32 on the GPU, tables resident there):

    python scripts/bench_mano_grad.py [--out profiles/r04_bench_mano_grad.json] [--reps 15] [--iters 20]

For B in {64, 1024, 4096} hands (synthetic model of MANO's structure, random parameters) three arms alternate within each
repetition: dvq forward only (no_grad), dvq forward+backward (autograd.grad of vertices and joints), torch forward+backward.
Each arm is warmed up, then timed with CUDA events around --iters steps; the median over --reps repetitions is reported.
The model tables (1.3 MB of pose-blend directions) stay L2-resident across steps, as they do in use.  A separate
torch.profiler pass counts the kernels per step.  At B = 64 the gradients of both float32 arms are compared with float64
autograd of the same restatement on the CPU.  Prints one JSON line and writes it to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "d-vqvae_b200"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import dvq  # noqa: E402
from dvq import _cabi  # noqa: E402
from _mano_torch import mano_forward_torch, torch_model  # noqa: E402
from oracle import mano_oracle as mo  # noqa: E402

BATCHES = (64, 1024, 4096)
ARMS = ("dvq_forward", "dvq_forward_backward", "torch_forward_backward")


def card():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = (x.strip() for x in r.stdout.strip().split(","))
    return name, power, clock


def make_inputs(B, dev, seed):
    rs = np.random.RandomState(seed)
    arrays = (rs.randn(B, 10), 0.8 * rs.randn(B, 3), 0.8 * rs.randn(B, 45), 0.3 * rs.randn(B, 3))
    ts = [torch.from_numpy(a.astype(np.float32)).to(dev).requires_grad_(True) for a in arrays]
    ups = [torch.from_numpy(rs.randn(B, 778, 3).astype(np.float32)).to(dev), torch.from_numpy(rs.randn(B, 16, 3).astype(np.float32)).to(dev)]
    return arrays, ts, ups


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_bench_mano_grad.json"))
    ap.add_argument("--reps", type=int, default=15)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_mano_grad.py measures on the GPU"
    dev = torch.device("cuda:0")
    name, power, clock = card()
    model = mo.synthetic_model(0)
    layer = dvq.ManoLayer(model, differentiable=True).to(dev)
    tables = torch_model(model, torch.float32, dev)

    def run(arm, ts, ups):
        if arm == "dvq_forward":
            with torch.no_grad():
                out = layer(betas=ts[0], global_orient=ts[1], hand_pose=ts[2], transl=ts[3])
            return out.vertices, out.joints
        if arm == "dvq_forward_backward":
            out = layer(betas=ts[0], global_orient=ts[1], hand_pose=ts[2], transl=ts[3])
            return torch.autograd.grad((out.vertices, out.joints), ts, ups)
        v, j = mano_forward_torch(tables, *ts)
        return torch.autograd.grad((v, j), ts, ups)

    res = {"card": name, "power_limit": power, "max_sm_clock": clock, "model": "oracle.mano_oracle.synthetic_model(0), use_pca=True, 45 components, flat_hand_mean",
           "method": "arms alternate within each of %d repetitions; %d warm-up steps per arm and batch, then CUDA events around %d steps; "
                     "median ms per step; kernel counts from a separate torch.profiler pass" % (args.reps, args.warmup, args.iters),
           "batches": {}}
    for B in BATCHES:
        _, ts, ups = make_inputs(B, dev, 100 + B)
        for arm in ARMS:
            for _ in range(args.warmup):
                run(arm, ts, ups)
        torch.cuda.synchronize()
        times = {a: [] for a in ARMS}
        for _ in range(args.reps):
            for arm in ARMS:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.iters):
                    run(arm, ts, ups)
                e1.record()
                e1.synchronize()
                times[arm].append(e0.elapsed_time(e1) / args.iters)
        row = {a: {"ms_median": statistics.median(t), "ms_min": min(t), "ms_max": max(t)} for a, t in times.items()}
        row["backward_ms_estimate"] = row["dvq_forward_backward"]["ms_median"] - row["dvq_forward"]["ms_median"]
        row["speedup_fwd_bwd_vs_torch"] = row["torch_forward_backward"]["ms_median"] / row["dvq_forward_backward"]["ms_median"]
        res["batches"][str(B)] = row
    # kernels per step (separate pass: the profiler slows the host)
    _, ts, ups = make_inputs(64, dev, 7)
    counts = {}
    for arm in ARMS:
        run(arm, ts, ups)
        torch.cuda.synchronize()
        n0 = _cabi.launch_count()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(4):
                run(arm, ts, ups)
            torch.cuda.synchronize()
        kernels = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith(("Memset", "Memcpy"))]
        counts[arm] = {"kernels_per_step": len(kernels) / 4, "dvq_launches_per_step": (_cabi.launch_count() - n0) / 4}
    res["kernels_per_step"] = counts
    # gradient error of both float32 arms against float64 autograd at B = 64
    arrays, ts, ups = make_inputs(64, dev, 11)
    t64 = [torch.from_numpy(a).requires_grad_(True) for a in arrays]
    v, j = mano_forward_torch(model, *t64)
    ref = torch.autograd.grad((v, j), t64, [u.double().cpu() for u in ups])
    errs = {}
    for arm in ("dvq_forward_backward", "torch_forward_backward"):
        got = run(arm, ts, ups)
        errs[arm] = {n: float((g.double().cpu() - r).abs().max() / r.abs().max()) for n, g, r in zip(("betas", "global_orient", "hand_pose", "transl"), got, ref)}
    res["grad_rel_max_err_vs_float64_B64"] = errs
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()

"""A/B of the exact refine stage at BASELINE config 2 (N = 4 194 304 fp32 latents, e_dim 64, K = 512, train path):
the code-stationary kernel (the default for this shape) against the per-row kernel, alternated in one process.

    python scripts/ab_refine.py OUT_DIR [--trials 7] [--steps 50] [--bench-runs 3]

Per trial and arm: 5 warm-up calls, then STEPS timed calls with the library's per-stage CUDA events (stage 1 = main
kernel, stage 2 = refine) and CUDA events around the whole window (step time).  Reports the median and the range of each
over the trials, a few more shapes the stationary kernel covers (3 trials each), then runs `bench.py` BENCH_RUNS times
per arm, alternating (the per-row arm through DVQ_REFINE_PER_ROW=1), and compares the two arms' `--dump-outputs`.
Writes OUT_DIR/ab_refine.json and prints it; the card's name and power limit are part of the record."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "d-vqvae_b200"))

ARMS = (("stationary", 3), ("per_row", 1))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = (x.strip() for x in q.split(","))
        return {"name": name, "power_limit": power, "sm_clock_max": clk}
    except Exception as e:                                  # noqa: BLE001
        return {"error": repr(e)}


def spread(xs):
    return {"median": round(statistics.median(xs), 4), "min": round(min(xs), 4), "max": round(max(xs), 4), "n": len(xs)}


def ab_shape(torch, dvq, _cabi, N, K, D, trials, steps):
    g = torch.Generator(device="cuda").manual_seed(2000)
    vq = dvq.VectorQuantizer(K, D, 0.25, 1.0).cuda()
    vq.onehot_limit_bytes = 0
    with torch.no_grad():
        vq.embedding.weight.copy_((torch.rand(K, D, device="cuda", generator=g) * 2 - 1) / K)
    z = torch.randn(N, D, device="cuda", generator=g)
    res = {name: {"refine_ms": [], "kernel_ms": [], "step_ms": []} for name, _ in ARMS}
    outs = {}
    try:
        for _ in range(trials):
            for name, mode in ARMS:
                _cabi.check(_cabi.lib.dvq_vq_set_refine(mode, 0), "dvq_vq_set_refine")
                with torch.no_grad():
                    for _ in range(5):
                        out = vq(z, True)
                    torch.cuda.synchronize()
                    _cabi.check(_cabi.lib.dvq_profile_enable(1), "dvq_profile_enable")
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(steps):
                        out = vq(z, True)
                    e1.record()
                    torch.cuda.synchronize()
                    ms, _ = _cabi.profile_mean()
                    _cabi.check(_cabi.lib.dvq_profile_enable(0), "dvq_profile_enable")
                res[name]["refine_ms"].append(ms[2])
                res[name]["kernel_ms"].append(ms[1])
                res[name]["step_ms"].append(e0.elapsed_time(e1) / steps)
                outs[name] = (out[4].clone(), out[1].clone(), vq.last_stats[:K].clone(), out[0].item(), out[2].item())
        undecided = vq.last_counters(N)[0]
    finally:
        _cabi.check(_cabi.lib.dvq_vq_set_refine(0, 0), "dvq_vq_set_refine")
    a, b = outs["stationary"], outs["per_row"]
    line = {"N": N, "K": K, "D": D, "undecided_rows": undecided,
            "identical_idx_zq_hist": bool(torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))
                                          and torch.equal(a[2], b[2])),
            "loss": [a[3], b[3]], "perplexity": [a[4], b[4]]}
    for name, _ in ARMS:
        line[name] = {k: spread(v) for k, v in res[name].items()}
    return line


def bench_arms(out_dir, runs):
    lines = {name: [] for name, _ in ARMS}
    dumps = {}
    tmp = tempfile.mkdtemp(prefix="ab_refine_")
    for i in range(runs):
        for name, _ in ARMS:
            env = dict(os.environ)
            env.pop("DVQ_REFINE_PER_ROW", None)
            if name == "per_row":
                env["DVQ_REFINE_PER_ROW"] = "1"
            cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "50", "--warmup", "5",
                   "--no-secondary", "--no-cpu-baseline"]
            if i == 0:
                dumps[name] = os.path.join(tmp, name)
                cmd += ["--dump-outputs", dumps[name]]
            r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
            try:
                j = json.loads(r.stdout.strip().splitlines()[-1])
                lines[name].append({"value": j["value"], "ms_per_step": j["ms_per_step"], "kernel_ms": j["roofline"]["kernel_ms"],
                                    "refine_ms": j["roofline"]["refine_ms"], "sm_mhz": j["clocks"]["sm_mhz"],
                                    "reasons": j["clocks"]["reasons"]})
            except Exception as e:                          # noqa: BLE001
                lines[name].append({"error": repr(e), "stderr": r.stderr[-2000:]})
    import numpy as np
    same = {}
    for f in ("indices", "z_q_rows", "z_q_sample", "usage_histogram", "loss", "perplexity"):
        try:
            x, y = (np.load(os.path.join(dumps[n], f + ".npy")) for n, _ in ARMS)
            same[f] = bool(np.array_equal(x.view(np.uint8), y.view(np.uint8))) if f not in ("loss", "perplexity") else \
                [float(x), float(y)]
        except Exception as e:                              # noqa: BLE001
            same[f] = repr(e)
    summary = {}
    for name, _ in ARMS:
        ok = [l for l in lines[name] if "value" in l]
        if ok:
            summary[name] = {k: spread([l[k] for l in ok]) for k in ("value", "ms_per_step", "kernel_ms", "refine_ms")}
    return {"runs": lines, "summary": summary, "dump_outputs_compared": same,
            "command": "bench.py --gpus 1 --steps 50 --warmup 5 --no-secondary --no-cpu-baseline (per-row arm: DVQ_REFINE_PER_ROW=1)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("out_dir")
    ap.add_argument("--trials", type=int, default=7)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--bench-runs", type=int, default=3)
    args = ap.parse_args()
    import torch
    import dvq
    from dvq import _cabi
    os.makedirs(args.out_dir, exist_ok=True)
    rec = {"card": card(), "torch_device": torch.cuda.get_device_name(0),
           "what": "refine_ms / kernel_ms: library stage events 2 / 1 (mean over STEPS calls per trial); step_ms: CUDA events "
                   "around the STEPS calls; median, min, max over the trials; arms alternate within each trial"}
    rec["config2"] = ab_shape(torch, dvq, _cabi, 4194304, 512, 64, args.trials, args.steps)
    print(json.dumps(rec["config2"]), flush=True)
    rec["other_shapes"] = []
    for K, D in ((32, 64), (64, 64), (128, 64), (256, 64), (128, 32), (512, 32), (128, 16), (992, 16), (128, 128), (256, 128)):
        rec["other_shapes"].append(ab_shape(torch, dvq, _cabi, 4194304, K, D, 3, 20))
        print(json.dumps(rec["other_shapes"][-1]), flush=True)
    if args.bench_runs > 0:
        rec["bench"] = bench_arms(args.out_dir, args.bench_runs)
    with open(os.path.join(args.out_dir, "ab_refine.json"), "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()

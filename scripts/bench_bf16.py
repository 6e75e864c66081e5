"""fp32 vs bf16 latents (DVQ_Z_BF16) through dvq.VectorQuantizer, train path, on the HBM-bound shapes:

    python scripts/bench_bf16.py [--out profiles/r03_bench_bf16.json] [--reps 5]

config 2 (N = 4M, e_dim 64, K = 512), K = 512 at e_dim 128 / 256 / 512 (N = 16.8M) and the config-4 corners K = 16 384 at
e_dim 128 / 512 (N = 4M).  Per shape the bf16 call and the fp32 call on the same (upcast) latents alternate: warm-up, then
CUDA-event times per call; inputs are larger than the 126 MB L2.  A separate pass with dvq_profile_enable gives the
main-kernel and refine stage times.  Prints one JSON line and writes it to --out."""
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

import torch  # noqa: E402

import dvq  # noqa: E402
from dvq import _cabi  # noqa: E402
from bench import measured_peaks  # noqa: E402

SHAPES = [("config2", 4194304, 512, 64), ("k512_d128", 16777216, 512, 128), ("k512_d256", 16777216, 512, 256),
          ("k512_d512", 16777216, 512, 512), ("k16384_d128", 4194304, 16384, 128), ("k16384_d512", 4194304, 16384, 512)]


def card():
    r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, _, power = r.stdout.strip().partition(",")
    return name.strip(), power.strip()


def algorithmic_bytes(N, K, D, zbytes):
    # z read once, z_q written once, idx (8 B) per row, the fp32 codebook once
    return N * (2 * zbytes * D + 8) + 4 * K * D


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_bench_bf16.json"))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_bf16.py measures on the GPU"
    dev = torch.device("cuda:0")
    hbm_gbs, _, peaks_src, bf16_tf = measured_peaks()
    name, power = card()
    res = {"card": name, "power_limit": power, "peaks": {"hbm_gbs": hbm_gbs, "bf16_tflops_sustained": bf16_tf, "source": peaks_src},
           "method": "train path, AUTO; fp32 and bf16 calls alternate after %d warm-up calls each; CUDA events around each call; "
                     "stage times from dvq_profile_enable in a separate pass" % args.warmup, "shapes": {}}
    for sname, N, K, D in SHAPES:
        g = torch.Generator(device=dev).manual_seed(9000 + K + D)
        E = (torch.rand(K, D, device=dev, generator=g) * 2 - 1) / K
        zb = torch.randn(N, D, device=dev, generator=g).to(torch.bfloat16)
        z32 = zb.float()            # the same latents: both calls must give the same indices
        mods = {}
        for kind in ("fp32", "bf16"):
            m = dvq.VectorQuantizer(K, D, 0.25, 1.0).to(dev)
            m.onehot_limit_bytes = 0
            with torch.no_grad():
                m.embedding.weight.copy_(E)
            mods[kind] = m
        inp = {"fp32": z32, "bf16": zb}
        out = {}
        with torch.no_grad():
            for kind in ("fp32", "bf16"):
                for _ in range(args.warmup):
                    out[kind] = mods[kind](inp[kind], True)
            times = {"fp32": [], "bf16": []}
            for _ in range(args.reps):
                for kind in ("fp32", "bf16"):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    out[kind] = mods[kind](inp[kind], True)
                    e1.record()
                    torch.cuda.synchronize()
                    times[kind].append(e0.elapsed_time(e1))
            undecided = {k: mods[k].last_counters(N)[0] for k in mods}
            idx_equal = bool(torch.equal(out["fp32"][4], out["bf16"][4]))
            zq_equal = bool(torch.equal(out["bf16"][1].view(torch.int16), out["fp32"][1].to(torch.bfloat16).view(torch.int16)))
            loss = {k: float(out[k][0]) for k in out}
            stages = {}
            for kind in ("fp32", "bf16"):
                _cabi.check(_cabi.lib.dvq_profile_enable(1), "dvq_profile_enable")
                for _ in range(3):
                    mods[kind](inp[kind], True)
                ms, cnt = _cabi.profile_mean()
                _cabi.check(_cabi.lib.dvq_profile_enable(0), "dvq_profile_enable")
                stages[kind] = {"main_kernel_ms": ms[1], "refine_ms": ms[2], "calls": cnt[1]}
        rec = {"N": N, "K": K, "e_dim": D, "idx_identical": idx_equal, "zq_bf16_equals_rounded_fp32_zq": zq_equal}
        for kind, zbytes in (("fp32", 4), ("bf16", 2)):
            ms = statistics.median(times[kind])
            nbytes = algorithmic_bytes(N, K, D, zbytes)
            rec[kind] = {"ms_median": ms, "ms_all": times[kind], "main_kernel_ms": stages[kind]["main_kernel_ms"],
                         "refine_ms": stages[kind]["refine_ms"], "undecided_rows": undecided[kind], "loss": loss[kind],
                         "algorithmic_bytes": nbytes, "frac_hbm": nbytes / (ms * 1e-3) / (hbm_gbs * 1e9),
                         "frac_bf16_sustained": 2.0 * N * K * D / (ms * 1e-3) / (bf16_tf * 1e12)}
        rec["speedup_bf16_vs_fp32"] = rec["fp32"]["ms_median"] / rec["bf16"]["ms_median"]
        res["shapes"][sname] = rec
        print(sname, json.dumps(rec), file=sys.stderr, flush=True)
        del out, zb, z32, inp, mods
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()

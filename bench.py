#!/usr/bin/env python
"""bench.py — the headline benchmark of the D-VQVAE hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (N > 1)

--dump-outputs DIR writes what the last timed step returned on rank 0 as DIR/<name>.npy (see dump_outputs): the
inputs are seeded, so two builds run with the same arguments can be compared output for output.

Workload (BASELINE.json configs[1]): fused VQ lookup, N = 4 194 304 fp32 latents PER GPU,
e_dim = 64, n_e = 512, train path (indices + z_q + loss + perplexity + usage histogram),
min_encodings lazy (not materialised).  A "step" is one pass of the path over that batch.
Weak scaling: every rank holds its own 4M-row shard, codebook replicated, one all-reduce of
(hist, sse) per step.  Prints ONE JSON line (rank 0).

  value    whole-job latents/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e      same metric through the host-buffer C-ABI call (dvq_vq_forward_host): pinned host
           z -> H2D -> kernels -> D2H z_q + idx, copies inside the timed region
  roofline dominant kernel vs the measured HBM peak (MEASURED_PEAKS.json), algorithmic bytes
           N*(8*D+8) + 4*K*D per launch (DESIGN.md §4), duration from CUDA events recorded
           around that kernel inside the library on the launching stream
  cpu_baseline  the reference's torch CPU op sequence (oracle/ref_port_torch.py, kind "port")
           on a bounded sample of the same workload, all host threads
  secondary  driver-timed lines for the other BASELINE configs (each with its own roofline fraction): the config-4
           corner K = 16384, e_dim 128 (16 777 216 latents in total, sharded over the GPUs), the PointNet encoder
           (C = 4, P = 3000, 4096 clouds per GPU, tcgen05 path) and grasp generation (config 3 / 5: batch 4096 per
           GPU, PixelCNN prior); whole-job aggregates, max-over-ranks time.  --no-secondary skips them.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "d-vqvae_b200"))

N_PER_GPU = 4194304
E_DIM = 64
N_E = 512
E2E_CHUNK_ROWS = 262144          # rows per chunk of the host-buffer pipeline (e2e leg)
AL, BETA = 1.0, 0.25
DUMP_ZQ_ROWS = 65536             # z_q rows written by --dump-outputs: all 4M rows would be 1 GiB
METRIC = "vq_latents_per_sec"
UNIT = "latents/s"
WORKLOAD = ("BASELINE config 2: fused VQ lookup, N=4194304 fp32 latents per GPU, e_dim=64, n_e=512, "
            "istrain=True (idx + z_q + loss + perplexity + histogram), min_encodings lazy")


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return (float(d["hbm_gbs"]), float(d.get("bf16_tflops", 0.0)), "measured (MEASURED_PEAKS.json)",
                float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 0.0))))
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)", 1590.0


def bind_to_gpu_numa_node(local_rank: int):
    """Pin this process (and therefore the pinned host buffers it first-touches) to the CPU cores of the NUMA node
    the GPU hangs off, so that the host-buffer (e2e) leg of every rank uses its own socket's memory controllers and
    PCIe root instead of node 0.  Returns a description for the JSON line; a no-op where sysfs has no NUMA data."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:                # nvml prints a 32-bit PCI domain, sysfs a 16-bit one
            bus = bus[4:]
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA information for %s" % bus}
        cpus = []
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.extend(range(int(lo), int(hi or lo) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return {"numa_node": node, "note": "no allowed core on that node"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cores": len(allowed)}
    except Exception as e:                              # noqa: BLE001
        return {"numa_node": None, "note": "binding skipped: %r" % (e,)}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 100 ms while the benchmark runs; the median SM
    clock is taken over the samples drawn under load (power above idle)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        pw = []
        for r in self.rows:
            try:
                pw.append(float(r[3]))
            except Exception:
                pass
        load_floor = (min(pw) + 0.25 * (max(pw) - min(pw))) if pw else 0.0
        for r in self.rows:
            try:
                if float(r[3]) < load_floor:
                    continue
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_port_rate(target_seconds: float, max_rows: int):
    """Reference op sequence on host cores (oracle/ref_port_torch.py), bounded sample."""
    import torch
    from oracle import ref_port_torch as port
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(2000)
    E = (torch.rand(N_E, E_DIM, generator=g) * 2 - 1) / N_E
    chunk = 65536
    z = torch.randn(chunk, E_DIM, generator=g)
    port.quantize_rows(z, E, AL, BETA, True)                      # warm-up
    t0 = time.perf_counter()
    port.quantize_rows(z, E, AL, BETA, True)
    per_chunk = max(time.perf_counter() - t0, 1e-4)
    n_chunks = int(max(1, min(max_rows // chunk, target_seconds / per_chunk)))
    zs = torch.randn(n_chunks * chunk, E_DIM, generator=g)
    t0 = time.perf_counter()
    port.quantize_chunked_timed(zs, E, AL, BETA, True, chunk)
    dt = time.perf_counter() - t0
    rows = n_chunks * chunk
    return rows / dt, torch.get_num_threads(), "%d rows (%d chunks of 65536) of the config-2 workload, train path, %.1f s" % (rows, n_chunks, dt)


def dump_outputs(out_dir, vq, out):
    """Write one train step's results as float32 / float64 .npy files, 48.5 MiB in all: the code index of every row
    (min_encodings is the lazy one-hot of it), z_q at a fixed seeded sample of rows (and those row numbers), loss,
    perplexity and the usage histogram."""
    import numpy as np
    import torch
    loss, z_q, ppl, _, idx = out
    rows = np.sort(np.random.RandomState(0).choice(z_q.shape[0], DUMP_ZQ_ROWS, replace=False))
    arrays = {
        "loss": loss.cpu().numpy().astype(np.float32),
        "perplexity": ppl.cpu().numpy().astype(np.float32),
        "indices": idx.reshape(-1).cpu().numpy().astype(np.float64),
        "z_q_rows": rows.astype(np.float64),
        "z_q_sample": z_q[torch.from_numpy(rows).to(z_q.device)].cpu().numpy().astype(np.float32),
        "usage_histogram": vq.last_stats[:vq.n_e].cpu().numpy().astype(np.float64),
    }
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (torch CPU port of
    network/vqvae/quantizer.py — the Python reference cannot travel to the GPU box)."""
    if rank != 0:
        return
    import torch
    from oracle import ref_port_torch as port
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(2000)
    E = (torch.rand(N_E, E_DIM, generator=g) * 2 - 1) / N_E
    chunk = 65536
    z1 = torch.randn(chunk, E_DIM, generator=g)
    port.quantize_rows(z1, E, AL, BETA, True)
    t0 = time.perf_counter()
    port.quantize_rows(z1, E, AL, BETA, True)
    per_chunk = max(time.perf_counter() - t0, 1e-4)
    budget = 150.0 / max(1, args.steps + args.warmup)            # whole run within a few minutes
    n_chunks = int(max(1, min(N_PER_GPU // chunk, budget / per_chunk)))
    rows = n_chunks * chunk
    z = torch.randn(rows, E_DIM, generator=g)
    # quantize_chunked_timed: exactly network/vqvae/quantizer.py:30-67 per chunk + bincount / weighted-mean combine
    for _ in range(args.warmup):
        port.quantize_chunked_timed(z, E, AL, BETA, True, chunk)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        port.quantize_chunked_timed(z, E, AL, BETA, True, chunk)
    dt = time.perf_counter() - t0
    value = rows * args.steps / dt
    sample = "%d of %d rows per step (%d chunks of 65536), train path" % (rows, N_PER_GPU, n_chunks)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample, "device": "host CPU"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def synthetic_mano_tables(seed=0):
    """Random tables with MANO's shapes and kinematic tree for the grasp line (MANO_RIGHT.pkl is not part of the repo)."""
    import numpy as np
    rs = np.random.RandomState(seed)
    w = rs.rand(778, 16) ** 4
    jr = rs.rand(16, 778) ** 8
    return {"v_template": 0.1 * rs.randn(778, 3), "shapedirs": 0.01 * rs.randn(778, 3, 10), "posedirs": 0.002 * rs.randn(778, 3, 135),
            "J_regressor": jr / jr.sum(1, keepdims=True), "weights": w / w.sum(1, keepdims=True),
            "hands_components": rs.randn(45, 45) / 45 ** 0.5, "hands_mean": 0.3 * rs.randn(45),
            "parents": np.array([-1, 0, 1, 2, 0, 4, 5, 0, 7, 8, 0, 10, 11, 0, 13, 14])}


def run_secondary(torch, tdist, dvq, dev, rank, world, fence):
    """Driver-timed lines for the other BASELINE configs (whole-job aggregate over `world` GPUs, CUDA events, max over
    ranks).  Every leg: synthetic inputs resident in HBM, >= 1 warm-up call, 3 timed calls."""
    import math
    hbm_gbs, bf16_tf, peak_src, bf16_sus = measured_peaks()
    out = {"peak_source": peak_src, "bf16_tflops_sustained": bf16_sus}

    def timed(fn, iters=3, warm=1):
        for _ in range(warm):
            fn()
        fence()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        fence()
        ms = a.elapsed_time(b) / iters
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    # ---- config 4 corners: K = 16384 at e_dim 128 and 512, 16 777 216 latents in total (rows sharded), train path.  Both are
    # streamed codebooks on the CTA-pair (cta_group::2) kernel ----
    for K4, D4 in ((16384, 128), (16384, 512)):
        key = "config4_k%d_d%d" % (K4, D4)
        try:
            N4 = 16777216 // world
            g = torch.Generator(device=dev).manual_seed(4000 + rank)
            cg = torch.Generator(device=dev).manual_seed(4000)
            vq4 = dvq.VectorQuantizer(K4, D4, BETA, AL).to(dev)
            vq4.onehot_limit_bytes = 0
            with torch.no_grad():
                vq4.embedding.weight.copy_((torch.rand(K4, D4, device=dev, generator=cg) * 2 - 1) / K4)
            if world > 1:
                dvq.dist.shard_module(vq4)
            z4 = torch.randn(N4, D4, device=dev, generator=g)

            def step4():
                with torch.no_grad():
                    return vq4(z4, True)
            ms = timed(step4, iters=3 if D4 <= 128 else 2)
            tf = 2.0 * N4 * world * K4 * D4 / (ms * 1e-3) / 1e12
            plan = (ctypes.c_int * 8)()
            dvq._cabi.lib.dvq_debug_tc_pair_layout(N4, K4, D4, plan)
            out[key] = {
                "metric": METRIC, "value": N4 * world / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "rows_per_gpu": N4, "n_e": K4, "e_dim": D4,
                "undecided_rows_rank0": vq4.last_counters(N4)[0], "kernel": "cta_pair (cta_group::2)" if plan[0] else "single CTA",
                "roofline": {"bound": "tensor", "achieved": tf, "peak": bf16_sus * world, "unit": "TFLOP/s", "frac": tf / (bf16_sus * world),
                             "what": "2*N*K*e_dim of the whole call (filter + exact refine + finalize) over the sustained BF16 peak x GPUs"}}
            del z4, vq4
            torch.cuda.empty_cache()
        except Exception as e:                                  # noqa: BLE001
            out[key] = {"error": repr(e)}

    # ---- PointNet encoder: C = 4, P = 3000, 4096 clouds per GPU, default (tcgen05) path ----
    try:
        B, P = 4096, 3000
        torch.manual_seed(0)
        enc = dvq.PointNetEncoder(channel=4).to(dev).eval().requires_grad_(False)
        g = torch.Generator(device=dev).manual_seed(3000 + rank)
        obj = 0.1 * torch.randn(B, 4, P, device=dev, generator=g)
        obj[:, 3, :] = 0.05 + 0.25 * torch.rand(B, 1, device=dev, generator=g)
        ms = timed(lambda: enc(obj))
        flop = B * world * P * 558080.0
        tf = flop / (ms * 1e-3) / 1e12
        out["pointnet_c4_p3000"] = {
            "metric": "pointnet_clouds_per_sec", "value": B * world / (ms * 1e-3), "unit": "clouds/s", "ms_per_call": ms, "clouds_per_gpu": B,
            "precision": enc.precision,
            "roofline": {"bound": "tensor", "achieved": tf, "peak": bf16_sus * world, "unit": "TFLOP/s", "frac": tf / (bf16_sus * world),
                         "what": "558 080 flop per point (STN trunk + main trunk) over the sustained BF16 peak x GPUs",
                         "hbm_gbs": B * world * (16.0 * P + 4096) / (ms * 1e-3) / 1e9}}
        del enc
    except Exception as e:                                  # noqa: BLE001
        out["pointnet_c4_p3000"] = {"error": repr(e)}
        obj = None

    # ---- grasp generation (config 3; at N GPUs the config-5 layout: objects sharded, weights replicated) ----
    try:
        from dvq.grasp import pixelcnn_prior
        from dvq.pixelcnn import GatedPixelCNN
        torch.manual_seed(0)
        net = dvq.GraspGenerator(hand_layer=dvq.ManoLayer(synthetic_mano_tables())).to(dev).eval().requires_grad_(False)
        torch.manual_seed(1)
        pcnn = GatedPixelCNN(512, 512, 15).to(dev).eval().requires_grad_(False)
        pcnn.precision = "fp16_tc"                          # the repo's tcgen05 GEMM kernel (csrc/pcnn_sm100.cu)
        net.prior = pixelcnn_prior(pcnn, n_valid=128)
        ms = timed(lambda: net.gen(obj))
        ms_sampler = timed(lambda: pcnn.generate(None, torch.zeros(B, dtype=torch.int64, device=dev), batch_size=B, n_valid=128))
        try:
            ms_graph = timed(lambda: net.gen_graphed(obj))
        except Exception as e:                              # noqa: BLE001
            ms_graph = None
        pcnn_flop = float(pcnn._tc_sampler.flops)             # tensor-core flops of one sample grid of B grasps, counted per launch
        flop = world * (B * (2 * P * 558080.0 + 778 * (2 * (3 * 64 + 64 * 128 + 128 * 1024) * 2.0)) + pcnn_flop)
        out["grasp_generation_b4096"] = {
            "metric": "grasps_per_sec", "value": B * world / (ms * 1e-3), "unit": "grasps/s", "ms_per_batch": ms, "batch_per_gpu": B, "points": P,
            "prior": "GatedPixelCNN(512,512,15), exact row-cached sampler, %s, random init, 128 valid classes" % pcnn.backend_name(),
            "hand_layer": "dvq.ManoLayer (LBS kernel, 55 parameters -> 778 vertices) on synthetic model tables of MANO's shapes (the asset does not travel to the GPU box)",
            "pixelcnn_sampler_ms": ms_sampler,
            "ms_per_batch_cuda_graph": ms_graph,
            "roofline": {"bound": "tensor", "achieved": flop / (ms * 1e-3) / 1e12, "peak": bf16_sus * world, "unit": "TFLOP/s",
                         "frac": flop / (ms * 1e-3) / 1e12 / (bf16_sus * world),
                         "pixelcnn_gflop_per_grasp": pcnn_flop / B / 1e9, "pixelcnn_sampler_tflops": pcnn_flop / (ms_sampler * 1e-3) / 1e12,
                         "what": "PointNets 3.78 GFLOP per grasp + the row-cached PixelCNN sampler's issued GEMM flops (counted per launch) over the sustained BF16 peak x GPUs"}}
    except Exception as e:                                  # noqa: BLE001
        out["grasp_generation_b4096"] = {"error": repr(e)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=0, help="steps of the host-buffer leg (default: min(steps, 10))")
    ap.add_argument("--path", default="auto", choices=["auto", "simt", "tc"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the config-3/4/5 lines of the `secondary` dict")
    ap.add_argument("--no-numa-bind", action="store_true", help="do not pin the rank to the GPU's NUMA node")
    ap.add_argument("--raw-nccl", action="store_true", help="all-reduce (hist, sse) through dvq_allreduce_stats instead of torch.distributed")
    ap.add_argument("--e2e-chunk-rows", type=int, default=E2E_CHUNK_ROWS, help="rows per chunk of the host-buffer pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs (rank 0) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as tdist
    import dvq
    from dvq import _cabi

    numa = {"numa_node": None, "note": "disabled"} if args.no_numa_bind else bind_to_gpu_numa_node(local_rank)
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        tdist.init_process_group("nccl", device_id=dev)
        if args.raw_nccl:
            dvq.dist.use_raw_nccl(True)

    gen = torch.Generator(device=dev).manual_seed(2000 + rank)
    cb_gen = torch.Generator(device=dev).manual_seed(2000)       # replicated codebook
    vq = dvq.VectorQuantizer(N_E, E_DIM, BETA, AL).to(dev)
    with torch.no_grad():
        vq.embedding.weight.copy_((torch.rand(N_E, E_DIM, device=dev, generator=cb_gen) * 2 - 1) / N_E)
    vq.path = {"auto": _cabi.DVQ_PATH_AUTO, "simt": _cabi.DVQ_PATH_SIMT, "tc": _cabi.DVQ_PATH_TC}[args.path]
    vq.onehot_limit_bytes = 0
    if world > 1:
        dvq.dist.shard_module(vq)
    z = torch.randn(N_PER_GPU, E_DIM, device=dev, generator=gen)

    def step():
        with torch.no_grad():
            return vq(z, True)

    def fence():
        torch.cuda.synchronize(dev)
        if world > 1:
            tdist.barrier()
            torch.cuda.synchronize(dev)

    # clocks / throttle reasons are sampled from the first warm-up step to the end of the e2e leg (the
    # device-resident timed region alone can be shorter than one 100 ms sampling period)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        out = step()
    fence()

    # ---- timed region: device-resident inputs --------------------------------------------------
    _cabi.lib.dvq_profile_enable(1)
    launches0 = _cabi.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    ev0.record()
    for _ in range(args.steps):
        out = step()
    ev1.record()
    fence()
    # the library's per-stage CUDA events (recorded on the launching stream), mean over the timed steps
    prof_ms, prof_cnt = _cabi.profile_mean()
    elapsed_ms = ev0.elapsed_time(ev1)
    launches = _cabi.launch_count() - launches0
    _cabi.lib.dvq_profile_enable(0)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    loss, z_q, ppl, enc, idx = out
    value = N_PER_GPU * world * args.steps / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, vq, out)

    # ---- e2e: host buffers through dvq_vq_forward_host --------------------------------------------
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    hq = dvq.HostQuantizer(chunk_rows=args.e2e_chunk_rows, n_e_max=N_E, e_dim_max=E_DIM, device=dev)
    z_host = torch.empty((N_PER_GPU, E_DIM), dtype=torch.float32, pin_memory=True)
    z_host.copy_(z)
    E_host = vq.embedding.weight.detach().cpu().pin_memory()
    zq_host = torch.empty((N_PER_GPU, E_DIM), dtype=torch.float32, pin_memory=True)
    idx_host = torch.empty((N_PER_GPU, 1), dtype=torch.int64, pin_memory=True)
    for _ in range(2):
        hq.forward(z_host, E_host, True, AL, BETA, out_zq=zq_host, out_idx=idx_host, path=vq.path)
    fence()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        l_h, _, p_h, _ = hq.forward(z_host, E_host, True, AL, BETA, out_zq=zq_host, out_idx=idx_host, path=vq.path)
    torch.cuda.synchronize(dev)
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = N_PER_GPU * world * e2e_steps / e2e_s
    same_idx = bool(torch.equal(idx_host, idx.cpu()))
    # copy-only ceiling of the same pipeline: identical chunks, streams and buffers, kernels skipped (DVQ_HOST_COPY_ONLY)
    zq_scratch = zq_host                                   # (outputs are undefined in this mode: the buffers are reused after the check above)
    hq.forward(z_host, E_host, True, AL, BETA, out_zq=zq_scratch, out_idx=idx_host, path=vq.path, copy_only=True)
    fence()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        hq.forward(z_host, E_host, True, AL, BETA, out_zq=zq_scratch, out_idx=idx_host, path=vq.path, copy_only=True)
    torch.cuda.synchronize(dev)
    copy_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([copy_s], device=dev, dtype=torch.float64)
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        copy_s = float(t.item())
    copy_value = N_PER_GPU * world * e2e_steps / copy_s
    hq.close()
    del z_host, zq_host, idx_host, hq
    secondary = None
    if not args.no_secondary:
        del z, out, z_q, enc, idx
        torch.cuda.empty_cache()
        secondary = run_secondary(torch, tdist, dvq, dev, rank, world, fence)
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        hbm_gbs, bf16_tf, peak_src, bf16_sus = measured_peaks()
        alg_bytes = N_PER_GPU * (8 * E_DIM + 8) + 4 * N_E * E_DIM
        k_ms = prof_ms[1]
        achieved = alg_bytes / (k_ms * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": hbm_gbs, "unit": "GB/s", "frac": achieved / hbm_gbs,
                "traffic": None, "traffic_source": None, "kernel": "vq main kernel (stage 1 of dvq_vq_forward)", "kernel_ms": k_ms,
                "refine_ms": prof_ms[2], "launches_averaged": prof_cnt[1], "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes,
                "whole_step_frac": alg_bytes / (elapsed_ms / args.steps * 1e-3) / 1e9 / hbm_gbs,
                # in-step tensor-pipe figure against the SUSTAINED BF16 peak (the kernel is timed inside a long step)
                "tensor_tflops": 2.0 * N_PER_GPU * N_E * E_DIM / (k_ms * 1e-3) / 1e12,
                "tensor_frac_of_bf16_sustained": (2.0 * N_PER_GPU * N_E * E_DIM / (k_ms * 1e-3) / 1e12) / bf16_sus if bf16_sus else None}
        for name in ("traffic_r02.json", "traffic_r01.json"):     # not measured in this run: one `ncu --set full` capture per round
            tr = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tr):
                try:
                    roof["traffic"] = json.load(open(tr)).get("dram_bytes_per_launch")
                    roof["traffic_source"] = "profiles/%s (ncu --set full capture of this kernel, dram__bytes_read.sum + dram__bytes_write.sum; not re-measured in this run)" % name
                    break
                except Exception:
                    pass
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            rate, cores, sample = cpu_port_rate(15.0, N_PER_GPU)
            cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "l2_policy": "inputs (1 GiB z per GPU) larger than the 126 MB L2; no flush needed",
                       "path": args.path, "parallelism": "rows sharded over %d GPU(s), codebook replicated, 1 all-reduce of (hist,sse)" % world,
                       "loss": float(loss.item()), "perplexity": float(ppl.item())},
            "roofline": roof, "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": N_PER_GPU * E_DIM * 4 + N_E * E_DIM * 4,
                    "d2h_bytes_per_step": N_PER_GPU * E_DIM * 4 + N_PER_GPU * 8 + 8, "steps": e2e_steps,
                    "ms_per_step": e2e_s / e2e_steps * 1e3, "api": "dvq_vq_forward_host (pinned host buffers, 3-stream chunk pipeline, %d-row chunks)" % args.e2e_chunk_rows,
                    "indices_equal_device_path": same_idx,
                    "copy_only_ceiling": {"value": copy_value, "unit": UNIT, "ms_per_step": copy_s / e2e_steps * 1e3,
                                          "frac_of_ceiling": e2e_value / copy_value,
                                          "what": "the same chunk pipeline (H2D z, D2H z_q + idx, pinned buffers, 3 streams) with the kernels skipped"},
                    "numa": numa},
            "secondary": secondary,
            "gpu_launches": launches, "clocks": clocks,
        }
        print(json.dumps(line))
    if world > 1:
        tdist.destroy_process_group()


if __name__ == "__main__":
    main()
